"""Write tests/golden/reference/kernels.npz: the reference's OWN kernels' outputs (oracle/_ref, built by
__graft_entry__.build() from the original project's sources) for every case the GPU tests compare with.

Run on a B200 where oracle/_ref was built:  python tests/golden/make_golden_reference.py OUT.npz
then copy OUT.npz to tests/golden/reference/kernels.npz.  The inputs are regenerated from the seeded case builders
of the tests, so the file holds outputs only (tests/refdata.py describes the format)."""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import common  # noqa: E402
import fuzz_cases  # noqa: E402
import refdata  # noqa: E402
import test_gpu_configs as configs  # noqa: E402
import test_gpu_fullsize as fullsize  # noqa: E402
import test_gpu_parity as parity  # noqa: E402
import test_gpu_reference_op as refop  # noqa: E402
from oracle import ref_gpu  # noqa: E402

dev = parity.to_dev  # (torch, array) -> cuda tensor


def run_ref(case, attr_dtype="float32", weight_threshold=0.001, max_intersections=1024, return_contribution=False,
            backward=True):
    f = case.foam
    half = attr_dtype == "float16"
    attrs = f.attributes.astype(np.float16) if half else f.attributes
    scene = [dev(torch, x) for x in (f.points, attrs, f.adjacency, f.offsets)]
    rays, start, dq = dev(torch, case.rays), dev(torch, case.start), dev(torch, case.quantiles)
    fwd = ref_gpu.trace_forward(*scene, rays, start, dq, weight_threshold, max_intersections, return_contribution)
    out = {k: v.cpu().numpy() for k, v in fwd.items()}
    if backward:
        g = case.grad_rgba.astype(np.float16) if half else case.grad_rgba
        bwd = ref_gpu.trace_backward(*scene, rays, start, fwd["rgba"], dev(torch, g), dq, fwd.get("depth_indices"),
                                     dev(torch, case.grad_depth), None, weight_threshold, max_intersections)
        out.update({k: v.cpu().numpy() for k, v in bwd.items() if k != "ray_grad"})
    torch.cuda.synchronize()
    return out


def grads_only(out):
    return {k: out[k] for k in ("points_grad", "attr_grad")}


def forward_only(out):
    return {k: out[k] for k in ("num_intersections", "depth_indices", "rgba", "depth") if k in out}


GRADS_WHOLE = {"points_grad": 1e-5, "attr_grad": 1e-5}  # the bar the tests hold these outputs to


def parity_cases(w):
    for deg in range(4):
        case = common.config1(deg, 2)
        w.add(f"config1_deg{deg}_q2", refdata.case_inputs(case), run_ref(case, return_contribution=True),
              tol=dict(GRADS_WHOLE, contribution=1e-8))  # contribution: atol 1e-6, kept to 6e-10 of its max
    for name, make in parity.LARGE_CASES.items():
        case = make()
        ref = run_ref(case)
        scalars = None
        if name.startswith("scene60k"):  # the reference's own run-to-run scatter-add noise
            ref2 = run_ref(case)
            scalars = {"noise": max(common.grad_error(ref2[k], ref[k]) for k in ("points_grad", "attr_grad"))}
        w.add(name, refdata.case_inputs(case), ref, scalars)
    case = common.scene_case()
    w.add("scene20k_half_forward", refdata.case_inputs(case), run_ref(case, attr_dtype="float16", backward=False),
          spread=4096)
    for model in ("pinhole", "fisheye"):
        for attr_dtype in ("float16", "float32"):
            scene, cam, start = parity.benchmark_inputs(torch, model, attr_dtype)
            diff = ref_gpu.prefetch_adjacent_diff(scene[0], scene[2], scene[3])
            out = torch.zeros((120, 200), dtype=torch.uint32, device="cuda")
            ref_gpu.trace_benchmark(*scene, diff, cam, start, out, weight_threshold=0.05)
            torch.cuda.synchronize()
            w.add(f"trace_benchmark_{model}_{attr_dtype}", (scene, cam, start),
                  {"adjacent_diff": diff.view(torch.int16), "frame": out})
    import tempfile

    with tempfile.TemporaryDirectory() as tmp:
        pt = parity.pt_checkpoint_world(torch, tmp)
    frames = {}
    for k in range(3):
        out = torch.zeros((pt["height"], pt["width"]), dtype=torch.uint32, device="cuda")
        cam_np = {key: (v.numpy() if isinstance(v, torch.Tensor) else v) for key, v in pt["cameras"][k].items()}
        ref_gpu.trace_benchmark(*pt["trace_data"], pt["diff"], cam_np, pt["starts"][k:k + 1], out,
                                weight_threshold=0.05)
        torch.cuda.synchronize()
        frames[f"frame{k}"] = out
    w.add("pt_checkpoint_frames", parity.pt_checkpoint_inputs(pt), frames)


def fuzz(w):
    for seed in range(240):
        _, _, f, rays, start, dq, kw = fuzz_cases.make_case(seed)
        full = dict(weight_threshold=0.001, max_intersections=1024)
        full.update(kw)
        case = common.Case(f, rays, start, dq, seed=seed)
        ref = run_ref(case, **full)
        inputs = refdata.case_inputs(case) + (kw,)
        w.add(f"fuzz{seed}", inputs, forward_only(ref), top=0, spread=0)
        w.add(f"fuzz{seed}", inputs, grads_only(ref), tol={"points_grad": 2e-5, "attr_grad": 2e-5})
    _, _, f, rays, start, dq, kw = fuzz_cases.make_case(3736)
    whole = common.Case(f, rays, start, dq, seed=3736)
    for i in range(0, rays.shape[0], 2):
        case = common.Case(f, rays[i:i + 1], start[i:i + 1], dq[i:i + 1], seed=3736)
        case.grad_rgba, case.grad_depth = whole.grad_rgba[i:i + 1], whole.grad_depth[i:i + 1]
        ref = run_ref(case, weight_threshold=0.0, max_intersections=1024)
        inputs = refdata.case_inputs(case) + (kw,)
        w.add(f"fuzz3736_ray{i}", inputs, {"rgba": ref["rgba"], "depth": ref["depth"]}, top=0, spread=0)
        w.add(f"fuzz3736_ray{i}", inputs, grads_only(ref), tol=GRADS_WHOLE)


def farthest(w):
    for make in ("edge", "scene200k"):
        f = common.farthest_edge_case() if make == "edge" else common.scene_case(200000, 8, 8, 0).foam
        idx, radius = ref_gpu.farthest_neighbor(dev(torch, f.points), dev(torch, f.adjacency), dev(torch, f.offsets))
        torch.cuda.synchronize()
        w.add(f"farthest_{make}", (f.points, f.adjacency, f.offsets), {"indices": idx, "radius": radius})


def full_size(w):
    x = fullsize.inputs(torch)
    rf = ref_gpu.trace_forward(*x["scene"], x["rays"], x["start"], x["dq"])
    rb = ref_gpu.trace_backward(*x["scene"], x["rays"], x["start"], rf["rgba"], x["g"], x["dq"], rf["depth_indices"],
                                x["gd"])
    w.add("config2_512k_1080p", fullsize.inputs_of(x), dict(forward_only(rf), **grads_only(rb)))


def config_sizes(w):
    for name, (num_points, width, height, max_intersections) in configs.STEPS.items():
        f, scene = configs.scene_tensors(torch, num_points)
        rays, start, dq, g, gd = configs.frame_tensors(torch, f, width, height, seed=num_points % 1000 + width)
        kw = {} if max_intersections is None else {"max_intersections": max_intersections}
        rf = ref_gpu.trace_forward(*scene, rays, start, dq, **kw)
        rb = ref_gpu.trace_backward(*scene, rays, start, rf["rgba"], g, dq, rf["depth_indices"], gd, **kw)
        rb2 = ref_gpu.trace_backward(*scene, rays, start, rf["rgba"], g, dq, rf["depth_indices"], gd, **kw)
        noise = {}
        for k in ("points_grad", "attr_grad"):  # radfoam_model/render.py:98-99 zeroes non-finite gradients
            rb[k][~rb[k].isfinite()] = 0
            rb2[k][~rb2[k].isfinite()] = 0
            noise["noise_" + k] = float((rb2[k] - rb[k]).abs().max() / rb[k].abs().max())
        w.add(name, (scene, rays, start, dq, g, gd), dict(forward_only(rf), **grads_only(rb)), noise)
        del rf, rb, rb2


def reference_op(w):
    mod = refop.load_reference_op()
    case = common.scene_case(20000, 160, 96, q=2)
    for with_error in (False, True):
        for contribution in (False, True):
            w.add(f"reference_op_error{int(with_error)}_contribution{int(contribution)}", refdata.case_inputs(case),
                  refop.drive(torch, mod.TraceRays, refop.ReferencePipeline(), case, with_error, contribution),
                  tol={"point_error": 1e-5, "contribution": 1e-5})
    # FoamScene.collect_error_map's loop (scene.py:497-548) spelled out with the reference's own autograd op on the
    # reference's own kernels, after the collect_error_map call the test makes, so that the scene is in the same state
    em = refop.error_map_world(torch)
    refop.our_error_map(torch, em)
    scene, f, rays, rgbs, cams = em["scene"], em["foam"], em["rays"], em["rgbs"], em["cams"]
    ref_pipe = refop.ReferencePipeline()
    gen = torch.Generator().manual_seed(9)
    want_err = torch.zeros((f.points.shape[0], 1), device="cuda")
    want_contrib = torch.zeros((f.points.shape[0], 1), device="cuda")
    from radfoam_b200 import foam

    starts = [int(foam.nearest_point(f.points, c)) for c in cams]
    for v in range(len(cams)):
        d = torch.randint(0, 2, (2,), generator=gen)
        ray_batch = rays[v:v + 1, int(d[0])::2, int(d[1])::2, :].cuda()
        rgb_batch = rgbs[v:v + 1, int(d[0])::2, int(d[1])::2, :].cuda()
        points, attributes, adjacency, offsets = scene.get_trace_data()
        start = torch.full(ray_batch.shape[:-1], starts[v], dtype=torch.int64, device="cuda").to(torch.uint32)
        rgba, _, contribution, _, _ = mod.TraceRays.apply(ref_pipe, points, attributes, adjacency, offsets, ray_batch,
                                                          start, None, True)
        rgb = rgba[..., :3] + (1 - rgba[..., -1:])
        (rgb_batch - rgb).abs().mean(dim=-1).sum().backward()
        want_err += scene.primal_points.grad.norm(dim=-1, keepdim=True).detach()
        want_contrib = torch.maximum(want_contrib, contribution.detach())
        for t in (scene.primal_points, scene.att_dc, scene.att_sh, scene.density):
            t.grad = None
    w.add("collect_error_map", refop.error_map_inputs(em), {"error": want_err, "contribution": want_contrib},
          tol={"error": 1e-5, "contribution": 1e-5})


def main(path):
    assert ref_gpu.available(), "oracle/_ref was not built"
    w = refdata.Writer()
    for part in (parity_cases, fuzz, farthest, reference_op, full_size, config_sizes):
        t0 = time.time()
        part(w)
        print(part.__name__, f"done in {time.time() - t0:.0f} s", flush=True)
    w.save(path)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main(sys.argv[1])
