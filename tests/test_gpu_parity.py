"""GPU parity tests proper: the hand-written sm_100a path, called through the public
Pipeline API -> ctypes -> C ABI, against
  (a) the CPU oracle (oracle/radfoam_oracle.c), and
  (b) the reference's own kernels, through their outputs stored in tests/golden/reference/kernels.npz
      (tests/refdata.py; made by tests/golden/make_golden_reference.py).
Bars (BASELINE.json north_star): integer outputs bit-exact; floats within 1e-5; gradients
within 1e-5 of max|ref| (they are float scatter-adds, order-nondeterministic in the reference)."""
import os

import numpy as np
import pytest

import common
import refdata

pytestmark = pytest.mark.gpu

GRAD_TOL = 1e-5


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def to_dev(torch, a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def run_ours(torch, case, attr_dtype="float32", weight_threshold=None, max_intersections=None,
             return_contribution=False, flat=False, backward=True, ray_error=None, tape=False, repeat=1):
    import radfoam_b200

    f = case.foam
    half = attr_dtype == "float16"
    pipe = radfoam_b200.create_pipeline(f.sh_degree, attr_dtype)
    attrs = f.attributes.astype(np.float16) if half else f.attributes
    rays, start, dq = case.rays, case.start, case.quantiles
    g, gd = case.grad_rgba, case.grad_depth
    if flat:
        rays = rays.reshape(-1, 6)
        start = start.reshape(-1)
        dq = None if dq is None else dq.reshape(-1, dq.shape[-1])
        g = g.reshape(-1, 4)
        gd = None if gd is None else gd.reshape(-1, gd.shape[-1])
    scene = [to_dev(torch, x) for x in (f.points, attrs, f.adjacency, f.offsets)]
    if tape:  # scene tensors that require grad make the forward record the walk tape
        scene[0].requires_grad_(True)
        scene[1].requires_grad_(True)
    pipe.record_tape = tape
    rays_d, start_d, dq_d = to_dev(torch, rays), to_dev(torch, start), to_dev(torch, dq)
    for _ in range(repeat):
        fwd = pipe.trace_forward(*scene, rays_d, start_d, depth_quantiles=dq_d,
                                 weight_threshold=weight_threshold, max_intersections=max_intersections,
                                 return_contribution=return_contribution)
        out = {k: v.cpu().numpy() for k, v in fwd.items()}
        if backward:
            g_d = to_dev(torch, g.astype(np.float16) if half else g)
            err_d = to_dev(torch, ray_error)
            bwd = pipe.trace_backward(*scene, rays_d, start_d, fwd["rgba"], g_d, dq_d,
                                      fwd.get("depth_indices"), to_dev(torch, gd), err_d,
                                      weight_threshold=weight_threshold, max_intersections=max_intersections)
            out.update({k: v.cpu().numpy() for k, v in bwd.items() if k != "ray_grad"})
        torch.cuda.synchronize()
    return out


def run_cpu_oracle(case, attr_dtype="float32", weight_threshold=0.001, max_intersections=1024,
                   return_contribution=False, backward=True, ray_error=None):
    from oracle import oracle

    f = case.foam
    attrs = f.attributes.astype(np.float16) if attr_dtype == "float16" else f.attributes
    fwd = oracle.trace_forward(f.points, attrs, f.adjacency, f.offsets, case.rays, case.start,
                               case.quantiles, weight_threshold, max_intersections, return_contribution)
    out = dict(fwd)
    if backward:
        g = case.grad_rgba.astype(attrs.dtype)
        out.update(oracle.trace_backward(f.points, attrs, f.adjacency, f.offsets, case.rays, case.start,
                                         fwd["rgba"], g, case.quantiles, fwd.get("depth_indices"),
                                         case.grad_depth, ray_error, weight_threshold, max_intersections))
    return out


def assert_matches_cpu_oracle(got, ref, case, grads=True):
    """Integers bit-exact; floats to the conditioning-aware CPU bars of tests/common.py."""
    common.assert_forward_close_cpu(got, ref, case.foam.attributes)
    if grads:
        assert_grads_close(got, ref, common.CPU_GRAD_TOL)


def assert_grads_close(got, ref, tol=GRAD_TOL):
    for k in ("points_grad", "attr_grad"):
        err = common.grad_error(got[k], ref[k])
        assert err <= tol, f"{k}: max|d| / max|ref| = {err:.3e} > {tol}"


# ------------------------------------------------------------------ vs the CPU oracle
@pytest.mark.parametrize("deg", [0, 1, 2, 3])
@pytest.mark.parametrize("q", [0, 2])
def test_config1_matches_cpu_oracle(torch_cuda, deg, q):
    case = common.config1(deg, q)
    got = run_ours(torch_cuda, case, return_contribution=True)
    ref = run_cpu_oracle(case, return_contribution=True)
    assert_matches_cpu_oracle(got, ref, case)


def test_random_quantiles_three(torch_cuda):
    case = common.config1(3, 3, fixed_quantiles=False)
    assert_matches_cpu_oracle(run_ours(torch_cuda, case, backward=False), run_cpu_oracle(case, backward=False),
                              case, grads=False)


def test_scene_matches_cpu_oracle(torch_cuda):
    case = common.scene_case()
    got, ref = run_ours(torch_cuda, case), run_cpu_oracle(case)
    assert_matches_cpu_oracle(got, ref, case)


def test_random_ray_batch_matches_cpu_oracle(torch_cuda):
    case = common.random_ray_case()
    got, ref = run_ours(torch_cuda, case), run_cpu_oracle(case)
    assert_matches_cpu_oracle(got, ref, case)


@pytest.mark.parametrize("kwargs", [dict(max_intersections=1), dict(max_intersections=7),
                                    dict(weight_threshold=0.5), dict(weight_threshold=0.0)])
def test_trace_settings(torch_cuda, kwargs):
    case = common.scene_case(q=2)
    full = dict(weight_threshold=0.001, max_intersections=1024)
    full.update(kwargs)
    got = run_ours(torch_cuda, case, **kwargs)
    ref = run_cpu_oracle(case, **full)
    assert_matches_cpu_oracle(got, ref, case)
    assert got["num_intersections"].max() <= full["max_intersections"] + 1


def test_ray_error_and_point_error(torch_cuda):
    case = common.config1(3, 2)
    err = np.random.default_rng(3).uniform(0, 1, size=(32, 32)).astype(np.float32)
    got = run_ours(torch_cuda, case, ray_error=err)
    ref = run_cpu_oracle(case, ray_error=err)
    np.testing.assert_allclose(got["point_error"], ref["point_error"], rtol=1e-5, atol=1e-6)


def test_prefetch_adjacent_diff_bit_exact(torch_cuda):
    import radfoam_b200
    from oracle import oracle

    f = common.scene_case().foam
    pipe = radfoam_b200.create_pipeline(3)
    got = pipe.prefetch_adjacent_diff(*[to_dev(torch_cuda, x) for x in (f.points, f.adjacency, f.offsets)])
    ref = oracle.prefetch_adjacent_diff(f.points, f.adjacency, f.offsets)
    assert np.array_equal(got.cpu().numpy().view(np.uint16), ref.view(np.uint16))


# ------------------------------------------------------------------ vs the reference's own kernels
LARGE_CASES = {
    "scene60k_outside": lambda: common.scene_case(num_points=60000, width=320, height=200),
    "scene60k_inside": lambda: common.scene_case(num_points=60000, width=320, height=200, inside=True),
    "random60k_100k": lambda: common.random_ray_case(num_points=60000, num_rays=100000),
}


@pytest.fixture(params=["cached", "direct"])
def bwd_mode(request, monkeypatch):
    """Both backward kernels (warp-aggregated shared-memory cache / direct reductions)."""
    monkeypatch.setenv("RFB_BWD_MODE", request.param)
    return request.param


@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_config1_matches_reference_kernels(torch_cuda, deg, bwd_mode):
    case = common.config1(deg, 2)
    got = run_ours(torch_cuda, case, return_contribution=True)
    ref = refdata.reference(f"config1_deg{deg}_q2", refdata.case_inputs(case))
    refdata.assert_forward_equal(got, ref)
    refdata.assert_close(got["contribution"], ref["contribution"], "contribution", rtol=1e-5, atol=1e-6)
    refdata.assert_grads_close(got, ref, GRAD_TOL)


@pytest.mark.parametrize("inside", [False, True])
def test_scene_matches_reference_kernels(torch_cuda, inside, bwd_mode):
    name = "scene60k_inside" if inside else "scene60k_outside"
    case = LARGE_CASES[name]()
    ref = refdata.reference(name, refdata.case_inputs(case))
    got = run_ours(torch_cuda, case)
    refdata.assert_forward_equal(got, ref)
    # the reference's own run-to-run scatter-add noise (measured when the reference outputs were stored)
    noise = ref["noise"]
    ours = max(refdata.grad_error(got[k], ref[k]) for k in ("points_grad", "attr_grad"))
    print(f"grad error vs reference {ours:.2e}; reference self-noise {noise:.2e}")
    assert ours <= max(GRAD_TOL, 4 * noise)


def test_random_ray_batch_matches_reference_kernels(torch_cuda, bwd_mode):
    case = LARGE_CASES["random60k_100k"]()
    got, ref = run_ours(torch_cuda, case), refdata.reference("random60k_100k", refdata.case_inputs(case))
    refdata.assert_forward_equal(got, ref)
    refdata.assert_grads_close(got, ref, GRAD_TOL)


def test_cpu_oracle_matches_reference_kernels(torch_cuda):
    """Pins the restatement (and the Eigen shim) against the reference source itself."""
    case = LARGE_CASES["scene60k_outside"]()
    ref, cpu = refdata.reference("scene60k_outside", refdata.case_inputs(case)), run_cpu_oracle(case)
    # common.assert_forward_close_cpu + the CPU gradient bar, on the stored entries of the reference's outputs
    refdata.assert_equal(cpu["num_intersections"], ref["num_intersections"], "num_intersections")
    refdata.assert_equal(cpu["depth_indices"], ref["depth_indices"], "depth_indices")
    refdata.assert_close(cpu["rgba"], ref["rgba"], "rgba")
    didx = ref["depth"].at(cpu["depth_indices"])  # equal to the reference's (checked above)
    tol = common.depth_tolerance(case.foam.attributes, ref["depth"].values.astype(np.float64), didx)
    bad = np.abs(ref["depth"].at(cpu["depth"]).astype(np.float64) - ref["depth"].values) > tol
    assert not bad.any(), f"{int(bad.sum())} depth entries outside the conditioned bound"
    refdata.assert_grads_close(cpu, ref, common.CPU_GRAD_TOL)


def test_half_attributes_forward(torch_cuda):
    case = common.scene_case()
    ref = refdata.reference("scene20k_half_forward", refdata.case_inputs(case))
    got = run_ours(torch_cuda, case, attr_dtype="float16", backward=False)
    assert got["rgba"].dtype == np.float16
    refdata.assert_equal(got["num_intersections"], ref["num_intersections"], "num_intersections")
    refdata.assert_equal(got["depth_indices"], ref["depth_indices"], "depth_indices")
    refdata.assert_close(got["rgba"], ref["rgba"], "rgba", rtol=1e-3, atol=1e-3)  # one half ulp
    assert (ref["rgba"].at(got["rgba"]).astype(np.float64) != ref["rgba"].values).mean() < 1e-3


def test_half_attributes_backward(torch_cuda):
    """fp16 mode: the reference accumulates gradients with half atomics (CAS loops, each add
    rounded to half); this library accumulates in fp32 and rounds once, so agreement is to
    half precision of the sums."""
    case = common.config1(3, 2)
    got = run_ours(torch_cuda, case, attr_dtype="float16")
    ref = run_cpu_oracle(case, attr_dtype="float16")
    assert got["attr_grad"].dtype == np.float16
    assert common.grad_error(got["points_grad"], ref["points_grad"]) < 1e-3
    assert common.grad_error(got["attr_grad"].astype(np.float32), ref["attr_grad"].astype(np.float32)) < 2e-2


def benchmark_inputs(torch, model, attr_dtype):
    """-> (scene tensors, camera dict, start cell) of test_trace_benchmark."""
    from radfoam_b200 import foam

    f = common.scene_case().foam
    attrs = f.attributes.astype(np.float16 if attr_dtype == "float16" else np.float32)
    scene = [to_dev(torch, x) for x in (f.points, attrs, f.adjacency, f.offsets)]
    pos = (2.5, 2.5, 2.5)
    cam = foam.camera_dict(pos, fov=0.9 if model == "pinhole" else 1.2, width=200, height=120, model=model)
    start = to_dev(torch, np.array([foam.nearest_point(f.points, pos)], dtype=np.uint32))
    return scene, cam, start


@pytest.mark.parametrize("model", ["pinhole", "fisheye"])
@pytest.mark.parametrize("attr_dtype", ["float16", "float32"])
def test_trace_benchmark(torch_cuda, model, attr_dtype):
    import radfoam_b200

    torch = torch_cuda
    scene, cam, start = benchmark_inputs(torch, model, attr_dtype)
    ref = refdata.reference(f"trace_benchmark_{model}_{attr_dtype}", (scene, cam, start))
    pipe = radfoam_b200.create_pipeline(3, attr_dtype)
    diff = pipe.prefetch_adjacent_diff(scene[0], scene[2], scene[3])
    refdata.assert_equal(diff.view(torch.int16).cpu().numpy(), ref["adjacent_diff"], "prefetch_adjacent_diff")
    out = torch.zeros((120, 200), dtype=torch.uint32, device="cuda")
    cam_t = {k: (torch.from_numpy(v) if isinstance(v, np.ndarray) else v) for k, v in cam.items()}
    pipe.trace_benchmark(*scene, diff, cam_t, start, out, weight_threshold=0.05)
    torch.cuda.synchronize()
    frame = out.cpu().numpy()
    refdata.assert_equal(frame, ref["frame"], "the frame's bytes")
    a = frame.view(np.uint8).reshape(120, 200, 4).astype(np.int32)
    assert (a[..., :3].sum(axis=-1) > 0).mean() > 0.2  # the frame is not empty


# ------------------------------------------------------------------ walk tape (record / replay)
@pytest.mark.parametrize("make_case", [("config1_deg3_q2", lambda: common.config1(3, 2))]
                         + list(LARGE_CASES.items()),
                         ids=["config1", "scene", "scene_inside", "random_batch"])
def test_tape_replay_matches_reference_kernels(torch_cuda, make_case):
    """Forward that records the tape == plain forward bit for bit; backward that replays it ==
    the reference's re-walk backward."""
    name, make = make_case
    case = make()
    got = run_ours(torch_cuda, case, tape=True)
    plain = run_ours(torch_cuda, case, tape=False)
    for k in ("rgba", "depth", "depth_indices", "num_intersections"):
        assert np.array_equal(got[k], plain[k]), k
    ref = refdata.reference(name, refdata.case_inputs(case))
    refdata.assert_forward_equal(got, ref)
    refdata.assert_grads_close(got, ref, GRAD_TOL)


def test_tape_overflow_falls_back_then_grows(torch_cuda):
    """The tape pool starts at one 32-step chunk per warp; this scene needs two.  First step:
    the pool overflows and the backward re-walks; the pool then grows and later steps replay.
    Every step must equal the reference's kernels."""
    import radfoam_b200

    torch = torch_cuda
    case = LARGE_CASES["scene60k_inside"]()
    ref = refdata.reference("scene60k_inside", refdata.case_inputs(case))
    f = case.foam
    pipe = radfoam_b200.create_pipeline(3)
    scene = [to_dev(torch, x) for x in (f.points, f.attributes, f.adjacency, f.offsets)]
    scene[0].requires_grad_(True)
    rays, start, dq = to_dev(torch, case.rays), to_dev(torch, case.start), to_dev(torch, case.quantiles)
    g, gd = to_dev(torch, case.grad_rgba), to_dev(torch, case.grad_depth)
    overflowed = []
    for step in range(3):
        fwd = pipe.trace_forward(*scene, rays, start, depth_quantiles=dq)
        overflowed.append(pipe.tape_status()["overflowed"])
        bwd = pipe.trace_backward(*scene, rays, start, fwd["rgba"], g, dq, fwd["depth_indices"], gd)
        got = {k: v.cpu().numpy() for k, v in list(fwd.items()) + list(bwd.items()) if k != "ray_grad"}
        refdata.assert_forward_equal(got, ref)
        refdata.assert_grads_close(got, ref, GRAD_TOL)
        assert got["num_intersections"].max() > 40  # equal to the reference's: the scene needs two chunks
    assert overflowed[0] and not overflowed[-1], overflowed
    st = pipe.tape_status()
    assert st["used_chunks"] <= st["capacity_chunks"]


def test_tape_is_not_replayed_for_other_rays(torch_cuda):
    """The tape is keyed on the ray / start tensors: a backward on different rays must re-walk."""
    import radfoam_b200

    torch = torch_cuda
    case = common.scene_case()
    f = case.foam
    pipe = radfoam_b200.create_pipeline(3)
    scene = [to_dev(torch, x) for x in (f.points, f.attributes, f.adjacency, f.offsets)]
    scene[0].requires_grad_(True)
    rays, start, dq = to_dev(torch, case.rays), to_dev(torch, case.start), to_dev(torch, case.quantiles)
    g, gd = to_dev(torch, case.grad_rgba), to_dev(torch, case.grad_depth)
    fwd = pipe.trace_forward(*scene, rays, start, depth_quantiles=dq)
    # same values, different tensors, mirrored image: must not use the tape of `rays`
    rays2, start2, dq2, g2, gd2 = [t.flip(1).contiguous() for t in (rays, start, dq, g, gd)]
    fwd2 = {k: v.flip(1).contiguous() for k, v in fwd.items() if k in ("rgba", "depth_indices")}
    a = pipe.trace_backward(*scene, rays2, start2, fwd2["rgba"], g2, dq2, fwd2["depth_indices"], gd2)
    b = pipe.trace_backward(*scene, rays, start, fwd["rgba"], g, dq, fwd["depth_indices"], gd)
    torch.cuda.synchronize()
    assert common.grad_error(a["attr_grad"].cpu().numpy(), b["attr_grad"].cpu().numpy()) < 1e-5
    assert common.grad_error(a["points_grad"].cpu().numpy(), b["points_grad"].cpu().numpy()) < 1e-5


# ------------------------------------------------------------------ entry cell (SURVEY.md §8f.1)
def test_nearest_point_and_starting_points(torch_cuda):
    import radfoam_b200
    from radfoam_b200 import foam

    torch = torch_cuda
    f = common.scene_case(num_points=60000, width=320, height=200).foam
    rng = np.random.default_rng(2)
    queries = np.concatenate([rng.normal(0, 2.0, size=(257, 3)), f.points[:5].astype(np.float64)]).astype(np.float32)
    got = radfoam_b200.nearest_point(to_dev(torch, f.points), to_dev(torch, queries)).cpu().numpy()
    d2 = ((f.points[None, :, :].astype(np.float64) - queries[:, None, :].astype(np.float64)) ** 2).sum(-1)
    want = d2.argmin(axis=1)
    # exact up to fp32-vs-fp64 near-ties: the chosen point must be (numerically) as close as the best
    chosen = d2[np.arange(len(queries)), got.astype(np.int64)]
    assert (chosen <= d2.min(axis=1) * (1 + 1e-5) + 1e-12).all()
    assert (got.astype(np.int64) == want).mean() > 0.99
    assert np.array_equal(got[-5:], np.arange(5))        # a point is its own nearest point
    # per-ray start cells: one frame (single origin) and a multi-camera batch
    case = common.scene_case(num_points=60000, width=320, height=200)
    sp = radfoam_b200.starting_points(to_dev(torch, case.rays), to_dev(torch, f.points))
    assert sp.dtype == torch.uint32 and sp.shape == case.start.shape
    assert np.array_equal(sp.cpu().numpy(), case.start)
    batch = common.random_ray_case(num_points=60000, num_rays=100000)
    sp = radfoam_b200.starting_points(to_dev(torch, batch.rays), to_dev(torch, batch.foam.points))
    assert np.array_equal(sp.cpu().numpy(), batch.start)


# ------------------------------------------------------------------ invariants
def test_tiled_and_linear_assignment_agree(torch_cuda):
    case = common.scene_case()
    tiled = run_ours(torch_cuda, case)
    flat = run_ours(torch_cuda, case, flat=True)
    h, w = case.rays.shape[:2]
    assert np.array_equal(tiled["num_intersections"].reshape(-1), flat["num_intersections"].reshape(-1))
    assert np.array_equal(tiled["rgba"].reshape(-1, 4), flat["rgba"].reshape(-1, 4))
    assert np.array_equal(tiled["depth"].reshape(h * w, -1), flat["depth"])
    assert common.grad_error(tiled["attr_grad"], flat["attr_grad"]) < 1e-5


def test_scene_cache_tracks_in_place_updates(torch_cuda):
    """The cached scene mirrors must be rebuilt when a scene tensor changes in place
    (optimizer.step()) and reused otherwise, with identical results either way."""
    import radfoam_b200

    torch = torch_cuda
    case = common.config1(3, 0)
    f = case.foam
    pipe = radfoam_b200.create_pipeline(3)
    pts, attrs, adj, off = [to_dev(torch, x) for x in (f.points, f.attributes, f.adjacency, f.offsets)]
    rays, start = to_dev(torch, case.rays), to_dev(torch, case.start)
    a = pipe.trace_forward(pts, attrs, adj, off, rays, start)["rgba"].clone()
    radfoam_b200.pipeline.reset_launch_count()
    b = pipe.trace_forward(pts, attrs, adj, off, rays, start)["rgba"].clone()
    assert radfoam_b200.pipeline.launch_count() == 2  # mirrors reused: only the ray kernel and its (idle) exact twin ran
    assert torch.equal(a, b)
    attrs[:, -1] *= 0.5  # in-place update bumps the version counter
    c = pipe.trace_forward(pts, attrs, adj, off, rays, start)["rgba"]
    fresh = radfoam_b200.create_pipeline(3).trace_forward(pts, attrs, adj, off, rays, start)["rgba"]
    assert torch.equal(c, fresh) and not torch.equal(a, c)


def test_backward_is_linear_in_upstream_gradient(torch_cuda):
    case = common.scene_case()
    import copy

    doubled = copy.copy(case)
    doubled.grad_rgba = case.grad_rgba * 2.0
    doubled.grad_depth = case.grad_depth * 2.0
    a, b = run_ours(torch_cuda, case), run_ours(torch_cuda, doubled)
    assert common.grad_error(b["attr_grad"], 2.0 * a["attr_grad"]) < 1e-5
    assert common.grad_error(b["points_grad"], 2.0 * a["points_grad"]) < 1e-5


def test_autograd_op_and_scrub(torch_cuda):
    """TraceRays mirror end to end + in-kernel non-finite scrub == the reference's post-pass."""
    import radfoam_b200

    torch = torch_cuda
    case = common.config1(3, 2)
    f = case.foam
    pipe = radfoam_b200.create_pipeline(3)
    pts = to_dev(torch, f.points).requires_grad_(True)
    attrs = to_dev(torch, f.attributes).requires_grad_(True)
    adj, off = to_dev(torch, f.adjacency), to_dev(torch, f.offsets)
    rgba, depth, contrib, nint, errbox = radfoam_b200.TraceRays.apply(
        pipe, pts, attrs, adj, off, to_dev(torch, case.rays), to_dev(torch, case.start),
        to_dev(torch, case.quantiles), False)
    assert contrib is None and nint.dtype == torch.uint32
    loss = (rgba * to_dev(torch, case.grad_rgba)).sum() + (depth * to_dev(torch, case.grad_depth)).sum()
    loss.backward()
    ref = run_cpu_oracle(case)
    for got, want in ((pts.grad, ref["points_grad"]), (attrs.grad, ref["attr_grad"])):
        assert torch.isfinite(got).all()
        want = np.where(np.isfinite(want), want, 0.0)
        assert common.grad_error(got.cpu().numpy(), want) < common.CPU_GRAD_TOL


def test_empty_ray_batch(torch_cuda):
    import radfoam_b200

    torch = torch_cuda
    f = common.config1(3, 0).foam
    pipe = radfoam_b200.create_pipeline(3)
    scene = [to_dev(torch, x) for x in (f.points, f.attributes, f.adjacency, f.offsets)]
    rays = torch.empty((0, 6), device="cuda")
    start = torch.empty((0,), dtype=torch.uint32, device="cuda")
    out = pipe.trace_forward(*scene, rays, start)
    assert out["rgba"].shape == (0, 4) and out["num_intersections"].shape == (0, 1)
    bwd = pipe.trace_backward(*scene, rays, start, out["rgba"], torch.empty((0, 4), device="cuda"))
    assert float(bwd["attr_grad"].abs().sum()) == 0.0 and float(bwd["points_grad"].abs().sum()) == 0.0


def test_validation_errors(torch_cuda):
    import radfoam_b200

    torch = torch_cuda
    case = common.config1(3, 0)
    f = case.foam
    pipe = radfoam_b200.create_pipeline(3)
    pts, attrs, adj, off = [to_dev(torch, x) for x in (f.points, f.attributes, f.adjacency, f.offsets)]
    rays, start = to_dev(torch, case.rays), to_dev(torch, case.start)
    with pytest.raises(RuntimeError, match="Unsupported SH degree"):
        radfoam_b200.create_pipeline(4)
    with pytest.raises(RuntimeError, match="Unsupported attribute type"):
        radfoam_b200.create_pipeline(3, "float64")
    with pytest.raises(RuntimeError, match="expected 49"):
        pipe.trace_forward(pts, attrs[:, :28].contiguous(), adj, off, rays, start)
    with pytest.raises(RuntimeError, match="uint32"):
        pipe.trace_forward(pts, attrs, adj.to(torch.int32), off, rays, start)
    with pytest.raises(RuntimeError, match="start_point must have the same batch size"):
        pipe.trace_forward(pts, attrs, adj, off, rays, start[:4])
    with pytest.raises(RuntimeError, match="CUDA device"):
        pipe.trace_forward(pts.cpu(), attrs, adj, off, rays, start)
    with pytest.raises(RuntimeError, match="rays must have 6"):
        pipe.trace_forward(pts, attrs, adj, off, rays[..., :5], start)


# ------------------------------------------------------------------ .pt checkpoint -> FPS loop (SURVEY.md §8f.3)
def pt_checkpoint_world(torch, directory):
    """A scene saved in the reference's .pt layout and loaded as benchmark.py:36-38 does (fp16 attributes), the
    cameras of benchmark.py's FPS loop, and what a direct trace_benchmark call of each camera needs."""
    import radfoam_b200
    from radfoam_b200 import foam, scene_io

    f = common.scene_case().foam
    path = os.path.join(directory, "model.pt")
    scene_io.FoamScene.from_foam(f, device="cpu").save_pt(path)
    scene = scene_io.FoamScene.load_pt(path, sh_degree=3, attr_dtype=torch.float16, device="cuda")
    width, height, fov = 160, 96, 0.9
    c2w = torch.zeros((17, 4, 4))
    for i in range(17):
        ang = 0.37 * i
        pos = (3.2 * np.cos(ang), 3.2 * np.sin(ang), 1.5)
        cam = foam.camera_dict(pos, fov=fov, width=width, height=height)
        c2w[i, :3, 0] = torch.from_numpy(cam["right"])
        c2w[i, :3, 1] = -torch.from_numpy(cam["up"])
        c2w[i, :3, 2] = torch.from_numpy(cam["forward"])
        c2w[i, :3, 3] = torch.from_numpy(cam["position"])
        c2w[i, 3, 3] = 1.0
    fy = height / (2.0 * np.tan(fov / 2.0))
    cameras, positions = scene_io.benchmark_cameras(c2w, fy, width, height)
    pipe = radfoam_b200.create_pipeline(3, "float16")
    trace_data = scene.get_trace_data()
    points, _, adjacency, offsets = trace_data
    return dict(scene=scene, width=width, height=height, fov=fov, cameras=cameras, positions=positions, pipe=pipe,
                trace_data=trace_data, diff=pipe.prefetch_adjacent_diff(points, adjacency, offsets),
                starts=radfoam_b200.nearest_point(points, positions.cuda()))


def pt_checkpoint_inputs(w):
    return w["trace_data"], w["cameras"], w["starts"], w["diff"]


def test_pt_checkpoint_benchmark_loop(torch_cuda, tmp_path):
    """A scene saved in the reference's .pt layout, loaded as benchmark.py:36-38 does (fp16 attributes), rendered
    through the FPS loop of benchmark.py:86-139; frames must equal direct trace_benchmark calls and the reference
    kernel's frames, byte for byte."""
    from radfoam_b200 import scene_io

    torch = torch_cuda
    w = pt_checkpoint_world(torch, tmp_path)
    height, width, cameras, pipe = w["height"], w["width"], w["cameras"], w["pipe"]
    assert len(cameras) == 3 and abs(cameras[0]["fov"] - w["fov"]) < 1e-6
    res = scene_io.benchmark_fps(pipe, w["scene"], cameras, w["positions"], n_reps=2)
    assert res["frames"] == 3 and res["fps"] > 0 and res["output"].shape == (3, height, width)
    frames = res["output"].cpu().numpy()
    assert w["trace_data"][1].dtype == torch.float16
    ref = refdata.reference("pt_checkpoint_frames", pt_checkpoint_inputs(w))
    for k in range(3):
        direct = torch.zeros((height, width), dtype=torch.uint32, device="cuda")
        pipe.trace_benchmark(*w["trace_data"], w["diff"], cameras[k], w["starts"][k:k + 1], direct,
                             weight_threshold=0.05)
        assert np.array_equal(frames[k], direct.cpu().numpy())
        a = frames[k].view(np.uint8).reshape(height, width, 4).astype(np.int32)
        assert (a[..., :3].sum(axis=-1) > 0).mean() > 0.05         # the frame is not empty
        refdata.assert_equal(frames[k], ref[f"frame{k}"], f"frame {k}'s bytes")
