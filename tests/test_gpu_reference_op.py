"""Drop-in boundary: the REFERENCE'S OWN autograd op -- radfoam_model/render.py::TraceRays, unmodified --
driving radfoam_b200.Pipeline, and radfoam_b200's own ops, compared with what the reference's op returned on the
reference's own kernels (stored in tests/golden/reference/kernels.npz by tests/golden/make_golden_reference.py).

The reference's file is not part of this repository: the two tests that run it need its byte-compiled copy
oracle/_ref/radfoam_model_render.pyc, which __graft_entry__.build() makes (`make -C oracle ref_py`) where the original
project's sources are present (and which travels with oracle/_ref to wherever that was built); on a clean checkout
they skip.  Nothing of it is re-typed here."""
import importlib.machinery
import importlib.util
import os

import numpy as np
import pytest

import common
import refdata

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_PYC = os.path.join(ROOT, "oracle", "_ref", "radfoam_model_render.pyc")


def load_reference_op():
    if not os.path.exists(REF_PYC):
        pytest.skip("oracle/_ref/radfoam_model_render.pyc was not built (the original project's sources were absent)")
    loader = importlib.machinery.SourcelessFileLoader("radfoam_reference_render", REF_PYC)
    spec = importlib.util.spec_from_loader(loader.name, loader)
    mod = importlib.util.module_from_spec(spec)
    loader.exec_module(mod)
    return mod


class ReferencePipeline:
    """The reference's kernels behind the dict API its pybind module gives render.py (tests/golden/
    make_golden_reference.py drives the reference's op with it)."""

    def __init__(self):
        from oracle import ref_gpu

        if not ref_gpu.available():
            pytest.skip("oracle/_ref not built")
        self.ref = ref_gpu

    def trace_forward(self, *args, **kwargs):
        return self.ref.trace_forward(*args, **kwargs)

    def trace_backward(self, *args, **kwargs):
        return self.ref.trace_backward(*args, **kwargs)


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def drive(torch, op, pipeline, case, with_error, contribution=False):
    """One training-shaped step through `op` (an autograd Function with the reference's contract)."""
    f = case.foam
    dev = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    points = dev(f.points).requires_grad_(True)
    base = dev(f.attributes).requires_grad_(True)
    attributes = base * 1.0  # a non-leaf, like get_trace_data()'s cat (scene.py:202-217)
    out = op.apply(pipeline, points, attributes, dev(f.adjacency), dev(f.offsets), dev(case.rays), dev(case.start),
                   dev(case.quantiles), contribution)
    rgba, depth, contrib, nint, box = out
    if with_error:
        rng = np.random.default_rng(3)
        box.ray_error = dev(rng.uniform(0.0, 1.0, size=case.rays.shape[:-1] + (1,)).astype(np.float32))
    loss = (rgba * dev(case.grad_rgba)).sum()
    if depth is not None:
        loss = loss + (depth * dev(case.grad_depth)).sum()
    loss.backward()
    res = {"rgba": rgba.detach(), "num_intersections": nint, "points_grad": points.grad, "attr_grad": base.grad}
    if depth is not None:
        res["depth"] = depth.detach()
    if contrib is not None:
        res["contribution"] = contrib.detach()
    if with_error:
        res["point_error"] = box.point_error
    return {k: v.cpu().numpy() for k, v in res.items()}


def compare_stored(got, ref):
    """got against the stored outputs of the reference's op (tests/refdata.py): integers bit-exact, rgba / depth within
    1e-5, gradients / error / contribution within 1e-5 of max|ref| with the same non-finite pattern."""
    refdata.assert_equal(got["num_intersections"], ref["num_intersections"], "num_intersections")
    refdata.assert_close(got["rgba"], ref["rgba"], "rgba")
    if "depth" in ref:
        refdata.assert_close(got["depth"], ref["depth"], "depth")
    for k in ("points_grad", "attr_grad", "point_error", "contribution"):
        if k in ref:
            assert ref[k].same_nonfinite(got[k]), k
            assert refdata.grad_error(got[k], ref[k]) <= 1e-5, k


@pytest.mark.parametrize("with_error", [False, True])
def test_reference_render_op_runs_unmodified_on_our_pipeline(torch_cuda, with_error):
    import radfoam_b200

    mod = load_reference_op()
    case = common.scene_case(20000, 160, 96, q=2)
    ours = drive(torch_cuda, mod.TraceRays, radfoam_b200.create_pipeline(3, "float32"), case, with_error)
    compare_stored(ours, refdata.reference(f"reference_op_error{int(with_error)}_contribution0",
                                           refdata.case_inputs(case)))


def test_reference_render_op_records_the_walk_tape(torch_cuda):
    """Inside the reference's Function.forward grad mode is off; the pipeline must still see that a backward is
    coming (attributes is a non-leaf that requires grad) and replay the tape -- and must NOT record under no_grad."""
    import radfoam_b200

    torch = torch_cuda
    mod = load_reference_op()
    case = common.scene_case(20000, 160, 96, q=2)
    pipe = radfoam_b200.create_pipeline(3, "float32")
    drive(torch, mod.TraceRays, pipe, case, False)
    assert pipe.tape_status()["used_chunks"] > 0
    pipe2 = radfoam_b200.create_pipeline(3, "float32")
    f = case.foam
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    points = torch.nn.Parameter(dev(f.points))
    with torch.no_grad():  # eval render of the reference: attributes are built under no_grad
        attributes = dev(f.attributes) * 1.0
        mod.TraceRays.apply(pipe2, points, attributes, dev(f.adjacency), dev(f.offsets), dev(case.rays),
                            dev(case.start), None, False)
    with pytest.raises(RuntimeError, match="no recorded tape"):
        pipe2.tape_status()


@pytest.mark.parametrize("with_error", [False, True])
def test_native_op_matches_reference_op(torch_cuda, with_error):
    """radfoam_b200.TraceRays (written independently: save_for_backward, in-kernel scrub) == the reference's op."""
    import radfoam_b200

    case = common.scene_case(20000, 160, 96, q=2)
    ours = drive(torch_cuda, radfoam_b200.TraceRays, radfoam_b200.create_pipeline(3, "float32"), case, with_error,
                 contribution=True)
    compare_stored(ours, refdata.reference(f"reference_op_error{int(with_error)}_contribution1",
                                           refdata.case_inputs(case)))


def test_native_op_leaves_no_reference_cycle(torch_cuda):
    """The step's graph must die by reference counting (no tensor -> grad_fn -> ctx -> tensor cycle)."""
    import gc
    import weakref

    import radfoam_b200

    torch = torch_cuda
    case = common.config1()
    f = case.foam
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    pipe = radfoam_b200.create_pipeline(3, "float32")
    points, attrs = dev(f.points).requires_grad_(True), dev(f.attributes).requires_grad_(True)
    gc.disable()
    try:
        rgba, depth, _, _, _ = radfoam_b200.TraceRays.apply(pipe, points, attrs, dev(f.adjacency), dev(f.offsets),
                                                            dev(case.rays), dev(case.start), dev(case.quantiles), False)
        ref = weakref.ref(rgba)
        (rgba.sum() + depth.sum()).backward()
        del rgba, depth
        assert ref() is None, "rgba survived: a reference cycle keeps the step's tensors alive until gc runs"
    finally:
        gc.enable()


@pytest.mark.parametrize("attr_dtype", ["float32", "float16"])
def test_parameter_form_scene_equals_torch_glue(torch_cuda, attr_dtype):
    """SURVEY.md §8f.2: get_trace_data's cat + softplus (scene.py:202-217) and the gradient split back through them,
    fused into the re-layout / finalize kernels (TraceRaysParams), against the same thing done with torch ops
    around TraceRays -- values and all four parameter gradients."""
    import radfoam_b200
    from radfoam_b200 import scene_io

    torch = torch_cuda
    case = common.scene_case(20000, 160, 96, q=2)
    dt = torch.float16 if attr_dtype == "float16" else torch.float32
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    results = []
    for fused in (False, True):
        scene = scene_io.FoamScene.from_foam(case.foam, device="cuda", activation_scale=1.7)
        scene.attr_dtype = dt
        params = [scene.primal_points, scene.att_dc, scene.att_sh, scene.density]
        for t in params:
            t.requires_grad_(True)
        pipe = radfoam_b200.create_pipeline(3, attr_dtype)
        rays, start = dev(case.rays), dev(case.start)
        if fused:
            out = radfoam_b200.TraceRaysParams.apply(pipe, *params, scene.activation_scale, scene.point_adjacency,
                                                     scene.point_adjacency_offsets, rays, start, dev(case.quantiles),
                                                     False)
        else:
            points, attributes, adjacency, offsets = scene.get_trace_data()
            out = radfoam_b200.TraceRays.apply(pipe, points, attributes, adjacency, offsets, rays, start,
                                               dev(case.quantiles), False)
        rgba, depth, _, nint, _ = out
        g = dev(case.grad_rgba).to(dt)
        ((rgba * g).sum().float() + (depth * dev(case.grad_depth)).sum()).backward()
        results.append(dict(rgba=rgba.detach().float(), depth=depth.detach(), nint=nint,
                            grads=[t.grad.clone() for t in params]))
    a, b = results
    assert torch.equal(a["nint"], b["nint"])
    assert torch.equal(a["rgba"], b["rgba"]) and torch.equal(a["depth"], b["depth"])  # same attribute values, bit for bit
    for name, ga, gb in zip(("points", "att_dc", "att_sh", "density"), a["grads"], b["grads"]):
        assert ga.shape == gb.shape
        err = float((ga - gb).abs().max() / ga.abs().max().clamp_min(1e-30))
        # fp16 pipelines round the attribute gradient to half once (1e-3 relative); the two runs sum their fp32
        # accumulators in different atomic orders, so the rounded values may differ by one half-ulp
        assert err <= (1e-5 if attr_dtype == "float32" or name == "points" else 2e-3), f"{name}: {err:.3g}"


def test_training_step_is_cuda_graph_capturable(torch_cuda):
    """SURVEY.md §7: the path must be graph-capturable.  Re-layout + recording forward + replaying backward +
    finalize of one step are captured into a CUDA graph (after a warm-up step sized the library's buffers) and
    replayed on new parameter values; the replay must equal an eager step on the same values."""
    import radfoam_b200

    torch = torch_cuda
    case = common.scene_case(20000, 160, 96, q=2)
    f = case.foam
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    points, attrs = dev(f.points).requires_grad_(True), dev(f.attributes).requires_grad_(True)
    adj, off, rays, start, dq = dev(f.adjacency), dev(f.offsets), dev(case.rays), dev(case.start), dev(case.quantiles)
    g, gd = dev(case.grad_rgba), dev(case.grad_depth)
    pipe = radfoam_b200.create_pipeline(3, "float32")

    def step():
        pipe.invalidate_cache()  # parameters changed
        fwd = pipe.trace_forward(points, attrs, adj, off, rays, start, depth_quantiles=dq)
        bwd = pipe.trace_backward(points, attrs, adj, off, rays, start, fwd["rgba"], g, dq, fwd["depth_indices"], gd,
                                  scrub_nonfinite=True)
        return fwd["rgba"], bwd["points_grad"], bwd["attr_grad"]

    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        for _ in range(3):  # sizes the tape pool, the mirrors and the accumulator
            step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_out = step()
    with torch.no_grad():  # "optimizer step": new values in the SAME tensors
        attrs[:, :48] *= 0.9
        points += 1e-4
    graph.replay()
    torch.cuda.synchronize()
    got = [t.clone() for t in static_out]
    want = step()
    torch.cuda.synchronize()
    assert torch.equal(got[0], want[0])
    for a, b in zip(got[1:], want[1:]):
        assert float((a - b).abs().max() / b.abs().max()) <= 1e-5


def error_map_world(torch):
    """Three views of the 20k-point scene, target colours, and the scene in parameter form (trainable)."""
    from radfoam_b200 import foam, scene_io

    f = common.scene_case(20000, 160, 96, q=2).foam
    views, height, width = 3, 48, 80
    cams = [(2.5, 2.5, 2.5), (-2.5, 2.0, 1.5), (0.5, -3.0, 2.0)]
    rays = torch.from_numpy(np.stack([foam.pinhole_rays(width, height, c, fov=0.9) for c in cams]))
    rgbs = torch.rand((views, height, width, 3), generator=torch.Generator().manual_seed(5))
    scene = scene_io.FoamScene.from_foam(f, device="cuda")
    for t in (scene.primal_points, scene.att_dc, scene.att_sh, scene.density):
        t.requires_grad_(True)
    return dict(foam=f, cams=cams, rays=rays, rgbs=rgbs, scene=scene)


def error_map_inputs(w):
    f = w["foam"]
    return f.points, f.attributes, f.adjacency, f.offsets, w["rays"], w["rgbs"], w["cams"]


def our_error_map(torch, w):
    import radfoam_b200

    pipe = radfoam_b200.create_pipeline(3, "float32")
    return w["scene"].collect_error_map(pipe, w["rays"], w["rgbs"], generator=torch.Generator().manual_seed(9))


def test_collect_error_map_matches_the_reference_loop(torch_cuda):
    """SURVEY.md §8f.4: the densification pass's error map (scene.py:497-548) through FoamScene.collect_error_map
    (parameter-form scene, device-side start points) against the same loop spelled out with the reference's own
    autograd op on the reference's own kernels (tests/golden/make_golden_reference.py ran that loop)."""
    w = error_map_world(torch_cuda)
    ref = refdata.reference("collect_error_map", error_map_inputs(w))
    err, contrib = our_error_map(torch_cuda, w)
    assert refdata.grad_error(err.cpu().numpy(), ref["error"]) <= 1e-5
    assert refdata.grad_error(contrib.cpu().numpy(), ref["contribution"]) <= 1e-5
    assert float((contrib > 0).float().mean()) > 0.02
