"""Parity AT THE SIZES THE METRIC IS QUOTED ON (BASELINE.json configs 3, 4 and the step-budget / 4K edge of
config 5), against the reference's own kernels (their outputs stored in tests/golden/reference/kernels.npz), through
the public autograd op with the walk tape on -- i.e. the exact path bench.py times:
  * config 4: 1,048,576-point foam, 1920x1080, Q = 2, fwd+bwd                       (the headline)
  * config 3: 2,097,152-point foam, 1920x1080, Q = 2, fwd+bwd
  * config 5's edges on the 2 M foam: a 3840x2160 frame (8.3 M rays) with max_intersections low enough that a
    large share of the rays runs out of step budget (n = max + 1), plus the default budget.
    (The full 4 M-point / 4K run is too slow to build under the driver -- Qhull needs ~2.5 min for 4 M points;
    it is run by tests/tools/configs_bench.py and recorded in profiles/.)
Bars: integer outputs equal; rgba / depth <= 1e-5; gradients <= 1e-5 of max|ref|.
The foams are cached where bench.py caches them (bench.load_or_build_foam)."""
import numpy as np
import pytest

import refdata

pytestmark = pytest.mark.gpu

CAMERA = (2.5, 2.5, 2.5)


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


# stored case -> (points, width, height, max_intersections)
STEPS = {"config4_1m_1080p": (1_048_576, 1920, 1080, None),
         "config3_2m_1080p": (2_097_152, 1920, 1080, None),
         "config5_2m_4k_max96": (2_097_152, 3840, 2160, 96),
         "config5_2m_4k": (2_097_152, 3840, 2160, None)}


_foams = {}


def scene_tensors(torch, num_points):
    if num_points not in _foams:
        import bench

        f = bench.load_or_build_foam(num_points, lambda m: None)
        d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
        _foams.clear()  # one foam resident at a time
        _foams[num_points] = (f, [d(f.points), d(f.attributes), d(f.adjacency), d(f.offsets)])
    return _foams[num_points]


def frame_tensors(torch, f, width, height, seed):
    from radfoam_b200 import foam

    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    rays = d(foam.pinhole_rays(width, height, CAMERA, fov=0.9))
    start = torch.full((height, width), int(foam.nearest_point(f.points, CAMERA)), dtype=torch.int64,
                       device="cuda").to(torch.uint32)
    gen = torch.Generator(device="cuda").manual_seed(seed)
    dq = torch.rand((height, width, 2), generator=gen, device="cuda").sort(dim=-1, descending=True).values.contiguous()
    g = torch.randn((height, width, 4), generator=gen, device="cuda")
    gd = torch.randn((height, width, 2), generator=gen, device="cuda") * 1e-4
    return rays, start, dq, g, gd


def check_step(torch, name, expect_budget_hits=False):
    import radfoam_b200

    num_points, width, height, max_intersections = STEPS[name]
    f, scene = scene_tensors(torch, num_points)
    rays, start, dq, g, gd = frame_tensors(torch, f, width, height, seed=num_points % 1000 + width)
    kw = {} if max_intersections is None else {"max_intersections": max_intersections}

    # The reference's gradients (non-finite entries zeroed, radfoam_model/render.py:98-99) are float atomicAdd sums
    # whose order changes from run to run; per-point position gradients cancel ~1e3x, so with 8.3 M rays the reference
    # differs from ITSELF by up to ~1e-5 of max.  The bar is the north star's 1e-5, widened to 4x the reference's own
    # run-to-run difference (measured when its outputs were stored) where that is larger.
    ref = refdata.reference(name, (scene, rays, start, dq, g, gd))
    noise = {k: ref["noise_" + k] for k in ("points_grad", "attr_grad")}

    pipe = radfoam_b200.create_pipeline(3, "float32")
    points = scene[0].detach().clone().requires_grad_(True)
    attrs = scene[1].detach().clone().requires_grad_(True)
    if max_intersections is None:
        rgba, depth, _, nint, _ = radfoam_b200.TraceRays.apply(pipe, points, attrs, scene[2], scene[3], rays, start,
                                                               dq, False)
        ((rgba * g).sum() + (depth * gd).sum()).backward()
        assert pipe.tape_status()["used_chunks"] > 0  # the recording forward ran (and a replay, unless it overflowed)
        didx = None
        pg, ag = points.grad, attrs.grad
        rgba, depth = rgba.detach(), depth.detach()
    else:  # trace settings are not part of the autograd op's contract: drive the pipeline directly
        fwd = pipe.trace_forward(points, attrs, scene[2], scene[3], rays, start, depth_quantiles=dq, **kw)
        bwd = pipe.trace_backward(points, attrs, scene[2], scene[3], rays, start, fwd["rgba"], g, dq,
                                  fwd["depth_indices"], gd, scrub_nonfinite=True, **kw)
        rgba, depth, nint, didx = fwd["rgba"], fwd["depth"], fwd["num_intersections"], fwd["depth_indices"]
        pg, ag = bwd["points_grad"], bwd["attr_grad"]

    refdata.assert_equal(nint.cpu().numpy(), ref["num_intersections"], "num_intersections")
    if didx is not None:
        refdata.assert_equal(didx.cpu().numpy(), ref["depth_indices"], "depth_indices")
    n = nint.to(torch.int64)
    if expect_budget_hits:
        assert float((n == max_intersections + 1).float().mean()) > 0.2, "the case must exhaust the step budget"
    refdata.assert_close(rgba.cpu().numpy(), ref["rgba"], "rgba", rtol=0, atol=1e-5)
    refdata.assert_close(depth.cpu().numpy(), ref["depth"], "depth", rtol=0, atol=1e-5 * max(1.0, ref["depth"].scale))
    for k, got in (("points_grad", pg), ("attr_grad", ag)):
        err = refdata.grad_error(got.cpu().numpy(), ref[k])
        assert err <= max(1e-5, 4.0 * noise[k]), f"{k}: {err:.3g} of max|ref| (reference vs itself: {noise[k]:.3g})"
    return float(n.float().mean()), int(n.max())


def test_config4_headline_1m_points_1080p(torch_cuda):
    mean_cells, _ = check_step(torch_cuda, "config4_1m_1080p")
    assert 60 < mean_cells < 140  # bench.py reports 97.3 for this frame


def test_config3_2m_points_1080p(torch_cuda):
    check_step(torch_cuda, "config3_2m_1080p")


def test_config5_edges_4k_frame_and_step_budget(torch_cuda):
    _, n_max = check_step(torch_cuda, "config5_2m_4k_max96", expect_budget_hits=True)
    assert n_max == 97
    check_step(torch_cuda, "config5_2m_4k")
