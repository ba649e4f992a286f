"""BASELINE.json-sized cases on the GPU (config 2: ~0.5 M points, one 1920x1080 frame), checked
through size-independent properties of the path plus against the reference's own kernels (their outputs stored in
tests/golden/reference/kernels.npz).  The foam build (Qhull) dominates the run time (~20 s)."""
import numpy as np
import pytest

import common
import refdata

pytestmark = pytest.mark.gpu

N_POINTS = 524_288
W, H = 1920, 1080


def inputs(torch):
    """The seeded frame: scene tensors, rays, start cells, quantiles and upstream gradients on the GPU."""
    from radfoam_b200 import foam

    f = foam.scene_foam(N_POINTS)
    pos = (2.5, 2.5, 2.5)
    rays = foam.pinhole_rays(W, H, pos, fov=0.9)
    start = np.full((H, W), foam.nearest_point(f.points, pos), dtype=np.uint32)
    rng = np.random.default_rng(9)
    dq = np.sort(rng.uniform(0, 1, size=(H, W, 2)).astype(np.float32), axis=-1)[..., ::-1].copy()
    g = rng.normal(size=(H, W, 4)).astype(np.float32)
    gd = (rng.normal(size=(H, W, 2)) * 1e-4).astype(np.float32)
    d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()  # noqa: E731
    return dict(foam=f, scene=[d(f.points), d(f.attributes), d(f.adjacency), d(f.offsets)],
                rays=d(rays), start=d(start), dq=d(dq), g=d(g), gd=d(gd))


def inputs_of(w):
    return w["scene"], w["rays"], w["start"], w["dq"], w["g"], w["gd"]


@pytest.fixture(scope="module")
def world():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import radfoam_b200

    w = dict(inputs(torch), torch=torch, pipe=radfoam_b200.create_pipeline(3))
    w["pipe"].record_tape = False
    w["fwd"] = w["pipe"].trace_forward(*w["scene"], w["rays"], w["start"], depth_quantiles=w["dq"])
    return w


def _bwd(w, pipe=None, rows=slice(None), scale=1.0, fwd=None):
    pipe = pipe or w["pipe"]
    fwd = fwd or w["fwd"]
    return pipe.trace_backward(*w["scene"], w["rays"][rows].contiguous(), w["start"][rows].contiguous(),
                               fwd["rgba"][rows].contiguous(), (w["g"][rows] * scale).contiguous(),
                               w["dq"][rows].contiguous(), fwd["depth_indices"][rows].contiguous(),
                               (w["gd"][rows] * scale).contiguous())


def test_forward_invariants(world):
    torch, fwd = world["torch"], world["fwd"]
    rgba, n = fwd["rgba"], fwd["num_intersections"].to(torch.int64)
    assert torch.isfinite(rgba).all()
    assert (rgba[..., 3] >= 0).all() and (rgba[..., 3] <= 1).all() and (rgba[..., :3] >= 0).all()
    assert n.min() >= 1 and n.max() <= 1025 and n.float().mean() > 20
    idx = fwd["depth_indices"].to(torch.int64)
    valid = idx != common.NONE
    assert (fwd["depth"][~valid] == -1).all() and (fwd["depth"][valid] >= 0).all()
    both = valid.all(dim=-1)
    assert (fwd["depth"][both][:, 0] <= fwd["depth"][both][:, 1]).all()  # quantiles are sorted descending
    again = world["pipe"].trace_forward(*world["scene"], world["rays"], world["start"], depth_quantiles=world["dq"])
    for k in ("rgba", "depth"):
        assert torch.equal(again[k], fwd[k])  # the forward is deterministic
    flat = world["pipe"].trace_forward(*world["scene"], world["rays"].reshape(-1, 6), world["start"].reshape(-1),
                                       depth_quantiles=world["dq"].reshape(-1, 2))
    assert torch.equal(flat["rgba"].reshape(H, W, 4), fwd["rgba"])  # tiling does not change results
    assert torch.equal(flat["num_intersections"].reshape(H, W, 1).to(torch.int64), n)


def test_contribution_sums_to_opacity(world):
    torch = world["torch"]
    out = world["pipe"].trace_forward(*world["scene"], world["rays"], world["start"], return_contribution=True)
    total = float(out["contribution"].double().sum())
    assert abs(total - float(out["rgba"][..., 3].double().sum())) <= 1e-4 * total


def test_backward_linear_additive_and_tape_equal(world):
    import radfoam_b200

    torch = world["torch"]
    full = _bwd(world)
    twice = _bwd(world, scale=2.0)
    top, bottom = _bwd(world, rows=slice(0, H // 2)), _bwd(world, rows=slice(H // 2, H))
    for k in ("points_grad", "attr_grad"):
        a = full[k].cpu().numpy()
        assert common.grad_error(twice[k].cpu().numpy(), 2.0 * a) < 1e-5            # linear in dL/dout
        assert common.grad_error((top[k] + bottom[k]).cpu().numpy(), a) < 1e-5      # rays shard additively
    # recording forward + replaying backward == plain forward + re-walk backward
    pipe = radfoam_b200.create_pipeline(3)
    scene = list(world["scene"])
    scene[0] = scene[0].detach().clone().requires_grad_(True)
    fwd = pipe.trace_forward(*scene, world["rays"], world["start"], depth_quantiles=world["dq"])
    assert torch.equal(fwd["rgba"], world["fwd"]["rgba"]) and torch.equal(fwd["depth"], world["fwd"]["depth"])
    rep = pipe.trace_backward(*scene, world["rays"], world["start"], fwd["rgba"], world["g"], world["dq"],
                              fwd["depth_indices"], world["gd"])
    for k in ("points_grad", "attr_grad"):
        assert common.grad_error(rep[k].cpu().numpy(), full[k].cpu().numpy()) < 1e-5


def test_matches_reference_kernels_at_full_size(world):
    ref = refdata.reference("config2_512k_1080p", inputs_of(world))
    fwd = {k: v.cpu().numpy() for k, v in world["fwd"].items()}
    refdata.assert_equal(fwd["num_intersections"], ref["num_intersections"], "num_intersections")  # bit-exact
    refdata.assert_equal(fwd["depth_indices"], ref["depth_indices"], "depth_indices")
    refdata.assert_close(fwd["rgba"], ref["rgba"], "rgba", rtol=0, atol=1e-5)
    refdata.assert_close(fwd["depth"], ref["depth"], "depth", rtol=0, atol=1e-5 * float(np.abs(fwd["depth"]).max()))
    ours = _bwd(world)
    for k in ("points_grad", "attr_grad"):
        assert refdata.grad_error(ours[k].cpu().numpy(), ref[k]) < 1e-5
