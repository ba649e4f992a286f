"""GPU parity of farthest_neighbor (SURVEY.md §8f.4) through the public wrapper -> ctypes -> C ABI, against the
CPU oracle and the reference's own kernel (its outputs stored in tests/golden/reference/kernels.npz).  Bar: both outputs bit-exact (integers,
and floats -- IEEE sqrt/divide with the fma association pinned; NaNs match as NaNs)."""
import numpy as np
import pytest

import common
import refdata

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch


def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def ours(torch, f):
    import radfoam_b200

    idx, radius = radfoam_b200.farthest_neighbor(dev(torch, f.points), dev(torch, f.adjacency), dev(torch, f.offsets))
    assert idx.dtype == torch.uint32 and radius.dtype == torch.float32
    assert idx.shape == radius.shape == (f.points.shape[0],)
    return idx.cpu().numpy(), radius.cpu().numpy()


@pytest.mark.parametrize("make", ["edge", "config1", "scene20k", "scene200k"])
def test_matches_oracle_bit_exact(torch_cuda, make):
    from oracle import oracle
    from radfoam_b200 import foam

    f = {"edge": common.farthest_edge_case,
         "config1": lambda: foam.small_foam(256),
         "scene20k": lambda: common.scene_case(20000, 8, 8, 0).foam,
         "scene200k": lambda: common.scene_case(200000, 8, 8, 0).foam}[make]()
    idx, radius = ours(torch_cuda, f)
    ref_idx, ref_radius = oracle.farthest_neighbor(f.points, f.adjacency, f.offsets)
    assert np.array_equal(idx, ref_idx)
    common.assert_same_floats(radius, ref_radius)


@pytest.mark.parametrize("make", ["edge", "scene200k"])
def test_matches_reference_kernel_bit_exact(torch_cuda, make):
    f = common.farthest_edge_case() if make == "edge" else common.scene_case(200000, 8, 8, 0).foam
    idx, radius = ours(torch_cuda, f)
    ref = refdata.reference(f"farthest_{make}", (f.points, f.adjacency, f.offsets))
    refdata.assert_equal(idx, ref["indices"], "indices")
    refdata.assert_equal(radius, ref["radius"], "radius")  # bit for bit, any NaN matching any NaN


def test_validation_and_empty(torch_cuda):
    import radfoam_b200

    torch = torch_cuda
    f = common.farthest_edge_case()
    p, a, o = dev(torch, f.points), dev(torch, f.adjacency), dev(torch, f.offsets)
    with pytest.raises(RuntimeError, match="unsupported scalar type"):
        radfoam_b200.farthest_neighbor(p.double(), a, o)
    with pytest.raises(RuntimeError, match="uint32"):
        radfoam_b200.farthest_neighbor(p, a.to(torch.int64), o)
    with pytest.raises(RuntimeError, match="num_points \\+ 1"):
        radfoam_b200.farthest_neighbor(p, a, o[:-1])
    idx, radius = radfoam_b200.farthest_neighbor(p[:0], a[:0], o[:1])
    assert idx.numel() == 0 and radius.numel() == 0
    # what prune_and_densify does with the result (scene.py:439, 461): index the points with it
    idx, radius = radfoam_b200.farthest_neighbor(p[40:] * 1, *_rebased(torch, f, 40))
    assert int(idx.to(torch.int64).max()) < p.shape[0] - 40


def _rebased(torch, f, first):
    """CSR of rows first.. with neighbour ids shifted to the sliced point array (rows >= 40 of the edge case only
    reference points >= 40)."""
    off = f.offsets[first:].astype(np.int64) - int(f.offsets[first])
    adj = f.adjacency[int(f.offsets[first]):].astype(np.int64) - first
    return dev(torch, adj.astype(np.uint32)), dev(torch, off.astype(np.uint32))
