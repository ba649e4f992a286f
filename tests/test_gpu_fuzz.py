"""Tie-heavy differential cases (tests/fuzz_cases.py) on the device: the sm_100a path through Pipeline -> ctypes ->
C ABI against the reference's own kernels, through their outputs stored in tests/golden/reference/kernels.npz (whole
forward outputs by hash; gradients at their largest and a spread of other entries: tests/refdata.py).  Forward outputs must be identical value for
value (integers and floats: the arithmetic of the walk is pinned to the reference's instruction sequence, and ties are
where a different association would pick another face); gradients within 2e-5 of max|ref| (float scatter-adds in both)
with identical non-finite patterns.  Odd seeds replay the recorded walk tape, even seeds re-walk.

`python tests/test_gpu_fuzz.py FIRST_SEED COUNT` runs a longer campaign: seeds without stored outputs are compared
with the reference's kernels run live, which needs oracle/_ref (built where the original project's sources are)."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import common  # noqa: E402
import fuzz_cases  # noqa: E402
import refdata  # noqa: E402
import test_gpu_parity as parity  # noqa: E402
from test_gpu_parity import torch_cuda  # noqa: E402,F401  (fixture)

pytestmark = pytest.mark.gpu


def live_reference(case, kw):
    """The reference's kernels run now, on every entry (oracle/_ref must have been built)."""
    from oracle import ref_gpu

    if not ref_gpu.available():
        raise SystemExit("no stored reference outputs for this seed (0-239 are stored), and oracle/_ref was not built "
                         "to run the reference's kernels live")
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_golden_reference

    full = dict(weight_threshold=0.001, max_intersections=1024)
    full.update(kw)
    return {k: refdata.Output.of(v) for k, v in make_golden_reference.run_ref(case, **full).items()}


def check_seeds(torch, seeds):
    """-> (failures [(seed, scene kind, ray kind, [what differs])], {(scene kind, ray kind)} covered)."""
    failures, seen = [], set()
    stored = refdata.stored_cases()
    for seed in seeds:
        scene_kind, ray_kind, f, rays, start, dq, kw = fuzz_cases.make_case(seed)
        seen.add((scene_kind, ray_kind))
        case = common.Case(f, rays, start, dq, seed=seed)
        got = parity.run_ours(torch, case, tape=bool(seed & 1), **kw)
        if f"fuzz{seed}" in stored:
            ref = refdata.reference(f"fuzz{seed}", refdata.case_inputs(case) + (kw,))
        else:
            ref = live_reference(case, kw)
        what = []
        for k in ("num_intersections", "depth_indices", "rgba", "depth"):
            if k in ref and not ref[k].equal(got[k]):
                what.append(k)
        for k in ("points_grad", "attr_grad"):
            if not ref[k].same_nonfinite(got[k]):
                what.append(k + " non-finite pattern")
            elif refdata.grad_error(got[k], ref[k]) > 2e-5:
                what.append("%s %.2e" % (k, refdata.grad_error(got[k], ref[k])))
        if what:
            failures.append((seed, scene_kind, ray_kind, what))
    return failures, seen


@pytest.mark.parametrize("first_seed", [0, 60, 120, 180])
def test_tie_heavy_cases_match_the_reference_kernels(torch_cuda, first_seed):  # noqa: F811
    failures, seen = check_seeds(torch_cuda, range(first_seed, first_seed + 60))
    assert not failures, failures
    assert len(seen) >= 15


def test_rays_traced_alone_with_threshold_zero(torch_cuda):  # noqa: F811
    """Seed 3736 (degree 2, weight threshold 0, one quantile): traced one ray per launch, seven of its rays had position
    gradients of 1e-6 where the reference has 1e-14 -- the backward's SH basis was rounded differently from the
    forward's (foam_device.cuh, sh_basis), so the late cells' (saved colour - recomputed colour) / T was rounding
    residue.  Every ray on its own, re-walk and tape replay, against the reference's kernels."""
    _, _, f, rays, start, dq, kw = fuzz_cases.make_case(3736)
    assert f.sh_degree == 2 and kw == {"weight_threshold": 0.0} and dq.shape[1] == 1
    whole = common.Case(f, rays, start, dq, seed=3736)
    worst = 0.0
    for i in range(0, rays.shape[0], 2):
        case = common.Case(f, rays[i:i + 1], start[i:i + 1], dq[i:i + 1], seed=3736)
        case.grad_rgba, case.grad_depth = whole.grad_rgba[i:i + 1], whole.grad_depth[i:i + 1]
        ref = refdata.reference(f"fuzz3736_ray{i}", refdata.case_inputs(case) + (kw,))
        got = parity.run_ours(torch_cuda, case, tape=bool(i & 2), **kw)
        assert ref["rgba"].equal(got["rgba"]) and ref["depth"].equal(got["depth"])
        worst = max(worst, refdata.grad_error(got["points_grad"], ref["points_grad"]),
                    refdata.grad_error(got["attr_grad"], ref["attr_grad"]))
    assert worst <= 1e-5, worst


if __name__ == "__main__":
    import torch

    first, count = int(sys.argv[1]), int(sys.argv[2])
    failures, seen = check_seeds(torch, range(first, first + count))
    for f in failures:
        print("FAIL", f)
    print("cases", count, "from seed", first, "kinds covered", len(seen), "failures", len(failures))
