"""CPU tests of the stored reference outputs (tests/refdata.py): a stored gradient holds every entry, so an error at an
entry where the reference is tiny is caught -- the failure test_gpu_fuzz.py::test_rays_traced_alone_with_threshold_zero
was written for (late cells with gradients of 1e-6 where the reference has 1e-14)."""
import numpy as np

import common
import fuzz_cases
import refdata


def test_single_ray_gradients_catch_an_error_at_the_smallest_entry():
    _, _, f, rays, start, dq, kw = fuzz_cases.make_case(3736)
    whole = common.Case(f, rays, start, dq, seed=3736)
    checked = 0
    for i in range(0, rays.shape[0], 2):
        case = common.Case(f, rays[i:i + 1], start[i:i + 1], dq[i:i + 1], seed=3736)
        case.grad_rgba, case.grad_depth = whole.grad_rgba[i:i + 1], whole.grad_depth[i:i + 1]
        ref = refdata.reference(f"fuzz3736_ray{i}", refdata.case_inputs(case) + (kw,))
        for k in ("points_grad", "attr_grad"):
            out = ref[k]
            assert out.index.size == int(np.prod(out.shape)), "every entry is stored"
            got = np.zeros(out.shape, dtype=np.float64)
            got.reshape(-1)[out.index] = out.values
            assert refdata.grad_error(got, out) <= 1e-5            # the stored values pass the bar themselves
            j = out.index[np.argmin(np.abs(out.values))]            # where the reference is smallest
            got.reshape(-1)[j] += 1.01e-5 * out.scale if out.scale > 0 else 1e-6  # all-zero reference: any error
            assert refdata.grad_error(got, out) > 1e-5, (i, k)
            got.reshape(-1)[j] = np.nan
            assert refdata.grad_error(got, out) == np.inf             # non-finite where the reference is finite
            checked += 1
    assert checked == 2 * len(range(0, rays.shape[0], 2))
