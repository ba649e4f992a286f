"""Stored outputs of the reference's own kernels, and the comparisons the GPU tests make against them.

tests/golden/make_golden_reference.py ran the reference's kernels (oracle/_ref, built from the original project's
sources) on a B200 for every case the GPU tests compare with, and wrote tests/golden/reference/kernels.npz.  The
file keeps each output compact:
  * a SHA-256 of the whole array (NaNs made canonical), for comparisons that must be bit-exact;
  * a SHA-256 of its finite mask, for "same non-finite pattern";
  * max |finite entry| of the whole array, the scale the gradient bars are relative to;
  * for tolerance comparisons, either
      - every entry ("quantized"): rounded to a step of tol/8 of the scale, tol being the bar the tests hold that
        output to; the comparisons add the rounding bound (tol/16) to what they measure, so a stored output checks
        every entry and never passes an error above the bar (and is at most tol/8 stricter than the bar); or
      - for outputs too large for that ("sketch"): the values at the largest entries plus a pseudo-random spread.
Each case also keeps a SHA-256 of its inputs, which the tests regenerate from seeded builders (numpy, Qhull, torch's
CUDA generator): reference() checks it first, so that a changed input generator is reported as such and not as a
kernel mismatch.  Values that are not outputs (the reference's run-to-run gradient noise, measured when the file was
made) are stored per case beside the outputs."""
from __future__ import annotations

import functools
import hashlib
import json
import os

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", "kernels.npz")
_SPREAD_STRIDE = 2654435761  # prime: the spread visits distinct entries unless the size is a multiple of it


def digest(a) -> str:
    a = np.ascontiguousarray(np.asarray(a))
    if a.dtype.kind == "f" and np.isnan(a).any():
        a = a.copy()
        a[np.isnan(a)] = np.nan
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()[:32]


def spread_index(size: int, count: int) -> np.ndarray:
    if count >= size:
        return np.arange(size, dtype=np.int64)
    return (np.arange(count, dtype=np.int64) * _SPREAD_STRIDE + 97) % size


def inputs_digest(*items) -> str:
    """One digest of a case's inputs: arrays / tensors (by value), dicts, sequences, scalars and None."""
    h = hashlib.sha256()

    def feed(x):
        if hasattr(x, "detach"):
            x = x.detach().cpu().numpy()
        if isinstance(x, np.ndarray):
            h.update(digest(x).encode())
        elif isinstance(x, dict):
            for k in sorted(x):
                h.update(repr(k).encode())
                feed(x[k])
        elif isinstance(x, (list, tuple)):
            h.update(b"[")
            for v in x:
                feed(v)
            h.update(b"]")
        else:
            h.update(repr(x).encode())

    feed(items)
    return h.hexdigest()[:32]


def case_inputs(case) -> tuple:
    """The arrays of a tests/common.Case."""
    f = case.foam
    return (f.points, f.attributes, f.adjacency, f.offsets, case.rays, case.start, case.quantiles, case.grad_rgba,
            case.grad_depth)


def sketch(a, top: int = 32, spread: int = 160, tol: float | None = None):
    """-> (metadata, indices, values, quantized values).  With tol, every entry is kept (quantized); the indices are
    then those of the non-finite entries.  Without, the indices are the top entries' and the values are those at the
    top entries, then at the spread."""
    a = np.asarray(a)
    flat = a.reshape(-1)
    meta = {"shape": list(a.shape), "dtype": a.dtype.str, "sha": digest(a)}
    idx = np.zeros(0, dtype=np.int64)
    vals = np.zeros(0, dtype=np.float32)
    quant = np.zeros(0, dtype=np.int32)
    if a.dtype.kind == "f":
        fin = np.isfinite(flat)
        meta["finite_sha"] = digest(np.isfinite(a))
        mag = np.where(fin, np.abs(flat.astype(np.float64)), -1.0)
        meta["scale"] = float(mag.max()) if fin.any() else 0.0
        if tol is not None:
            step = tol / 8 * meta["scale"]
            meta["step"] = step
            idx = np.flatnonzero(~fin)
            quant = (np.rint(np.where(fin, flat.astype(np.float64), 0.0) / step) if step > 0
                     else np.zeros(flat.size)).astype(np.int32)
        else:
            idx = np.argsort(-mag, kind="stable")[:top]
            idx = idx[mag[idx] >= 0]
            meta["spread"] = int(min(spread, flat.size))
            vals = np.concatenate([flat[idx], flat[spread_index(flat.size, spread)]]).astype(np.float32)
    return meta, idx, vals, quant


class Output:
    """One stored output of the reference."""

    def __init__(self, meta, index, values, quant=None):
        self.shape = tuple(meta["shape"])
        self.dtype = np.dtype(meta["dtype"])
        self.sha = meta["sha"]
        self.finite_sha = meta.get("finite_sha")
        self.scale = meta.get("scale")
        self.bound = 0.0  # |stored value - reference value| <= bound
        self.index, self.values = None, None
        size = int(np.prod(self.shape))
        if "spread" in meta:
            self.index = np.concatenate([index, spread_index(size, meta["spread"])])
            self.values = values.astype(np.float64)
        elif "step" in meta:
            fin = np.ones(size, dtype=bool)
            fin[index] = False
            self.index = np.flatnonzero(fin)
            self.values = quant[self.index].astype(np.float64) * meta["step"]
            self.bound = meta["step"] / 2

    @classmethod
    def of(cls, a):
        """Every finite entry of a, exactly (for comparisons with a reference run live)."""
        a = np.asarray(a)
        meta, _, _, _ = sketch(a, top=0, spread=0)
        meta.pop("spread", None)
        out = cls(meta, None, None)
        if a.dtype.kind == "f":
            out.index = np.flatnonzero(np.isfinite(a.reshape(-1)))
            out.values = a.reshape(-1)[out.index].astype(np.float64)
        return out

    def equal(self, got) -> bool:
        """Bit for bit (any NaN matching any NaN); integers compare by value whatever their width."""
        got = np.asarray(got)
        if got.dtype.kind in "iu" and self.dtype.kind in "iu" and got.dtype != self.dtype:
            if got.size and (got.min() < np.iinfo(self.dtype).min or got.max() > np.iinfo(self.dtype).max):
                return False
            got = got.astype(self.dtype)
        return got.shape == self.shape and digest(got) == self.sha

    def at(self, got) -> np.ndarray:
        """got's values at the stored entries."""
        got = np.asarray(got)
        assert got.shape == self.shape, (got.shape, self.shape)
        return got.reshape(-1)[self.index]

    def same_nonfinite(self, got) -> bool:
        return digest(np.isfinite(np.asarray(got))) == self.finite_sha


@functools.lru_cache(maxsize=None)
def _load():
    z = np.load(PATH)
    zigzag = z["quantized_planes"].T.copy().view(np.uint32).reshape(-1).astype(np.int64)
    quantized = (zigzag >> 1) ^ -(zigzag & 1)
    return json.loads(z["meta"].tobytes().decode()), z["index"].astype(np.int64), z["values"], quantized


def stored_cases() -> set:
    return set(_load()[0])


def reference(case: str, inputs) -> dict:
    """{output name: Output, plus the case's stored scalars under their own names}, after checking that `inputs`
    (a tuple, see inputs_digest) are those the stored outputs were made from."""
    meta, index, values, quantized = _load()
    rec = meta[case]
    assert inputs_digest(*inputs) == rec["inputs_sha"], (
        f"the inputs of case {case} differ from those the stored reference outputs were made from: an input "
        "generator (numpy, scipy's Qhull, torch's CUDA generator) changed; this is not a kernel mismatch")
    out = dict(rec.get("scalars", {}))
    for name, m in rec["outputs"].items():
        i0, ni = m["index_at"]
        v0, nv = m["values_at"]
        q0, nq = m["quantized_at"]
        out[name] = Output(m, index[i0:i0 + ni], values[v0:v0 + nv], quantized[q0:q0 + nq])
    return out


class Writer:
    """Collects sketches of many cases into one .npz (used by tests/golden/make_golden_reference.py)."""

    def __init__(self):
        self.meta, self.index, self.values, self.quantized = {}, [], [], []
        self.ni = self.nv = self.nq = 0

    def add(self, case: str, inputs, outputs: dict, scalars: dict | None = None, tol: dict | None = None,
            **sketch_args):
        """tol: {output name: the bar the tests hold it to} for the outputs to keep whole (quantized)."""
        rec = self.meta.setdefault(case, {"outputs": {}})
        rec["inputs_sha"] = inputs_digest(*inputs)
        if scalars:
            rec["scalars"] = {k: float(v) for k, v in scalars.items()}
        for name, a in outputs.items():
            if a is None:
                continue
            if hasattr(a, "detach"):
                a = a.detach().cpu().numpy()
            m, idx, vals, quant = sketch(a, tol=(tol or {}).get(name), **sketch_args)
            m["index_at"] = [self.ni, int(idx.size)]
            m["values_at"] = [self.nv, int(vals.size)]
            m["quantized_at"] = [self.nq, int(quant.size)]
            self.index.append(idx.astype(np.uint32))
            self.values.append(vals)
            self.quantized.append(quant)
            self.ni += idx.size
            self.nv += vals.size
            self.nq += quant.size
            rec["outputs"][name] = m

    def save(self, path: str):
        save(path, self.meta, np.concatenate(self.index), np.concatenate(self.values),
             np.concatenate(self.quantized))


def save(path, meta, index, values, quantized):
    """The quantized values go in zigzag form as four byte planes, which deflate compresses about a quarter better."""
    q = quantized.astype(np.int64)
    zigzag = ((q << 1) ^ (q >> 63)).astype(np.uint32)
    np.savez_compressed(path, meta=np.frombuffer(json.dumps(meta, sort_keys=True, separators=(",", ":")).encode(),
                                                 dtype=np.uint8),
                        index=index.astype(np.uint32), values=values.astype(np.float32),
                        quantized_planes=np.ascontiguousarray(zigzag.view(np.uint8).reshape(-1, 4).T))


# ---- comparisons ------------------------------------------------------------------------------
def assert_equal(got, ref: Output, what: str):
    assert ref.equal(got), f"{what} differs from the reference's kernels"


def assert_close(got, ref: Output, what: str, rtol=1e-5, atol=1e-5):
    """|got - ref| <= atol + rtol |ref| on the stored entries, the stored values' rounding bound taken off."""
    g = ref.at(got).astype(np.float64)
    r = ref.values
    both = np.isfinite(g) & np.isfinite(r)
    assert np.array_equal(np.isfinite(g), np.isfinite(r)), f"{what}: non-finite where the reference is finite"
    err = np.abs(g[both] - r[both]) + ref.bound
    allowed = atol + rtol * np.maximum(np.abs(r[both]) - ref.bound, 0.0)
    bad = err > allowed
    assert not bad.any(), f"{what}: {int(bad.sum())} of {bad.size} entries differ, worst by {float(err.max()):.3g}"


def grad_error(got, ref: Output) -> float:
    """tests/common.grad_error on the stored entries: max |got - ref| / max |ref| (the whole array's maximum), plus
    the stored values' rounding bound, so an upper bound of the true figure.  An entry that is finite in the
    reference but not in got counts as infinite."""
    g = ref.at(got).astype(np.float64)
    r = ref.values
    ok = np.isfinite(r)
    if not np.isfinite(g[ok]).all():
        return float("inf")
    if not ok.any():
        return 0.0
    return float((np.abs(g[ok] - r[ok]).max() + ref.bound) / max(ref.scale, 1e-30))


def assert_forward_equal(got: dict, ref: dict):
    """Integer traversal outputs bit-exact, rgba / depth within 1e-5 (tests/test_gpu_parity.py's bar)."""
    assert_equal(got["num_intersections"], ref["num_intersections"], "num_intersections")
    if "depth_indices" in ref:
        assert_equal(got["depth_indices"], ref["depth_indices"], "depth_indices")
        assert_close(got["depth"], ref["depth"], "depth")
    assert_close(got["rgba"], ref["rgba"], "rgba")


def assert_grads_close(got: dict, ref: dict, tol: float):
    for k in ("points_grad", "attr_grad"):
        err = grad_error(got[k], ref[k])
        assert err <= tol, f"{k}: max|d| / max|ref| = {err:.3e} > {tol}"
