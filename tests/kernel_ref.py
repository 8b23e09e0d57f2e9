"""Helpers of the kernel-by-kernel reference tests (test_gpu_conv_forward.py, test_gpu_fc.py,
test_gpu_heads.py, test_gpu_nature_scale.py): a per-slice error metric, NaN-filled canary
buffers, the sensitivity self-check of the per-slice gate and the bit-identical repeat.

Imports torch only; nothing here touches a CUDA device at import, so the test modules collect on a
machine without one."""
import torch

from util import REL_TOL

SLICE_FLOOR = 1e-3      # a slice whose max|ref| is below this fraction of the global max is scaled by it
CANARY = 0xFF           # 0xFF bytes: NaN in fp16, bf16 and fp32
SLACK = 4096            # canary bytes after the last sample of every output


def _f64(x):
    return torch.as_tensor(x).to(torch.float64)


def rel_err(x, ref):
    """util.rel_err on the device: max|x - ref| / max|ref| over the whole tensor (0/0 -> 0)."""
    x, ref = _f64(x), _f64(ref).to(torch.as_tensor(x).device)
    assert x.shape == ref.shape, (x.shape, ref.shape)
    if x.numel() == 0:
        return 0.0
    d, s = float((x - ref).abs().max()), float(ref.abs().max())
    return d / s if s > 0 else d


def _slice_max(t, dims):
    """max over everything but ``dims`` (the dimensions that index a slice)."""
    red = [d for d in range(t.dim()) if d not in [d % t.dim() for d in dims]]
    return t.amax(dim=red) if red else t


def slice_err(x, ref, dims):
    """max over slices of  max|x - ref| / max|ref|  within the slice.  A slice is one index of each of
    ``dims`` (``dims=(0,)``: per sample row; ``dims=(-1,)``: per output channel).  A slice whose max|ref|
    is below SLICE_FLOOR of the global max is divided by that floor instead, so an all-zero slice (a
    relu that is off for a whole channel) is judged against the tensor's scale, not against 0."""
    x, ref = _f64(x), _f64(ref).to(torch.as_tensor(x).device)
    assert x.shape == ref.shape, (x.shape, ref.shape)
    if x.numel() == 0:
        return 0.0
    a = ref.abs()
    g = float(a.max())
    if g == 0.0:
        return float((x - ref).abs().max())
    num = _slice_max((x - ref).abs(), dims)
    den = _slice_max(a, dims).clamp_min(SLICE_FLOOR * g)
    return float((num / den).max())


def errs(x, ref, dims):
    """(rel_err, slice_err) of one comparison; both are gated."""
    return rel_err(x, ref), slice_err(x, ref, dims)


def check(name, x, ref, dims, tol, report):
    """Gate one comparison with both metrics at ``tol``, run its sensitivity self-check and record the
    two errors in ``report`` (printed by the tests)."""
    r, s = errs(x, ref, dims)
    report[name] = (r, s)
    assert r <= tol and s <= tol, (name, r, s, tol)
    self_check(x, ref, dims)
    return r, s


def self_check(x, ref, dims, tol=REL_TOL):
    """The per-slice gate sees what rel_err cannot: in a copy of the device output, one element of a
    small slice (max|ref| below a tenth of the global max, above the floor) is moved by 2e-3 of that
    slice's max.  slice_err must then exceed ``tol`` (the 1e-3 bar) and rel_err must stay within it.
    When the data has no slice that small (every sample alike), the smallest slice is first scaled by
    1/20 in both copies, which is the same comparison on data that has one."""
    x, ref = _f64(x).clone(), _f64(ref).to(torch.as_tensor(x).device).clone()
    nd = x.dim()
    dims = sorted(d % nd for d in dims)
    g = float(ref.abs().max())
    assert g > 0, "self-check needs a non-zero reference"
    smax = _slice_max(ref.abs(), dims)
    if smax.numel() < 2:
        return                      # one slice: slice_err is rel_err, there is nothing to show
    ok = (smax >= 10 * SLICE_FLOOR * g) & (smax < 0.1 * g)
    if bool(ok.any()):
        cand = torch.where(ok, smax, torch.full_like(smax, float("inf")))
    else:                           # the smallest live slice other than the one holding the maximum
        cand = torch.where(smax >= 10 * SLICE_FLOOR * g, smax, torch.full_like(smax, float("inf")))
        cand.reshape(-1)[int(smax.reshape(-1).argmax())] = float("inf")
        if not bool(torch.isfinite(cand).any()):
            return
    flat = int(cand.reshape(-1).argmin())
    idx = list(torch.unravel_index(torch.tensor(flat), smax.shape)) if smax.dim() else []
    sel = [slice(None)] * nd
    for d, i in zip(dims, idx):
        sel[d] = int(i)
    sel = tuple(sel)
    if not bool(ok.any()):
        x[sel] *= 0.05
        ref[sel] *= 0.05
    sl = ref[sel]
    m = float(sl.abs().max())
    assert 0 < m < 0.1 * g
    base_r = rel_err(x, ref)
    # perturb the element of the slice where the reference is largest, away from the current error
    j = int(sl.abs().reshape(-1).argmax())
    xs = x[sel].reshape(-1)
    d0 = float(xs[j] - sl.reshape(-1)[j])
    xs[j] += (2e-3 * m) * (1.0 if d0 >= 0 else -1.0)
    x[sel] = xs.reshape(x[sel].shape)
    r, s = rel_err(x, ref), slice_err(x, ref, dims)
    assert s > tol, ("slice gate missed a 2e-3 error in a small slice", s, tol)
    assert r <= tol, ("rel_err tripped on the self-check: the base error is too close to the gate", r, base_r)


def canary(nbytes, device, dtype=torch.float32):
    """A buffer of ``nbytes`` + SLACK bytes filled with 0xFF; returns (whole uint8 buffer, the first
    ``nbytes`` viewed as ``dtype``).  16-byte aligned (torch allocations are)."""
    buf = torch.full((nbytes + SLACK,), CANARY, dtype=torch.uint8, device=device)
    return buf, buf[:nbytes].view(dtype)


def check_canary(buf, nbytes, view_dtype, what):
    """The slack after the region is byte-identical to the fill, and no NaN is left in the region
    (read as ``view_dtype``: every element of it was written)."""
    assert bool(buf[nbytes:].eq(CANARY).all()), "%s: wrote past its last sample" % what
    region = buf[:nbytes].view(view_dtype)
    assert not bool(region.isnan().any()), "%s: %d elements left unwritten" % (what, int(region.isnan().sum()))


def same_bits(a, b):
    """Two results are bit-identical (compared as bytes)."""
    a, b = a.contiguous(), b.contiguous()
    return torch.equal(a.view(torch.uint8) if a.dtype != torch.uint8 else a,
                       b.view(torch.uint8) if b.dtype != torch.uint8 else b)


def show(title, report):
    """One line per comparison: the worst rel_err and slice_err."""
    for k, (r, s) in report.items():
        print("%-46s %-10s rel_err %.3e  slice_err %.3e" % (title, k, r, s))
