"""GPU: the 'nature' trunk (arl_nature_forward / arl_nature_backward) at rollout sizes, kernel by
kernel against a float64 reference written here: torch on the device, each layer fed with the
device's own input to it, and the device's relu pattern taken as the relu derivative, as in
test_gpu_nature.py, so that a pre-activation within rounding distance of 0 cannot flip a column.

(B, T) = (300, 5) gives 1500 samples: 12 row tiles of 128 in the fc512 forward and the d_a3
contraction, the last one partial, several split-K slices in the fc512 weight gradient and several
samples per block in nat_heads_wgrad_kernel.  (4096, 5) gives 20 480.  A in {6, 32}.

Every output -- a1, a2, a3, h, logits, probs, value, the 12 gradients and d_h, d_a3, d_a2, d_a1 -- is
gated with rel_err and with slice_err per output channel (the last dimension) at the 1e-3 bar, the
tolerance of the existing nature tests on the same kernels.  Every output sits in a canary buffer
(nothing written past row N, nothing left unwritten) and forward and backward each run twice with
bit-identical results."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import kernel_ref as kr
from util import REL_TOL

pytestmark = pytest.mark.gpu

NAMES = ("l1_w", "l1_b", "l2_w", "l2_b", "l3_w", "l3_b", "l4_w", "l4_b", "p_w", "p_b", "q_w", "q_b")


def _layer(fn, inputs, grad_out):
    """float64 value of fn(*inputs) and its input gradients for the output gradient grad_out."""
    leaves = [t.detach().clone().requires_grad_(True) for t in inputs]
    out = fn(*leaves)
    out.backward(grad_out)
    return out.detach(), [t.grad for t in leaves]


def reference(p, x, dev, dlogits, dvalue):
    """float64 reference of each kernel of the trunk, fed with the device's own inputs to it: every
    layer's forward from the device's activations of the layer before, every backward from the device's
    gradient of the layer after (``dev`` holds both, float32 as the C-ABI wrote them), with the
    device's relu pattern (activation > 0) as the relu derivative.  Returns the forward outputs, the
    12 parameter gradients and the four pre-relu layer gradients."""
    f = lambda k: dev[k].double()
    nchw = lambda t: t.permute(0, 3, 1, 2)
    nhwc = lambda t: t.permute(0, 2, 3, 1)
    conv = lambda a, w, b, s: F.conv2d(a, w.permute(3, 2, 0, 1), b, stride=s)
    N = x.shape[0]
    fwd, grads, layer = {}, {}, {}
    # heads: logits = h p_w + p_b, value = h q_w + q_b;  d_h = (h > 0) (dlogits p_w^T + dvalue q_w^T)
    heads = lambda h, pw, pb, qw, qb: torch.cat([h @ pw + pb, h @ qw + qb], 1)
    out, (gh, gpw, gpb, gqw, gqb) = _layer(heads, [f("h"), p["p_w"], p["p_b"], p["q_w"], p["q_b"]],
                                           torch.cat([dlogits, dvalue[:, None]], 1))
    fwd["logits"], fwd["value"] = out[:, :-1], out[:, -1]
    fwd["probs"] = torch.softmax(f("logits"), 1)
    grads.update(p_w=gpw, p_b=gpb, q_w=gqw, q_b=gqb)
    layer["d_h"] = gh * (dev["h"] > 0)
    # fc512 on the device's a3, backward from the device's d_h
    out, (ga3, gw4, gb4) = _layer(lambda a, w, b: a @ w + b, [f("a3"), p["l4_w"], p["l4_b"]], f("d_h"))
    fwd["h"] = F.relu(out)
    grads.update(l4_w=gw4, l4_b=gb4)
    layer["d_a3"] = ga3 * (dev["a3"] > 0)
    # conv3 (3x3/1) on the device's a2, backward from the device's d_a3 (NHWC flatten)
    out, (ga2, gw3, gb3) = _layer(lambda a, w, b: nhwc(conv(nchw(a), w, b, 1)).reshape(N, -1),
                                  [f("a2"), p["l3_w"], p["l3_b"]], f("d_a3"))
    fwd["a3"] = F.relu(out)
    grads.update(l3_w=gw3, l3_b=gb3)
    layer["d_a2"] = ga2 * (dev["a2"] > 0)
    # conv2 (4x4/2) on the device's a1, backward from the device's d_a2
    out, (ga1, gw2, gb2) = _layer(lambda a, w, b: nhwc(conv(nchw(a), w, b, 2)),
                                  [f("a1"), p["l2_w"], p["l2_b"]], f("d_a2"))
    fwd["a2"] = F.relu(out)
    grads.update(l2_w=gw2, l2_b=gb2)
    layer["d_a1"] = ga1 * (dev["a1"] > 0)
    # conv1 (8x8/4) on the stacks / 255, backward from the device's d_a1 (no gradient w.r.t. the stacks)
    out, (gw1, gb1) = _layer(lambda w, b: nhwc(conv(nchw(x) / 255.0, w, b, 4)), [p["l1_w"], p["l1_b"]],
                             f("d_a1"))
    fwd["a1"] = F.relu(out)
    grads.update(l1_w=gw1, l1_b=gb1)
    return fwd, grads, layer


def run_canaried(cuda, shapes, call):
    """Every output in a canary buffer (kr.canary): ``call`` gets the float32 views; afterwards the slack
    of each is intact and no element is left unwritten.  Returns (raw buffers, views)."""
    bufs = {k: kr.canary(int(np.prod(s)) * 4, cuda) for k, s in shapes.items()}
    views = {k: bufs[k][1].view(s) for k, s in shapes.items()}
    call(views)
    torch.cuda.synchronize()
    for k, (buf, v) in bufs.items():
        kr.check_canary(buf, v.numel() * 4, torch.float32, k)
    return {k: b for k, (b, _) in bufs.items()}, views


def check_at_scale(pkg, cuda, B, T, A):
    from oracle import a3c
    f = pkg._cabi
    N = B * T
    assert N > 128, "more than one fc512 row tile"
    rng = np.random.default_rng(A * 10 + B)
    params = a3c.init_params(A, seed=A + B, trunk="nature")
    for k in params:
        params[k] = (params[k] * 2.0 if k.endswith("_w") else rng.normal(0, 0.01, params[k].shape)).astype(np.float32)
    flat = torch.as_tensor(a3c.flatten_params(params), device=cuda)
    off = f.nature_param_layout(A)
    gen = torch.Generator(device=cuda).manual_seed(N + A)
    x = torch.randint(0, 256, (N, 84, 84, 4), device=cuda, generator=gen).float()
    shapes = dict(a1=(N, 20, 20, 32), a2=(N, 9, 9, 64), a3=(N, 3136), h=(N, 512), logits=(N, A), probs=(N, A),
                  value=(N,))
    fwd_call = lambda o: f.call("arl_nature_forward", flat.data_ptr(), A, x.data_ptr(),
                                *(o[k].data_ptr() for k in shapes), N, f.stream_ptr())
    raw, out = run_canaried(cuda, shapes, fwd_call)
    raw2, _ = run_canaried(cuda, shapes, fwd_call)
    assert all(kr.same_bits(raw[k], raw2[k]) for k in shapes), "nature forward not repeatable"

    dlogits = torch.randn(N, A, device=cuda, generator=gen) / B
    dvalue = torch.randn(N, device=cuda, generator=gen) / B
    ws = torch.empty(int(f.load().arl_nature_workspace_bytes(A)), dtype=torch.uint8, device=cuda)
    lshapes = dict(d_h=(N, 512), d_a3=(N, 3136), d_a2=(N, 9, 9, 64), d_a1=(N, 20, 20, 32), grads=(off[-1],))
    bwd_call = lambda o: f.call("arl_nature_backward", flat.data_ptr(), A, x.data_ptr(), out["a1"].data_ptr(),
                                out["a2"].data_ptr(), out["a3"].data_ptr(), out["h"].data_ptr(), dlogits.data_ptr(),
                                dvalue.data_ptr(), *(o[k].data_ptr() for k in lshapes), ws.data_ptr(), N,
                                f.stream_ptr())
    braw, d = run_canaried(cuda, lshapes, bwd_call)
    braw2, _ = run_canaried(cuda, lshapes, bwd_call)
    assert all(kr.same_bits(braw[k], braw2[k]) for k in lshapes), "nature backward not repeatable"
    grads = d.pop("grads")

    p64 = {k: torch.as_tensor(v, device=cuda).double() for k, v in params.items()}
    fwd, gref, lref = reference(p64, x.double(), dict(out, **d), dlogits.double(), dvalue.double())
    # a3 and d_a3 are the NHWC flatten (h*7+w)*64+c: judged per output channel c, as the convs are
    chan = lambda k, t: t.reshape(N, 49, 64) if k in ("a3", "d_a3") else t
    report = {}
    for k in ("a1", "a2", "a3", "h", "logits", "probs", "value"):
        kr.check(k, chan(k, out[k]), chan(k, fwd[k]), (-1,) if out[k].dim() > 1 else (0,), REL_TOL, report)
    for i, k in enumerate(NAMES):
        got = grads[off[i]:off[i + 1]].view(gref[k].shape)
        kr.check(k, got, gref[k], (-1,), REL_TOL, report)
    for k in d:
        kr.check(k, chan(k, d[k]), chan(k, lref[k]), (-1,), REL_TOL, report)
    kr.show("nature B=%d T=%d (N=%d, %d fc512 row tiles) A=%d" % (B, T, N, -(-N // 128), A), report)


@pytest.mark.parametrize("A", [6, 32])
def test_nature_1500_samples_partial_last_tile(pkg, cuda, A):
    """(300, 5): 11 full fc512 row tiles and a partial twelfth (1500 = 11 * 128 + 92)."""
    check_at_scale(pkg, cuda, 300, 5, A)


@pytest.mark.parametrize("A", [6, 32])
def test_nature_20480_samples(pkg, cuda, A):
    """(4096, 5): the rollout size of the bench, 160 fc512 row tiles."""
    check_at_scale(pkg, cuda, 4096, 5, A)
