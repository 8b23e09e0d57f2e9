"""GPU: the fc256 layer's kernels on their own against float64 of their decoded inputs.

  arl_fc_forward       M = 1 .. 20 480 rows, on both sides of Mc = 128 * floor(SMs / 4), the largest M
                       the 4-CTA cluster kernel (FcFwdCluster, split-K over the cluster with a DSMEM
                       reduction) takes; above it the streaming kernel (FcFwd) runs (fc.cu).
  arl_fc_heads_forward at M = Mc and Mc + 1, with the action draw bit-exact against the Philox oracle.
  arl_fc_backward      at rollout sizes: 20 480 samples in one a2 block, 81 920 = 4096 envs x 20 steps
                       (20 blocks of 4096 rows) and 4 x 9216 (blocks of 9216 rows), with the d_h pair
                       (block + transposed copy) written by arl_heads_backward, grad_unscale != 1.

Tolerance, fixed from the formats before the first run: bf16 hi + lo operands (2^-17) in K-term fp32
sums, 4 * 2^-17 * sqrt(K) capped at the 1e-3 bar -> 1e-3 for the forward (K = 2592) and for the
weight gradient (K = the sample count); 4 * 2^-17 * sqrt(256) = 4.9e-4 for d_a2 (K = 256)."""
import math

import numpy as np
import pytest
import torch

import kernel_ref as kr
from util import REL_TOL

pytestmark = pytest.mark.gpu

A2, FC = 2592, 256
TOL_FWD = min(REL_TOL, 4 * 2.0 ** -17 * math.sqrt(A2))
TOL_WGRAD = REL_TOL
TOL_DGRAD = min(REL_TOL, 4 * 2.0 ** -17 * math.sqrt(FC))


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def mc():
    """Largest row count of the cluster kernel: ceil(M/128) * 4 <= SMs  <=>  M <= 128 * floor(SMs/4)."""
    return 128 * (sms() // 4)


def rows_of(key):
    return {"Mc": mc(), "Mc+1": mc() + 1}.get(key, key)


def cluster_kernel_runs(m):
    return (m + 127) // 128 * 4 <= sms()


def make_weights(pkg, cuda, A=6, seed=2):
    from oracle import a3c
    p = a3c.init_params(A, seed)
    rng = np.random.default_rng(seed)
    for k in p:
        p[k] = (p[k] * 2.0 if k.endswith("_w") else rng.normal(0, 0.02, p[k].shape)).astype(np.float32)
    flat = torch.as_tensor(a3c.flatten_params(p), device=cuda)
    prepared = torch.empty(pkg._cabi.prepared_floats(), device=cuda)
    pkg._cabi.call("arl_prepare_weights", flat.data_ptr(), prepared.data_ptr(), pkg._cabi.stream_ptr())
    return p, flat, prepared


def make_a2(pkg, cuda, m, seed):
    """A post-relu conv2 output: 30 % exact zeros, the rest in [1e-3, 1) (no value near the mask's
    threshold), as the split block the kernels read, and its decoded float values."""
    gen = torch.Generator(device=cuda).manual_seed(seed)
    x = torch.rand(m, A2, device=cuda, generator=gen) * 0.999 + 1e-3
    x[torch.rand(m, A2, device=cuda, generator=gen) < 0.3] = 0.0
    blk = pkg.network.encode_split(x)
    return blk, pkg.network.decode_split(blk, m, A2)


def run_fc_forward(pkg, flat, prepared, blk, m):
    buf, h = kr.canary(m * FC * 4, blk.device)
    pkg._cabi.call("arl_fc_forward", flat.data_ptr(), prepared.data_ptr(), blk.data_ptr(), h.data_ptr(), m,
                   pkg._cabi.stream_ptr())
    torch.cuda.synchronize()
    return buf


def test_fc_forward_shapes_reach_both_kernels(pkg, cuda):
    """The parametrization below holds a row count the cluster kernel takes and one it does not."""
    assert cluster_kernel_runs(rows_of("Mc")) and not cluster_kernel_runs(rows_of("Mc+1"))
    ms = [rows_of(k) for k in FC_ROWS]
    assert any(cluster_kernel_runs(m) for m in ms) and any(not cluster_kernel_runs(m) for m in ms)


FC_ROWS = [1, 127, 128, 129, 4096, "Mc", "Mc+1", 9216, 20480]


@pytest.mark.parametrize("m", FC_ROWS, ids=str)
def test_fc_forward_vs_float64(pkg, cuda, m):
    m = rows_of(m)
    p, flat, prepared = make_weights(pkg, cuda)
    blk, a2 = make_a2(pkg, cuda, m, seed=m)
    nbytes = m * FC * 4
    buf = run_fc_forward(pkg, flat, prepared, blk, m)
    kr.check_canary(buf, nbytes, torch.float32, "h")
    buf2 = run_fc_forward(pkg, flat, prepared, blk, m)
    assert kr.same_bits(buf, buf2), "fc256 forward is not repeatable"
    w = torch.as_tensor(p["l4_w"], device=cuda).double()
    b = torch.as_tensor(p["l4_b"], device=cuda).double()
    ref = torch.relu(a2.double() @ w + b)
    report = {}
    kr.check("h/row", buf[:nbytes].view(torch.float32).view(m, FC), ref, (0,), TOL_FWD, report)
    kr.show("fc256 fwd M=%d (%s, Mc=%d)" % (m, "FcFwdCluster" if cluster_kernel_runs(m) else "FcFwd", mc()), report)


@pytest.mark.parametrize("m", ["Mc", "Mc+1"])
def test_fc_heads_forward_with_actions(pkg, cuda, m):
    from oracle import philox
    m = rows_of(m)
    A = 6
    p, flat, prepared = make_weights(pkg, cuda, A, seed=5)
    blk, a2 = make_a2(pkg, cuda, m, seed=m + 1)
    outs = []
    for _ in range(2):
        bufs = dict(h=kr.canary(m * FC * 4, cuda), logits=kr.canary(m * A * 4, cuda),
                    probs=kr.canary(m * A * 4, cuda), value=kr.canary(m * 4, cuda))
        actions = torch.full((m + 64,), -7, dtype=torch.int32, device=cuda)
        P = {k: v[1].data_ptr() for k, v in bufs.items()}
        pkg._cabi.call("arl_fc_heads_forward", flat.data_ptr(), prepared.data_ptr(), A, blk.data_ptr(), P["h"],
                       P["logits"], P["probs"], P["value"], actions.data_ptr(), 100, 9, None, 4321, m,
                       pkg._cabi.stream_ptr())
        torch.cuda.synchronize()
        for k, (buf, v) in bufs.items():
            kr.check_canary(buf, v.numel() * 4, torch.float32, k)
        assert bool(actions[m:].eq(-7).all())
        outs.append((bufs, actions))
    for k in outs[0][0]:
        assert kr.same_bits(outs[0][0][k][1], outs[1][0][k][1]), k
    assert torch.equal(outs[0][1], outs[1][1])
    bufs, actions = outs[0]
    h, logits = bufs["h"][1].view(m, FC), bufs["logits"][1].view(m, A)
    probs, value = bufs["probs"][1].view(m, A), bufs["value"][1].view(m)
    d = lambda k: torch.as_tensor(p[k], device=cuda).double()
    report = {}
    kr.check("h", h, torch.relu(a2.double() @ d("l4_w") + d("l4_b")), (0,), TOL_FWD, report)
    kr.check("logits", logits, h.double() @ d("p_w") + d("p_b"), (0,), REL_TOL, report)
    kr.check("probs", probs, torch.softmax(logits.double(), 1), (0,), REL_TOL, report)
    kr.check("value", value, (h.double() @ d("q_w") + d("q_b")).reshape(-1), (0,), REL_TOL, report)
    kr.show("fc256+heads fwd M=%d (%s)" % (m, "FcFwdCluster" if cluster_kernel_runs(m) else "FcFwd"), report)
    ref_act = philox.sample_actions(probs.cpu().numpy(), np.arange(100, 100 + m), 9, 4321)
    assert np.array_equal(actions[:m].cpu().numpy(), ref_act)


@pytest.mark.parametrize("n,block", [(20480, 20480), (81920, 4096), (4 * 9216, 9216)])
def test_fc_backward_rollout_sizes_vs_float64(pkg, cuda, n, block):
    A = 6
    p, flat, prepared = make_weights(pkg, cuda, A, seed=7)
    f = pkg._cabi
    gen = torch.Generator(device=cuda).manual_seed(n + block)
    # the rollout's a2: one split block per forward call of `block` rows
    blks, a2s = zip(*[make_a2(pkg, cuda, block, seed=n + o) for o in range(0, n, block)])
    blk, a2 = torch.cat(blks), torch.cat(a2s)
    # d_h as arl_heads_backward writes it: split block of n rows + the transposed copy
    h = torch.relu(torch.randn(n, FC, device=cuda, generator=gen))
    dlogits = torch.randn(n, A, device=cuda, generator=gen) / n
    dvalue = torch.randn(n, device=cuda, generator=gen) / n
    scale = 2.0 ** 14
    ws = torch.empty(f.workspace_bytes(A), dtype=torch.uint8, device=cuda)
    d_h = torch.empty(n + (n + 7) // 8 * 8, FC, device=cuda)
    hg = torch.zeros(f.param_layout(A)[-1], device=cuda)
    f.call("arl_heads_backward", flat.data_ptr(), A, h.data_ptr(), dlogits.data_ptr(), dvalue.data_ptr(),
           d_h.data_ptr(), hg.data_ptr(), ws.data_ptr(), n, scale, f.stream_ptr())
    off = f.param_layout(A)
    unscale = 1.0 / scale

    def run():
        grads = torch.full((off[-1],), 7.0, device=cuda)
        buf, d_a2 = kr.canary(n * A2 * 4, cuda)
        f.call("arl_fc_backward", prepared.data_ptr(), blk.data_ptr(), block, d_h.data_ptr(), d_a2.data_ptr(),
               grads.data_ptr(), ws.data_ptr(), n, unscale, f.stream_ptr())
        torch.cuda.synchronize()
        return grads, buf

    grads, buf = run()
    grads2, buf2 = run()
    assert kr.same_bits(grads, grads2) and kr.same_bits(buf, buf2), "fc256 backward is not repeatable"
    kr.check_canary(buf, n * A2 * 4, torch.float32, "d_a2")
    outside = torch.cat([grads[:off[4]], grads[off[6]:]])
    assert bool(outside.eq(7.0).all()), "fc256 backward wrote outside l4_w / l4_b"

    dh = pkg.network.decode_split(d_h[:n], n, FC).double()            # x scale, as the kernel reads it
    w = torch.as_tensor(p["l4_w"], device=cuda).double()
    ref_w = (a2.double().t() @ dh) * unscale
    ref_b = dh.sum(0) * unscale
    ref_da2 = (dh @ w.t()) * (a2 > 0)
    got_w = grads[off[4]:off[5]].view(A2, FC)
    got_b = grads[off[5]:off[6]]
    got_da2 = buf[:n * A2 * 4].view(torch.float32).view(n, A2)
    report = {}
    kr.check("l4_w/out", got_w, ref_w, (1,), TOL_WGRAD, report)
    kr.check("l4_w/in", got_w, ref_w, (0,), TOL_WGRAD, report)
    kr.check("l4_b", got_b, ref_b, (0,), TOL_WGRAD, report)
    kr.check("d_a2/sample", got_da2, ref_da2, (0,), TOL_DGRAD, report)
    kr.show("fc256 bwd N=%d a2 blocks of %d" % (n, block), report)
