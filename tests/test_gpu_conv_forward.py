"""GPU: the forward kernels of the nips trunk one by one -- arl_conv1_forward and arl_conv2_forward
on their own, then every sample of a whole arl_forward / arl_forward_sample -- against float64
references of the same operation computed on the device from the kernel's own (decoded) inputs.

Shapes: single samples, a tile count of SMs + 1 (conv1) and SMs +- 1 (conv2) with the SM count
read from the device, a conv1 sample count whose last 128-row tile holds fewer than 16 valid grid
rows, t_max = 20 windows and the rollout sizes (4096 x 5, 16 384, 20 480).  In every ring the T + 3
planes of each env wrap past the last slot.

Tolerances, fixed from the storage formats before the first run:
  a1 (fp16, conv1's s8 limbs w = s*(L0/64 + L1/2^13 + L2/2^20)): 2^-11 for the storage plus the
     same again for the limb residual and the fp32 epilogue -> 2^-10 per (sample, channel);
  a2, h (bf16 hi + lo = 2^-17 per operand and per stored value, K-term fp32 sums whose cancellation
     grows the error relative to the result by about sqrt(K)): 4 * 2^-17 * sqrt(K), capped at the
     1e-3 bar -> 4.9e-4 for conv2 (K = 256), 1e-3 for fc256 (K = 2592);
  logits, probs, value (fp32 arithmetic): the 1e-3 bar.
Every comparison gates rel_err and slice_err (kernel_ref.py) and runs the slice gate's self-check."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import kernel_ref as kr
from util import REL_TOL, unblock

pytestmark = pytest.mark.gpu

TOL_A1 = 2.0 ** -10
TOL_A2 = min(REL_TOL, 4 * 2.0 ** -17 * math.sqrt(256))
TOL_H = min(REL_TOL, 4 * 2.0 ** -17 * math.sqrt(2592))
A1_BYTES, A2_FLOATS, GRID = 12800, 2592, 441


def encode_a1(a1):
    """float [n,20,20,16] -> the fp16 blocked a1 storage (inverse of network.decode_a1)."""
    n = a1.shape[0]
    return a1.reshape(n, 10, 2, 10, 2, 2, 8).permute(0, 2, 4, 5, 1, 3, 6).half().contiguous()


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def conv1_tiles(n):
    return -(-n * GRID // 128)


def conv2_tiles(n):
    return -(-n * 100 // 128)


def first_n(pred):
    return next(n for n in range(1, 1 << 20) if pred(n))


def conv1_shape(key):
    """(num_envs, steps) of a symbolic conv1 shape."""
    if key == "tiles=sms+1":
        # a tile is 128 of the sample's 441 grid rows, so the count grows by ~3.4 per sample: take the
        # sample count whose tile count is exactly SMs + 1 (none exists for a few SM counts; then the
        # first count past one tile per SM, within 4 of it)
        n = next((n for n in range(1, 64 * sms()) if conv1_tiles(n) == sms() + 1), None)
        n = n or first_n(lambda n: conv1_tiles(n) > sms())
        assert sms() < conv1_tiles(n) <= sms() + 4
        return n, 1
    if key == "tail<16rows":
        return first_n(lambda n: n > 1 and 0 < n * GRID % 128 < 16), 1
    return key


def params_for(kind, A=6, seed=11):
    """standard: the init x 2 with negative conv biases (exact relu zeros); zero: l1_w = 0 (the limb
    scale clamps at 1e-30) and fp16-exact l1_b of both signs; spread: output channel c of l1_w (and of
    l1_b) scaled by 10^(-2c/15), 1 down to 1e-2."""
    from oracle import a3c
    p = a3c.init_params(A, seed)
    rng = np.random.default_rng(seed)
    for k in p:
        if k.endswith("_w"):
            p[k] = (p[k] * 2.0).astype(np.float32)
    p["l1_b"] = -np.abs(rng.normal(0, 0.05, 16)).astype(np.float32)
    p["l2_b"] = -np.abs(rng.normal(0, 0.02, 32)).astype(np.float32)
    p["l4_b"] = rng.normal(0, 0.02, 256).astype(np.float32)
    p["p_b"] = rng.normal(0, 0.02, A).astype(np.float32)
    p["q_b"] = rng.normal(0, 0.02, 1).astype(np.float32)
    if kind == "zero":
        p["l1_w"] = np.zeros_like(p["l1_w"])
        p["l1_b"] = (np.arange(16) - 7.5).astype(np.float32) / 16.0       # +-k/32: exact in fp16
    elif kind == "spread":               # the bias shrinks with its channel, so every channel stays live
        f = 10.0 ** (-2.0 * np.arange(16) / 15.0)
        p["l1_w"] = (p["l1_w"] * f).astype(np.float32)
        p["l1_b"] = (p["l1_b"] * f).astype(np.float32)
    return p


def prepare(pkg, cuda, p):
    from oracle import a3c
    flat = torch.as_tensor(a3c.flatten_params(p), device=cuda)
    prepared = torch.empty(pkg._cabi.prepared_floats(), device=cuda)
    pkg._cabi.call("arl_prepare_weights", flat.data_ptr(), prepared.data_ptr(), pkg._cabi.stream_ptr())
    return flat, prepared


def make_ring(cuda, B, T, seed):
    slots = T + 5
    first = slots - 1 - T % 3                    # the T + 3 planes of an env wrap past the last slot
    gen = torch.Generator(device=cuda).manual_seed(seed)
    ring = torch.randint(0, 256, (B, slots, GRID * 16), dtype=torch.uint8, device=cuda, generator=gen)
    return ring, slots, first


def conv1_ref(ring, slots, first, T, l1_w, l1_b, env_lo=0, env_hi=None):
    """float64 relu(conv 8x8/4 of the stacked planes / 255 + b) -> [T*B, 20, 20, 16], t-major."""
    B = ring.shape[0] if env_hi is None else env_hi - env_lo
    w = torch.as_tensor(l1_w, device=ring.device).double().permute(3, 2, 0, 1)
    b = torch.as_tensor(l1_b, device=ring.device).double()
    out = torch.empty(T * B, 20, 20, 16, dtype=torch.float64, device=ring.device)
    for t in range(T):
        planes = [(first + t + k) % slots for k in range(4)]
        for o in range(0, B, 4096):
            e = min(B, o + 4096)
            x = unblock(ring[env_lo + o:env_lo + e][:, planes].reshape(e - o, 4, 84, 84)).double() / 255.0
            out[t * B + o:t * B + e] = F.relu(F.conv2d(x, w, b, stride=4)).permute(0, 2, 3, 1)
    return out


def conv2_ref(a1, l2_w, l2_b):
    """float64 relu(conv 4x4/2 + b) of a1 [n,20,20,16] -> [n, 2592] (NHWC flatten)."""
    w = torch.as_tensor(l2_w, device=a1.device).double().permute(3, 2, 0, 1)
    b = torch.as_tensor(l2_b, device=a1.device).double()
    out = torch.empty(a1.shape[0], A2_FLOATS, dtype=torch.float64, device=a1.device)
    for o in range(0, a1.shape[0], 4096):
        x = a1[o:o + 4096].double().permute(0, 3, 1, 2)
        out[o:o + 4096] = F.relu(F.conv2d(x, w, b, stride=2)).permute(0, 2, 3, 1).reshape(-1, A2_FLOATS)
    return out


def run_conv1(pkg, prepared, ring, B, slots, first, T):
    N = B * T
    buf, a1 = kr.canary(N * A1_BYTES, ring.device)
    pkg._cabi.call("arl_conv1_forward", prepared.data_ptr(), ring.data_ptr(), a1.data_ptr(), B, slots, first, T,
                   pkg._cabi.stream_ptr())
    torch.cuda.synchronize()
    return buf


@pytest.mark.parametrize("kind", ["standard", "zero", "spread"])
@pytest.mark.parametrize("shape", [(1, 1), (2, 1), (3, 2), "tiles=sms+1", "tail<16rows", (37, 20), (4096, 1),
                                   (4096, 5), (16384, 1)], ids=str)
def test_conv1_forward_vs_float64(pkg, cuda, shape, kind):
    B, T = conv1_shape(shape)
    N = B * T
    p = params_for(kind)
    _, prepared = prepare(pkg, cuda, p)
    ring, slots, first = make_ring(cuda, B, T, seed=N)
    buf = run_conv1(pkg, prepared, ring, B, slots, first, T)
    kr.check_canary(buf, N * A1_BYTES, torch.float16, "a1")
    buf2 = run_conv1(pkg, prepared, ring, B, slots, first, T)
    assert kr.same_bits(buf, buf2), "conv1 forward is not repeatable"

    got = pkg.network.decode_a1(buf[:N * A1_BYTES].view(torch.float32), N)
    title = "conv1 fwd %s B=%d T=%d tiles=%d (SMs %d)" % (kind, B, T, conv1_tiles(N), sms())
    if kind == "zero":
        # every output is relu(b), exactly: the bias is fp16-exact and the products are all 0
        want = torch.as_tensor(p["l1_b"], device=cuda).clamp_min(0).expand(N, 20, 20, 16)
        assert torch.equal(got, want), "all-zero l1_w: a1 is not exactly relu(l1_b)"
        print(title, "exact relu(b)")
        return
    ref = conv1_ref(ring, slots, first, T, p["l1_w"], p["l1_b"])
    report = {}
    kr.check("a1", got, ref, (0, 3), TOL_A1, report)
    if kind == "standard":                                  # the negative biases switch many outputs off
        assert float((got == 0).double().mean()) > 0.1
    if kind == "spread":
        # the worst error of one output channel relative to that channel's own scale (1 .. 1e-2)
        per_ch = kr.slice_err(got, ref, (3,))
        report["a1/channel"] = (kr.rel_err(got, ref), per_ch)
        assert per_ch <= REL_TOL, per_ch
    kr.show(title, report)


def conv2_n(key):
    if key == "tiles=sms-1":
        return first_n(lambda n: conv2_tiles(n) >= sms() - 1)
    if key == "tiles=sms+1":
        return first_n(lambda n: conv2_tiles(n) >= sms() + 1)
    return key


def run_conv2(pkg, prepared, a1s, n):
    buf, a2 = kr.canary(n * A2_FLOATS * 4, a1s.device)
    pkg._cabi.call("arl_conv2_forward", prepared.data_ptr(), a1s.data_ptr(), a2.data_ptr(), n, pkg._cabi.stream_ptr())
    torch.cuda.synchronize()
    return buf


@pytest.mark.parametrize("n", [1, 2, 3, 37, "tiles=sms-1", "tiles=sms+1", 4096, 16384, 20480], ids=str)
def test_conv2_forward_vs_float64(pkg, cuda, n):
    """arl_conv2_forward in its default (serpentine: tiles walked in reverse) order on an a1 of
    fp16-exact values with 20 % exact zeros, against float64 of those inputs."""
    n = conv2_n(n)
    p = params_for("standard")
    _, prepared = prepare(pkg, cuda, p)
    gen = torch.Generator(device=cuda).manual_seed(1000 + n)
    a1 = torch.rand(n, 20, 20, 16, device=cuda, generator=gen) * 2.0
    a1[torch.rand(n, 20, 20, 16, device=cuda, generator=gen) < 0.2] = 0.0
    a1s = encode_a1(a1)
    a1 = pkg.network.decode_a1(a1s.view(torch.float32), n)  # the fp16 values the kernel reads
    nbytes = n * A2_FLOATS * 4
    buf = run_conv2(pkg, prepared, a1s, n)
    kr.check_canary(buf, nbytes, torch.bfloat16, "a2 (hi and lo)")
    buf2 = run_conv2(pkg, prepared, a1s, n)
    assert kr.same_bits(buf, buf2), "conv2 forward is not repeatable"
    got = pkg.network.decode_split(buf[:nbytes].view(torch.float32), n, A2_FLOATS)
    ref = conv2_ref(a1, p["l2_w"], p["l2_b"])
    report = {}
    kr.check("a2/sample", got, ref, (0,), TOL_A2, report)
    kr.check("a2/channel", got.reshape(n, 81, 32), ref.reshape(n, 81, 32), (2,), TOL_A2, report)
    kr.show("conv2 fwd n=%d tiles=%d (SMs %d)" % (n, conv2_tiles(n), sms()), report)


def fc_switch():
    """Largest sample count the 4-CTA cluster kernel of the fc256 forward takes (fc.cu:
    ceil(M/128) * 4 <= SMs)."""
    return 128 * (sms() // 4)


def forward_outputs(pkg, cuda, entry, flat, prepared, A, ring, B, slots, first, T):
    """arl_forward (steps T) or arl_forward_sample (T == 1, with actions) into fresh canary buffers;
    returns the decoded float tensors and the raw buffers."""
    N = B * T
    f = pkg._cabi
    bufs = dict(a1=kr.canary(N * A1_BYTES, cuda), a2=kr.canary(N * A2_FLOATS * 4, cuda),
                h=kr.canary(N * 256 * 4, cuda), logits=kr.canary(N * A * 4, cuda), probs=kr.canary(N * A * 4, cuda),
                value=kr.canary(N * 4, cuda))
    P = {k: v[1].data_ptr() for k, v in bufs.items()}
    if entry == "arl_forward":
        f.call("arl_forward", flat.data_ptr(), prepared.data_ptr(), 0, A, ring.data_ptr(), B, slots, first, T,
               P["a1"], P["a2"], P["h"], P["logits"], P["probs"], P["value"], f.stream_ptr())
        actions = None
    else:
        actions = torch.full((N + 1024,), -7, dtype=torch.int32, device=cuda)
        f.call("arl_forward_sample", flat.data_ptr(), prepared.data_ptr(), 0, A, ring.data_ptr(), B, slots, first,
               P["a1"], P["a2"], P["h"], P["logits"], P["probs"], P["value"], actions.data_ptr(), 0, 77, None,
               12345, f.stream_ptr())
    torch.cuda.synchronize()
    for k, (buf, v) in bufs.items():
        kr.check_canary(buf, v.numel() * v.element_size(), torch.bfloat16 if k == "a2" else
                        torch.float16 if k == "a1" else torch.float32, k)
    if actions is not None:
        assert bool(actions[N:].eq(-7).all())
    rows = f.a2_block_rows(B) if T == 1 else N
    a2raw = bufs["a2"][1]
    out = dict(a1=pkg.network.decode_a1(bufs["a1"][1], N),
               a2=torch.cat([pkg.network.decode_split(a2raw.view(N, A2_FLOATS)[o:o + rows], rows, A2_FLOATS)
                             for o in range(0, N, rows)]),
               h=bufs["h"][1].view(N, 256), logits=bufs["logits"][1].view(N, A), probs=bufs["probs"][1].view(N, A),
               value=bufs["value"][1].view(N), actions=None if actions is None else actions[:N])
    return out, bufs


def check_every_sample(pkg, out, p, ring, slots, first, T, title):
    """Each layer against float64 of its own device input, per sample (and per channel for the
    convs)."""
    N = out["h"].shape[0]
    dev = out["h"].device
    d = lambda k: torch.as_tensor(p[k], device=dev).double()
    report = {}
    kr.check("a1", out["a1"], conv1_ref(ring, slots, first, T, p["l1_w"], p["l1_b"]), (0, 3), TOL_A1, report)
    kr.check("a2", out["a2"], conv2_ref(out["a1"], p["l2_w"], p["l2_b"]), (0,), TOL_A2, report)
    kr.check("h", out["h"], F.relu(out["a2"].double() @ d("l4_w") + d("l4_b")), (0,), TOL_H, report)
    h = out["h"].double()
    logits = h @ d("p_w") + d("p_b")
    kr.check("logits", out["logits"], logits, (0,), REL_TOL, report)
    kr.check("probs", out["probs"], torch.softmax(out["logits"].double(), dim=1), (0,), REL_TOL, report)
    kr.check("value", out["value"], (h @ d("q_w") + d("q_b")).reshape(-1), (0,), REL_TOL, report)
    kr.show(title, report)


def sub_batch(out, B, T, b_small):
    """The rows of envs 0 .. b_small-1 of every step (t-major) of a batch of B envs."""
    idx = torch.cat([torch.arange(t * B, t * B + b_small) for t in range(T)]).to(out["h"].device)
    return {k: (None if v is None else v[idx]) for k, v in out.items()}


def test_whole_forward_every_sample_target_form(pkg, cuda):
    """arl_forward with steps = 5 at 4096 envs (N = 20 480: the Q learners' target forward; fc256 runs
    as FcFwd), every sample of every layer; then batch independence: the same envs in a smaller batch
    on the same side of the fc256 kernel switch give bit-identical a1 .. value, and in a batch on the
    cluster side bit-identical a1 and a2."""
    A, B, T = 6, 4096, 5
    p = params_for("standard", A)
    flat, prepared = prepare(pkg, cuda, p)
    ring, slots, first = make_ring(cuda, B, T, seed=4242)
    mc = fc_switch()
    assert B * T > mc
    out, bufs = forward_outputs(pkg, cuda, "arl_forward", flat, prepared, A, ring, B, slots, first, T)
    out2, bufs2 = forward_outputs(pkg, cuda, "arl_forward", flat, prepared, A, ring, B, slots, first, T)
    for k in bufs:
        assert kr.same_bits(bufs[k][1], bufs2[k][1]), k
    check_every_sample(pkg, out, p, ring, slots, first, T, "arl_forward B=%d T=%d (FcFwd, Mc=%d)" % (B, T, mc))
    for b_small, same_side in ((mc // T + 1, True), (37, False)):
        assert (b_small * T > mc) == same_side
        small, _ = forward_outputs(pkg, cuda, "arl_forward", flat, prepared, A, ring[:b_small].contiguous(), b_small,
                                   slots, first, T)
        big = sub_batch(out, B, T, b_small)
        keys = ("a1", "a2", "h", "logits", "probs", "value") if same_side else ("a1", "a2")
        for k in keys:
            assert kr.same_bits(small[k], big[k]), (b_small, k)
        print("batch of %d envs: %s bit-identical to the 4096-env batch" % (b_small, ", ".join(keys)))


def test_whole_forward_sample_two_env_ranges(pkg, cuda):
    """arl_forward_sample at 18 432 envs (two env ranges of arl_a2_block_rows = 9216), every sample of
    every layer and the draw bit-exact against the Philox oracle on the probabilities written."""
    from oracle import philox
    A, B = 6, 18432
    p = params_for("standard", A, seed=3)
    flat, prepared = prepare(pkg, cuda, p)
    ring, slots, first = make_ring(cuda, B, 1, seed=777)
    rows = pkg._cabi.a2_block_rows(B)
    assert B // rows == 2 and rows > fc_switch()
    out, bufs = forward_outputs(pkg, cuda, "arl_forward_sample", flat, prepared, A, ring, B, slots, first, 1)
    out2, bufs2 = forward_outputs(pkg, cuda, "arl_forward_sample", flat, prepared, A, ring, B, slots, first, 1)
    for k in bufs:
        assert kr.same_bits(bufs[k][1], bufs2[k][1]), k
    assert torch.equal(out["actions"], out2["actions"])
    check_every_sample(pkg, out, p, ring, slots, first, 1, "arl_forward_sample B=%d (2 x %d)" % (B, rows))
    ref_act = philox.sample_actions(out["probs"].cpu().numpy(), np.arange(B), 77, 12345)
    assert np.array_equal(out["actions"].cpu().numpy(), ref_act)
    # envs 0..b-1 of a smaller batch that also runs FcFwd: every output bit-identical
    b_small = fc_switch() + 1
    small, _ = forward_outputs(pkg, cuda, "arl_forward_sample", flat, prepared, A, ring[:b_small].contiguous(),
                               b_small, slots, first, 1)
    for k in ("a1", "a2", "h", "logits", "probs", "value", "actions"):
        assert kr.same_bits(small[k], out[k][:b_small]), k
