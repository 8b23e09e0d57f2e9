"""GPU: the policy/value heads at every action count the C-ABI accepts, against float64.

Action counts A in {1, 2, 3, 7, 8, 18, 19, 20, 31, 32}: the edges of the three instantiations of
heads_bwd_kernel (J = A + 1 <= 8, <= 20, <= 33: A = 19 is the last of the second, A >= 20 runs the
third) and of the warp (heads_fwd_kernel keeps logit j in lane j: at A = 32, J = 33 outputs exceed
it; A = 1 is the degenerate softmax and the degenerate dueling mean).  Sample counts
N in {1, 7, 8, 9, 63, 65, 1000, 20480}: the 8-sample chunks of the transposed d_h copy, the 64-sample
staging chunk and a grid-stride loop that runs more than once per warp.

Heads, loss entries and draws are float32 arithmetic; their gate is the 1e-3 bar (the printed errors
show how far below it they sit).  d_h is stored as bf16 hi + lo (2^-17) of float32 sums."""
import numpy as np
import pytest
import torch

import kernel_ref as kr
from util import REL_TOL

pytestmark = pytest.mark.gpu

ACTIONS = [1, 2, 3, 7, 8, 18, 19, 20, 31, 32]
SAMPLES = [1, 7, 8, 9, 63, 65, 1000, 20480]
FC = 256


def bwd_instantiation(A):
    J = A + 1
    return "heads_bwd_kernel<8>" if J <= 8 else "heads_bwd_kernel<20>" if J <= 20 else "heads_bwd_kernel<33>"


def make_params(pkg, cuda, A, seed=0):
    from oracle import a3c
    p = a3c.init_params(A, seed)
    rng = np.random.default_rng(seed)
    for k in p:
        p[k] = (p[k] * 4.0 if k.endswith("_w") else rng.normal(0, 0.05, p[k].shape)).astype(np.float32)
    return p, torch.as_tensor(a3c.flatten_params(p), device=cuda)


def make_h(cuda, n, seed):
    gen = torch.Generator(device=cuda).manual_seed(seed)
    return torch.relu(torch.randn(n, FC, device=cuda, generator=gen)).contiguous()


def dd(p, k, cuda):
    return torch.as_tensor(p[k], device=cuda).double()


def run_heads_forward(pkg, flat, A, h, n):
    cuda = h.device
    bufs = dict(logits=kr.canary(n * A * 4, cuda), probs=kr.canary(n * A * 4, cuda), value=kr.canary(n * 4, cuda))
    pkg._cabi.call("arl_heads_forward", flat.data_ptr(), A, h.data_ptr(), bufs["logits"][1].data_ptr(),
                   bufs["probs"][1].data_ptr(), bufs["value"][1].data_ptr(), n, pkg._cabi.stream_ptr())
    torch.cuda.synchronize()
    for k, (buf, v) in bufs.items():
        kr.check_canary(buf, v.numel() * 4, torch.float32, k)
    return bufs


@pytest.mark.parametrize("A", ACTIONS)
def test_heads_forward_vs_float64(pkg, cuda, A):
    p, flat = make_params(pkg, cuda, A, seed=A)
    worst = {}
    for n in SAMPLES:
        h = make_h(cuda, n, seed=A * 1000 + n)
        b1, b2 = run_heads_forward(pkg, flat, A, h, n), run_heads_forward(pkg, flat, A, h, n)
        for k in b1:
            assert kr.same_bits(b1[k][1], b2[k][1]), (A, n, k)
        logits, probs = b1["logits"][1].view(n, A), b1["probs"][1].view(n, A)
        value = b1["value"][1].view(n)
        hd = h.double()
        ref_l = hd @ dd(p, "p_w", cuda) + dd(p, "p_b", cuda)
        report = {}
        kr.check("logits", logits, ref_l, (0,), REL_TOL, report)
        kr.check("probs", probs, torch.softmax(logits.double(), 1), (0,), REL_TOL, report)
        kr.check("value", value, (hd @ dd(p, "q_w", cuda) + dd(p, "q_b", cuda)).reshape(-1), (0,), REL_TOL, report)
        if A == 1:
            assert bool(probs.eq(1.0).all()), "A = 1: the softmax of one logit is 1"
        for k, v in report.items():
            worst[k] = tuple(max(a, b) for a, b in zip(worst.get(k, (0, 0)), v))
    kr.show("heads fwd A=%d N<=%d" % (A, SAMPLES[-1]), worst)


def run_heads_backward(pkg, flat, A, h, dlogits, dvalue, n, scale):
    cuda = h.device
    f = pkg._cabi
    off = f.param_layout(A)
    grads = torch.full((off[-1],), 7.0, device=cuda)
    n8 = (n + 7) // 8 * 8
    nbytes = (n + n8) * FC * 4
    buf, d_h = kr.canary(nbytes, cuda)
    ws = torch.empty(f.workspace_bytes(A), dtype=torch.uint8, device=cuda)
    f.call("arl_heads_backward", flat.data_ptr(), A, h.data_ptr(), dlogits.data_ptr(), dvalue.data_ptr(),
           d_h.data_ptr(), grads.data_ptr(), ws.data_ptr(), n, scale, f.stream_ptr())
    torch.cuda.synchronize()
    kr.check_canary(buf, nbytes, torch.bfloat16, "d_h (both copies, hi and lo)")
    return grads, buf


@pytest.mark.parametrize("A", ACTIONS)
def test_heads_backward_vs_float64(pkg, cuda, A):
    p, flat = make_params(pkg, cuda, A, seed=A + 50)
    off = pkg._cabi.param_layout(A)
    scale = 2.0 ** 10
    worst = {}
    for n in SAMPLES:
        gen = torch.Generator(device=cuda).manual_seed(A * 7 + n)
        h = make_h(cuda, n, seed=A * 999 + n)
        dlogits = torch.randn(n, A, device=cuda, generator=gen) / n
        dvalue = torch.randn(n, device=cuda, generator=gen) / n
        grads, buf = run_heads_backward(pkg, flat, A, h, dlogits, dvalue, n, scale)
        grads2, buf2 = run_heads_backward(pkg, flat, A, h, dlogits, dvalue, n, scale)
        assert kr.same_bits(grads, grads2) and kr.same_bits(buf, buf2), (A, n)
        assert bool(grads[:off[6]].eq(7.0).all()), "heads backward wrote below p_w"
        hd, dl, dv = h.double(), dlogits.double(), dvalue.double()
        ref = dict(p_w=hd.t() @ dl, p_b=dl.sum(0), q_w=(hd.t() @ dv[:, None]), q_b=dv.sum().reshape(1))
        ref_dh = (hd > 0) * (dl @ dd(p, "p_w", cuda).t() + dv[:, None] @ dd(p, "q_w", cuda).t()) * scale
        n8 = (n + 7) // 8 * 8
        raw = buf[:(n + n8) * FC * 4].view(torch.float32)
        dh_block = pkg.network.decode_split(raw[:n * FC], n, FC)
        t = raw[n * FC:].view(torch.bfloat16).reshape(2, n8 // 8, FC, 8)
        dh_t = (t[0].float() + t[1].float()).permute(0, 2, 1).reshape(n8, FC)
        assert bool(dh_t[n:].eq(0).all()), "transposed d_h: padding samples >= N are not zero"
        report = {}
        for i, k in enumerate(("p_w", "p_b", "q_w", "q_b")):
            got = grads[off[6 + i]:off[7 + i]].view(ref[k].shape)
            kr.check(k, got, ref[k], (-1,) if got.dim() == 2 else (0,), REL_TOL, report)
        kr.check("d_h", dh_block, ref_dh, (0,), REL_TOL, report)
        kr.check("d_h^T", dh_t[:n], ref_dh, (0,), REL_TOL, report)
        for k, v in report.items():
            worst[k] = tuple(max(a, b) for a, b in zip(worst.get(k, (0, 0)), v))
    kr.show("heads bwd A=%d (%s)" % (A, bwd_instantiation(A)), worst)


def small_ring(cuda, B, seed):
    slots = 6
    gen = torch.Generator(device=cuda).manual_seed(seed)
    return torch.randint(0, 256, (B, slots, 441 * 16), dtype=torch.uint8, device=cuda, generator=gen), slots, 5


def forward_entry(pkg, cuda, name, flat, A, ring, slots, first, ep=0.3):
    """One env step through ``name`` with the draw, every output in a canary buffer: the slack after each
    is intact, nothing is left unwritten and every action lies in [0, A).  Returns (raw buffers, views:
    h, logits, probs, value as float32, actions as int32)."""
    f = pkg._cabi
    B = ring.shape[0]
    prepared = torch.empty(f.prepared_floats(), device=cuda)
    sizes = dict(a1=B * 12800, a2=B * 2592 * 4, h=B * FC * 4, logits=B * A * 4, probs=B * A * 4, value=B * 4,
                 actions=B * 4)
    bufs = {k: kr.canary(n, cuda, torch.int32 if k == "actions" else torch.float32) for k, n in sizes.items()}
    P = {k: v[1].data_ptr() for k, v in bufs.items()}
    common = (flat.data_ptr(), prepared.data_ptr(), 1, A, ring.data_ptr(), B, slots, first)
    outs = (P["a1"], P["a2"], P["h"], P["logits"], P["probs"], P["value"], P["actions"], 3, 11, None, 99)
    if name == "arl_forward_dueling":
        f.call(name, *common[:-1], first, 1, *outs, ep, 1.0, 0.1, 1000.0, 0.0, f.stream_ptr())
    elif name == "arl_forward_egreedy":
        f.call(name, *common, *outs, ep, 1.0, 0.1, 1000.0, 0.0, f.stream_ptr())
    else:
        f.call(name, *common, *outs, f.stream_ptr())
    torch.cuda.synchronize()
    stored = dict(a1=torch.float16, a2=torch.bfloat16, actions=None)
    for k, (buf, v) in bufs.items():
        if k == "actions":
            assert bool(buf[sizes[k]:].eq(kr.CANARY).all()), "actions: wrote past its last sample"
            assert bool(((v >= 0) & (v < A)).all()), "actions: unwritten or outside [0, A)"
        else:
            kr.check_canary(buf, sizes[k], stored.get(k, torch.float32), k)
    o = dict(h=bufs["h"][1].view(B, FC), logits=bufs["logits"][1].view(B, A), probs=bufs["probs"][1].view(B, A),
             value=bufs["value"][1], actions=bufs["actions"][1])
    return {k: b for k, (b, _) in bufs.items()}, o


def forward_twice(pkg, cuda, name, flat, A, ring, slots, first):
    """forward_entry twice: every output byte of the second call equals the first's."""
    raw, o = forward_entry(pkg, cuda, name, flat, A, ring, slots, first)
    raw2, _ = forward_entry(pkg, cuda, name, flat, A, ring, slots, first)
    for k in raw:
        assert kr.same_bits(raw[k], raw2[k]), (name, k)
    return o


def draw(pkg, cuda, kind, scores, A, ep=0.3):
    f = pkg._cabi
    B = scores.shape[0]
    act = torch.full((B,), -7, dtype=torch.int32, device=cuda)
    if kind == "egreedy":
        f.call("arl_egreedy_actions", scores.data_ptr(), act.data_ptr(), B, A, ep, 3, 11, 99, f.stream_ptr())
    else:
        f.call("arl_sample_actions", scores.data_ptr(), act.data_ptr(), B, A, 3, 11, 99, f.stream_ptr())
    torch.cuda.synchronize()
    return act


@pytest.mark.parametrize("A", [1, 2, 32])
def test_dueling_egreedy_and_sample_draws(pkg, cuda, A):
    """arl_forward_dueling (with the ε-greedy draw), arl_forward_egreedy and arl_forward_sample on a
    small ring, each called twice with canary outputs: the heads' outputs against float64 of the h each
    call wrote, the draws bit-exact against the stand-alone draw entries on the scores each call wrote."""
    p, flat = make_params(pkg, cuda, A, seed=A + 300)
    ring, slots, first = small_ring(cuda, 37, seed=A)
    report = {}
    # dueling: Q = v + adv - mean(adv)
    o = forward_twice(pkg, cuda, "arl_forward_dueling", flat, A, ring, slots, first)
    hd = o["h"].double()
    adv = hd @ dd(p, "p_w", cuda) + dd(p, "p_b", cuda)
    v = (hd @ dd(p, "q_w", cuda) + dd(p, "q_b", cuda)).reshape(-1)
    q_ref = v[:, None] + adv - adv.mean(1, keepdim=True)
    kr.check("dueling Q", o["logits"], q_ref, (0,), REL_TOL, report)
    kr.check("dueling v", o["value"], v, (0,), REL_TOL, report)
    kr.check("dueling probs", o["probs"], torch.softmax(o["logits"].double(), 1), (0,), REL_TOL, report)
    if A == 1:
        assert torch.equal(o["logits"].view(-1), o["value"]), "A = 1: Q must equal v exactly"
    assert torch.equal(o["actions"], draw(pkg, cuda, "egreedy", o["logits"], A))
    # plain ε-greedy: the Q values are the p_w/p_b head
    o = forward_twice(pkg, cuda, "arl_forward_egreedy", flat, A, ring, slots, first)
    kr.check("egreedy logits", o["logits"], o["h"].double() @ dd(p, "p_w", cuda) + dd(p, "p_b", cuda), (0,),
             REL_TOL, report)
    assert torch.equal(o["actions"], draw(pkg, cuda, "egreedy", o["logits"], A))
    # policy sample
    o = forward_twice(pkg, cuda, "arl_forward_sample", flat, A, ring, slots, first)
    kr.check("sample probs", o["probs"], torch.softmax(o["logits"].double(), 1), (0,), REL_TOL, report)
    assert torch.equal(o["actions"], draw(pkg, cuda, "sample", o["probs"], A))
    kr.show("dueling / egreedy / sample A=%d" % A, report)


def loss_inputs(cuda, T, B, A, seed):
    rng = np.random.default_rng(seed)
    x = dict(rew=rng.choice([-3.0, -1.0, 0.0, 0.5, 1.0, 7.0], (T, B)).astype(np.float32),
             term=(rng.random((T, B)) < 0.25).astype(np.uint8),
             acts=rng.integers(0, A, ((T + 1) * B,)).astype(np.int32),
             q=rng.normal(0, 1.5, (T * B, A)).astype(np.float32),
             q_next=rng.normal(0, 1.5, (T * B, A)).astype(np.float32),
             q_boot=rng.normal(0, 1.5, (B, A)).astype(np.float32),
             value=rng.normal(0, 1, (T, B)).astype(np.float32),
             v_boot=rng.normal(0, 1, B).astype(np.float32))
    return x, {k: torch.as_tensor(v, device=cuda) for k, v in x.items()}


def run_twice(cuda, sizes, written, call):
    """``call`` (pointers of fresh canary buffers of sizes[k] floats) twice: the outputs in ``written``
    are complete and have their slack intact, the others stay all canary bytes, and both calls give the
    same bits.  Returns the float32 views of the first call."""
    runs = []
    for _ in range(2):
        bufs = {k: kr.canary(n * 4, cuda) for k, n in sizes.items()}
        call({k: v[1].data_ptr() for k, v in bufs.items()})
        torch.cuda.synchronize()
        runs.append(bufs)
    for k, n in sizes.items():
        buf = runs[0][k][0]
        assert kr.same_bits(buf, runs[1][k][0]), k
        if k in written:
            kr.check_canary(buf, n * 4, torch.float32, k)
        else:
            assert bool(buf.eq(kr.CANARY).all()), "%s written by an entry that does not take it" % k
    return {k: v for k, (_, v) in runs[0].items()}


@pytest.mark.parametrize("A", [1, 32])
def test_loss_kernels_at_extreme_action_counts(pkg, cuda, A):
    """arl_returns_lossgrad, arl_q_lossgrad, arl_nstep_q_lossgrad, arl_sarsa_lossgrad and the dueling
    forms of the three Q losses, each called twice into canary buffers, against the float64 oracles; at
    A = 1 the dueling advantage gradient is exactly 0."""
    from oracle import a3c
    import dueling_oracle
    import sarsa_oracle
    T, B, gamma, scale = 5, 37, 0.99, 1.0 / 37
    f, st = pkg._cabi, pkg._cabi.stream_ptr()
    x, g = loss_inputs(cuda, T, B, A, seed=A)
    N = T * B
    acts0 = x["acts"][:N]
    report = {}

    # A3C: returns, dlogits, dvalue
    o = run_twice(cuda, dict(R=N, dl=N * A, dv=N), ("R", "dl", "dv"), lambda P: f.call(
        "arl_returns_lossgrad", g["rew"].data_ptr(), g["term"].data_ptr(), g["acts"].data_ptr(), g["q"].data_ptr(),
        g["value"].data_ptr(), g["v_boot"].data_ptr(), P["R"], P["dl"], P["dv"], None, T, B, A, gamma, 0.01, -1.0,
        1.0, scale, st))
    R, dl, dv = o["R"], o["dl"].view(N, A), o["dv"]
    Rref = a3c.nstep_returns(a3c.clip_rewards(x["rew"]), x["term"].astype(bool), x["v_boot"].astype(np.float64), gamma)
    dlr, dvr = a3c.analytic_head_grads(torch.tensor(x["q"], dtype=torch.float64),
                                       torch.tensor(x["value"].reshape(-1), dtype=torch.float64),
                                       torch.tensor(acts0), torch.tensor(Rref.reshape(-1)), 0.01, scale)
    kr.check("a3c R", R, Rref.reshape(-1), (0,), REL_TOL, report)
    kr.check("a3c dvalue", dv, dvr, (0,), REL_TOL, report)
    if A == 1:       # one action: p = 1, log p = 0, H = 0 -> no policy gradient at all
        assert float(dl.abs().max()) == 0.0
    else:
        kr.check("a3c dlogits", dl, dlr, (0,), REL_TOL, report)

    def q_entry(name, dueling):
        def call(P):
            extra = (P["dval"],) if dueling else ()
            nm = name + ("_dueling" if dueling else "")
            nxt = g["q_boot"] if name == "arl_nstep_q_lossgrad" else g["q_next"]
            size = (N,) if name == "arl_q_lossgrad" else (T, B)
            f.call(nm, g["rew"].data_ptr(), g["term"].data_ptr(), g["acts"].data_ptr(), g["q"].data_ptr(),
                   nxt.data_ptr(), P["tgt"], P["dq"], *extra, None, *size, A, gamma, -1.0, 1.0, scale, st)
        o = run_twice(cuda, dict(tgt=N, dq=N * A, dval=N), ("tgt", "dq", "dval") if dueling else ("tgt", "dq"),
                      call)
        return o["tgt"], o["dq"].view(N, A), o["dval"]

    q64 = x["q"].astype(np.float64)
    tgt_ref = dict(
        arl_q_lossgrad=a3c.q_targets(x["q_next"], x["rew"].reshape(-1), x["term"].reshape(-1), gamma),
        # the n-step targets of tests/nstep_q_oracle.py (nstep_q_gradients): the returns recurrence on
        # clip(r) bootstrapped with max_a q_boot
        arl_nstep_q_lossgrad=a3c.nstep_returns(a3c.clip_rewards(x["rew"]), x["term"].astype(bool),
                                               x["q_boot"].astype(np.float64).max(1), gamma).reshape(-1),
        arl_sarsa_lossgrad=sarsa_oracle.sarsa_targets(x["q_next"], x["acts"][B:], x["rew"], x["term"], gamma))
    for name, yref in tgt_ref.items():
        delta = yref - q64[np.arange(N), acts0]
        plain_dq = np.zeros((N, A))
        plain_dq[np.arange(N), acts0] = -2.0 * delta * scale
        for dueling in (False, True):
            tgt, dq, dval = q_entry(name, dueling)
            tag = name.replace("arl_", "").replace("_lossgrad", "") + ("/duel" if dueling else "")
            kr.check(tag + " target", tgt, yref, (0,), REL_TOL, report)
            if dueling:
                dadv, gref = dueling_oracle.head_gradients(acts0, delta, A, scale)
                kr.check(tag + " dvalue", dval, gref, (0,), REL_TOL, report)
                if A == 1:
                    assert float(dq.abs().max()) == 0.0, "A = 1: the dueling advantage gradient must be 0"
                else:
                    kr.check(tag + " dadv", dq, dadv, (0,), REL_TOL, report)
            else:
                kr.check(tag + " dq", dq, plain_dq, (0,), REL_TOL, report)
    kr.show("loss kernels A=%d" % A, report)


@pytest.mark.parametrize("A", [0, 33])
def test_invalid_action_counts_are_refused(pkg, cuda, A):
    """A outside [1, ARL_MAX_ACTIONS]: every entry that takes an action count returns nonzero with a
    message, and no output buffer is touched -- the composed forwards included, which must refuse
    before their conv launches write a1 and a2 (and arl_prepare_weights the prepared images)."""
    f = pkg._cabi
    lib = f.load()
    st = f.stream_ptr()
    n = 64
    flat = torch.zeros(f.param_layout(32)[-1] + 1024, device=cuda)
    prepared = torch.full((f.prepared_floats(),), 7.0, device=cuda)
    h = torch.rand(n, FC, device=cuda)
    a2 = torch.zeros(n, 2592, device=cuda)
    ring = torch.zeros(n, 6, 441 * 16, dtype=torch.uint8, device=cuda)
    out = {k: torch.full((n * 40,), 7.0, device=cuda) for k in ("h", "logits", "probs", "value", "grads", "tgt", "dq",
                                                               "dval")}
    out["a1big"] = torch.full((n * 3200,), 7.0, device=cuda)
    out["a2big"] = torch.full((n * 2592,), 7.0, device=cuda)
    out["hbig"] = torch.full((n * 2 * FC,), 7.0, device=cuda)
    acts = torch.full((n,), -7, dtype=torch.int32, device=cuda)
    ws = torch.empty(f.workspace_bytes(1), dtype=torch.uint8, device=cuda)
    P = {k: v.data_ptr() for k, v in out.items()}
    i32 = torch.zeros(2 * n, dtype=torch.int32, device=cuda)
    u8 = torch.zeros(n, dtype=torch.uint8, device=cuda)
    fl = torch.zeros(n * 40, device=cuda)
    calls = {
        "arl_heads_forward": (flat.data_ptr(), A, h.data_ptr(), P["logits"], P["probs"], P["value"], n, st),
        "arl_heads_backward": (flat.data_ptr(), A, h.data_ptr(), fl.data_ptr(), fl.data_ptr(), P["hbig"], P["grads"],
                               ws.data_ptr(), n, 1.0, st),
        "arl_fc_heads_forward": (flat.data_ptr(), prepared.data_ptr(), A, a2.data_ptr(), P["h"], P["logits"],
                                 P["probs"], P["value"], acts.data_ptr(), 0, 0, None, 1, n, st),
        "arl_forward": (flat.data_ptr(), prepared.data_ptr(), 1, A, ring.data_ptr(), n, 6, 0, 1, P["a1big"],
                        P["a2big"], P["hbig"], P["logits"], P["probs"], P["value"], st),
        "arl_forward_sample": (flat.data_ptr(), prepared.data_ptr(), 0, A, ring.data_ptr(), n, 6, 0, P["a1big"],
                               P["a2big"], P["hbig"], P["logits"], P["probs"], P["value"], acts.data_ptr(), 0, 0,
                               None, 1, st),
        "arl_sample_actions": (fl.data_ptr(), acts.data_ptr(), n, A, 0, 0, 1, st),
        "arl_egreedy_actions": (fl.data_ptr(), acts.data_ptr(), n, A, 0.5, 0, 0, 1, st),
        "arl_returns_lossgrad": (fl.data_ptr(), u8.data_ptr(), i32.data_ptr(), fl.data_ptr(), fl.data_ptr(),
                                 fl.data_ptr(), P["tgt"], P["dq"], P["dval"], None, 1, n, A, 0.99, 0.01, -1.0, 1.0,
                                 1.0, st),
        "arl_q_lossgrad": (fl.data_ptr(), u8.data_ptr(), i32.data_ptr(), fl.data_ptr(), fl.data_ptr(), P["tgt"],
                           P["dq"], None, n, A, 0.99, -1.0, 1.0, 1.0, st),
        "arl_nstep_q_lossgrad": (fl.data_ptr(), u8.data_ptr(), i32.data_ptr(), fl.data_ptr(), fl.data_ptr(),
                                 P["tgt"], P["dq"], None, 1, n, A, 0.99, -1.0, 1.0, 1.0, st),
        "arl_sarsa_lossgrad": (fl.data_ptr(), u8.data_ptr(), i32.data_ptr(), fl.data_ptr(), fl.data_ptr(), P["tgt"],
                               P["dq"], None, 1, n // 2, A, 0.99, -1.0, 1.0, 1.0, st),
        "arl_q_lossgrad_dueling": (fl.data_ptr(), u8.data_ptr(), i32.data_ptr(), fl.data_ptr(), fl.data_ptr(),
                                   P["tgt"], P["dq"], P["dval"], None, n, A, 0.99, -1.0, 1.0, 1.0, st),
        "arl_nstep_q_lossgrad_dueling": (fl.data_ptr(), u8.data_ptr(), i32.data_ptr(), fl.data_ptr(), fl.data_ptr(),
                                         P["tgt"], P["dq"], P["dval"], None, 1, n, A, 0.99, -1.0, 1.0, 1.0, st),
        "arl_sarsa_lossgrad_dueling": (fl.data_ptr(), u8.data_ptr(), i32.data_ptr(), fl.data_ptr(), fl.data_ptr(),
                                       P["tgt"], P["dq"], P["dval"], None, 1, n // 2, A, 0.99, -1.0, 1.0, 1.0, st),
        "arl_forward_egreedy": (flat.data_ptr(), prepared.data_ptr(), 1, A, ring.data_ptr(), n, 6, 0, P["a1big"],
                                P["a2big"], P["hbig"], P["logits"], P["probs"], P["value"], acts.data_ptr(), 0, 0,
                                None, 1, 0.5, 1.0, 0.1, 1000.0, 0.0, st),
        "arl_forward_dueling": (flat.data_ptr(), prepared.data_ptr(), 1, A, ring.data_ptr(), n, 6, 0, 1, P["a1big"],
                                P["a2big"], P["hbig"], P["logits"], P["probs"], P["value"], acts.data_ptr(), 0, 0,
                                None, 1, 0.5, 1.0, 0.1, 1000.0, 0.0, st),
        "arl_backward": (flat.data_ptr(), prepared.data_ptr(), A, ring.data_ptr(), n, 6, 0, 1, fl.data_ptr(),
                         fl.data_ptr(), fl.data_ptr(), fl.data_ptr(), fl.data_ptr(), P["hbig"], P["a2big"],
                         P["a1big"], P["grads"], ws.data_ptr(), 1.0, 0, st),
        "arl_nature_forward": (flat.data_ptr(), A, fl.data_ptr(), P["a1big"], P["a2big"], P["a2big"], P["hbig"],
                               P["logits"], P["probs"], P["value"], n, st),
        "arl_nature_backward": (flat.data_ptr(), A, fl.data_ptr(), fl.data_ptr(), fl.data_ptr(), fl.data_ptr(),
                                fl.data_ptr(), fl.data_ptr(), fl.data_ptr(), P["hbig"], P["a2big"], P["a2big"],
                                P["a1big"], P["grads"], ws.data_ptr(), n, st),
    }
    for name, args in calls.items():
        rc = getattr(lib, name)(*args)
        torch.cuda.synchronize()
        msg = lib.arl_last_error().decode()
        assert rc != 0, "%s accepted action_size %d" % (name, A)
        assert "action" in msg.lower() or str(A) in msg, (name, msg)
        print("%-30s A=%-3d rc=%d  %s" % (name, A, rc, msg))
    for k, v in list(out.items()) + [("prepared", prepared)]:
        assert bool(v.eq(7.0).all()), "%s written by a refused call" % k
    assert bool(acts.eq(-7).all())
