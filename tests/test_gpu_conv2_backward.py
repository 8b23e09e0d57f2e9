"""GPU: arl_conv2_backward on its own -- weight gradient, both bias gradients and the input
gradient of conv2, from one fused tensor-core kernel -- against a float64 conv2 backward of the
same (decoded) inputs.  Sample counts cover a single tile, tile totals below and above the SM
count (not a multiple of it) and the bench size."""
import numpy as np
import pytest
import torch

from util import REL_TOL, rel_err

pytestmark = pytest.mark.gpu

A1_BYTES, DA1_BYTES = 12800, 14112          # per sample: fp16 a1 blocks, fp16 d_a1 on the 21x21 grid


def encode_a1(a1):
    """float [n,20,20,16] -> the fp16 blocked a1 storage (inverse of network.decode_a1)."""
    n = a1.shape[0]
    return a1.reshape(n, 10, 2, 10, 2, 2, 8).permute(0, 2, 4, 5, 1, 3, 6).half().contiguous()


def run(pkg, cuda, prepared, workspace, a1s, d_a2, n, unscale):
    lib = pkg._cabi.load()
    P = pkg._cabi.ptr
    grads = torch.full((4112 + 8192 + 32,), 7.0, device=cuda)
    d_a1 = torch.full((n * DA1_BYTES,), 0xFF, dtype=torch.uint8, device=cuda)
    assert lib.arl_conv2_backward(P(prepared), P(a1s), P(d_a2), P(d_a1), P(grads), P(workspace), n,
                                  unscale, pkg._cabi.stream_ptr()) == 0
    torch.cuda.synchronize()
    return grads, d_a1


@pytest.mark.parametrize("n", [1, 2, 3, 37, 200, 20480])
def test_conv2_backward_vs_float64(pkg, cuda, n):
    A = 6
    gen = torch.Generator(device=cuda).manual_seed(n)
    net = pkg.Network(action_size=A, num_envs=1, t_max=1, device="cuda:0")
    from oracle import a3c
    params = a3c.init_params(A, seed=5)
    params["l2_w"] = (params["l2_w"] * 2.0).astype(np.float32)
    net.set_weights(params)
    lib = pkg._cabi.load()
    assert lib.arl_prepare_weights(pkg._cabi.ptr(net.params), pkg._cabi.ptr(net.fc_w),
                                   pkg._cabi.stream_ptr()) == 0
    # a1 with exact zeros and negatives: the relu mask keeps only a1 > 0
    a1 = torch.randn(n, 20, 20, 16, device=cuda, generator=gen)
    a1[torch.rand(n, 20, 20, 16, device=cuda, generator=gen) < 0.2] = 0.0
    a1s = encode_a1(a1)
    d_a2 = torch.randn(n, 2592, device=cuda, generator=gen) * 8.0
    unscale = 0.125

    grads, d_a1 = run(pkg, cuda, net.fc_w, net.workspace, a1s, d_a2, n, unscale)

    # float64 reference on the decoded inputs
    x = a1s.float().permute(0, 4, 1, 5, 2, 3, 6).reshape(n, 20, 20, 16).double()
    w = torch.as_tensor(params["l2_w"], device=cuda).double()                   # [kh, kw, cin, co]
    dy = d_a2.double().reshape(n, 9, 9, 32).permute(0, 3, 1, 2)
    xt = x.permute(0, 3, 1, 2).requires_grad_(True)
    wt = w.permute(3, 2, 0, 1).contiguous().requires_grad_(True)
    torch.nn.functional.conv2d(xt, wt, stride=2).backward(dy)
    ref_w = wt.grad.permute(2, 3, 1, 0) * unscale
    ref_b2 = dy.sum(dim=(0, 2, 3)) * unscale
    ref_da1 = xt.grad.permute(0, 2, 3, 1) * (x > 0)
    ref_b1 = ref_da1.sum(dim=(0, 1, 2)) * unscale

    raw = d_a1.view(torch.float16).reshape(2, n, 21, 21, 8)
    got_da1 = raw.float().permute(1, 2, 3, 0, 4).reshape(n, 21, 21, 16)[:, :20, :20]
    errs = dict(l1_b=rel_err(grads[4096:4112].cpu(), ref_b1.cpu()),
                l2_w=rel_err(grads[4112:4112 + 8192].reshape(4, 4, 16, 32).cpu(), ref_w.detach().cpu()),
                l2_b=rel_err(grads[4112 + 8192:].cpu(), ref_b2.cpu()),
                d_a1=rel_err(got_da1.cpu(), ref_da1.cpu()))
    print("n", n, "rel-err", errs)
    assert max(errs.values()) <= REL_TOL, errs
    assert bool(grads[:4096].eq(7.0).all())                          # l1_w is conv1 backward's
    # every byte of d_a1 is written: the rows y = 20 / x = 20 are zeros, not the 0xFF fill (a NaN)
    assert not bool(raw.isnan().any())
    assert float(raw[:, :, 20].abs().max()) == 0.0 and float(raw[:, :, :, 20].abs().max()) == 0.0

    # fixed-order sums: a second call is bit-identical
    grads2, d_a1_2 = run(pkg, cuda, net.fc_w, net.workspace, a1s, d_a2, n, unscale)
    assert torch.equal(grads.view(torch.int32), grads2.view(torch.int32))
    assert torch.equal(d_a1, d_a1_2)
