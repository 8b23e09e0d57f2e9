"""GPU: arl_conv1_backward on its own -- conv1's weight gradient from the u8 ring and the fp16 d_a1
grid -- against a float64 weight gradient of the decoded stacks.  The shapes cover one sample,
windows shorter than the kernel's (t_max < 5), t_max not a multiple of it (7), several windows per
env (20) and the bench sizes; every ring window wraps past the last slot."""
import pytest
import torch

from util import REL_TOL, rel_err

pytestmark = pytest.mark.gpu

GRID = 441                                   # 21 x 21 rows of 16 B per ring plane / d_a1 co group


def run(pkg, ring, d_a1, B, slots, first, T, unscale, cuda):
    lib = pkg._cabi.load()
    P = pkg._cabi.ptr
    grads = torch.full((4096 + 64,), 7.0, device=cuda)
    sms = torch.cuda.get_device_properties(cuda).multi_processor_count
    workspace = torch.empty(sms * 4096, device=cuda)
    assert lib.arl_conv1_backward(P(ring), P(d_a1), P(grads), P(workspace), B, slots, first, T, unscale,
                                  pkg._cabi.stream_ptr()) == 0
    torch.cuda.synchronize()
    return grads


def reference(ring, d_a1, B, slots, first, T, unscale):
    """float64 dW1[kh, kw, cin, co] = sum over samples and output pixels of x[4y+kh, 4x+kw, cin] *
    dy[y, x, co], x = the stacked planes / 255, on the space-to-depth grid: block (y', x') of plane
    cin holds pixel (4y'+i, 4x'+j) at byte i*4 + j."""
    dw = torch.zeros(8, 8, 4, 16, dtype=torch.float64, device=ring.device)
    dy_all = d_a1.view(2, T, B, 21, 21, 8)
    for t in range(T):
        slot = [(first + t + c) % slots for c in range(4)]
        x = ring[:, slot].reshape(B, 4, 21, 21, 4, 4).double()                         # b, cin, y', x', i, j
        dy = dy_all[:, t, :, :20, :20].double().permute(1, 2, 3, 0, 4).reshape(B * 400, 16)
        for a in range(2):
            for bb in range(2):
                xs = x[:, :, a:a + 20, bb:bb + 20].permute(0, 2, 3, 1, 4, 5).reshape(B * 400, 64)
                g = (xs.t() @ dy).reshape(4, 4, 4, 16)                                  # cin, i, j, co
                dw[4 * a:4 * a + 4, 4 * bb:4 * bb + 4] += g.permute(1, 2, 0, 3)
    return dw * (unscale / 255.0)


@pytest.mark.parametrize("B,T", [(1, 1), (3, 2), (7, 5), (5, 7), (37, 20), (4096, 5), (4096, 20)])
def test_conv1_backward_vs_float64(pkg, cuda, B, T):
    gen = torch.Generator(device=cuda).manual_seed(B * 100 + T)
    slots = T + 5
    first = slots - 1 - T % 3                # the T + 3 planes of an env wrap past the last slot
    ring = torch.randint(0, 256, (B, slots, GRID * 16), dtype=torch.uint8, device=cuda, generator=gen)
    dy = torch.randn(2, T * B, 21, 21, 8, device=cuda, generator=gen) * 4.0
    dy[:, :, 20] = 0.0                       # no conv1 output at y = 20 / x = 20
    dy[:, :, :, 20] = 0.0
    d_a1 = dy.half().contiguous()
    unscale = 0.25

    grads = run(pkg, ring, d_a1, B, slots, first, T, unscale, cuda)
    ref = reference(ring, d_a1, B, slots, first, T, unscale)
    err = rel_err(grads[:4096].reshape(8, 8, 4, 16).cpu(), ref.cpu())
    print("B", B, "T", T, "first_slot", first, "of", slots, "l1_w rel-err", err)
    assert err <= REL_TOL, err
    assert bool(grads[4096:].eq(7.0).all())  # l1_b and beyond are conv2 backward's

    # fixed-order sums: a second call is bit-identical
    grads2 = run(pkg, ring, d_a1, B, slots, first, T, unscale, cuda)
    assert torch.equal(grads.view(torch.int32), grads2.view(torch.int32))
