"""K1 loads its frames with an L2 evict_first hint up to kK1EvictFirstMaxEnvs (8192) frames per
launch and without it above (csrc/preprocess.cu): both instantiations must give the oracle's
screens, so the batch sizes on either side of the switch are checked here."""
import numpy as np
import pytest
import torch

from oracle import preprocess as P
from util import unblock

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("B", [8192, 8193])
def test_both_sides_of_the_evict_first_switch_match_the_oracle(pkg, cuda, B):
    g = torch.Generator(device=cuda).manual_seed(B)
    base = torch.randint(0, 256, (64, 210, 160, 3), dtype=torch.uint8, device=cuda, generator=g)
    perm = torch.randint(0, 64, (B,), device=cuda, generator=g)
    frames = base[perm].contiguous()
    ring = torch.full((B, 5, 84, 84), 7, dtype=torch.uint8, device=cuda)
    pkg._cabi.call("arl_preprocess_push", pkg._cabi.ptr(frames), pkg._cabi.ptr(ring), B, 5, 3, 1,
                   pkg._cabi.stream_ptr())
    torch.cuda.synchronize()
    ref = torch.as_tensor(P.screen(base.cpu().numpy()), device=cuda)
    assert bool((unblock(ring[:, 3]) == ref[perm]).all())
    assert bool((ring[:, [0, 1, 2, 4]] == 7).all())
