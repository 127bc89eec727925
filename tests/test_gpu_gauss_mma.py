"""GPU parity of the tensor-core Gaussian (csrc/k2_gauss.cu gauss_mma_kernel) against the oracle.

A rank-2 matrix with radius 5..16 takes the tensor path with single f16 operands; radius <= 4 (Squirrel) stays on the exact
CUDA-core kernel.  Tolerance: BASELINE.json north_star, <= 1 LSB on uint8 output; the differing-byte fraction is asserted
too (measured: 0.3 .. 1.4 % of all bytes)."""
import numpy as np
import pytest

import frames
from oracle import mammals as M

pytestmark = pytest.mark.gpu


def test_every_radius():
    """squirrel 7 taps, lion 11, fox 11, wolf 13, bear 15, elephant 15, raccoon 17, dog 29 taps."""
    import torch
    import animal_vision_b200.animals as A
    for name in ("squirrel", "lion", "wolf", "bear", "elephant", "raccoon", "dog"):
        sp = A.MAMMALS[name]()
        worst, tot, dif = 0, 0, 0
        for (h, w) in ((270, 480), (61, 67), (40, 1100), (37, 1), (8, 200)):
            for case, f in frames.parity_set(h, w):
                ref = M.mammal_visualize(f, name)[1]
                out = sp.visualize(f)[1]
                d = np.abs(out.astype(np.int16) - ref.astype(np.int16))
                worst = max(worst, int(d.max())); tot += d.size; dif += int((d > 0).sum())
        assert worst <= 1, (name, worst)
        assert dif / tot <= 0.03, (name, dif / tot)
        # unaligned rows (scalar producer / byte-wise store path) and a strided batch must match the packed result
        f0 = frames.natural(300, 520)
        batch = torch.from_numpy(np.stack([f0, frames.noise(300, 520, 4)])).cuda()
        _, ref_out = sp.visualize_batch(batch)
        wide = torch.zeros((2, 300, 600, 3), dtype=torch.uint8, device="cuda")
        wide[:, :, 39:559] = batch
        _, out2 = sp.visualize_batch(wide[:, :, 39:559])
        assert torch.equal(out2, ref_out), name


def test_default_route_dog_1080p_and_canaries():
    """Default dispatch (tensor path for Dog): 1080p parity with the output inside a canary-filled buffer
    (padded rows: the staged 128-bit store path must not touch the pad)."""
    import torch
    from animal_vision_b200.animals import Dog
    f0, f1 = frames.bars(1080, 1920), frames.natural(1080, 1920)
    refs = [M.mammal_visualize(f, "dog")[1] for f in (f0, f1)]
    batch = torch.from_numpy(np.stack([f0, f1])).cuda()
    big = torch.full((2, 1080 + 8, 1920 + 16, 3), 0xA5, dtype=torch.uint8, device="cuda")
    out = big[:, 4:-4, 16:1936]                    # a view with padded rows and frames inside the canary buffer
    Dog().visualize_batch(batch, out)
    for i in range(2):
        d = np.abs(out[i].cpu().numpy().astype(np.int16) - refs[i].astype(np.int16))
        assert d.max() <= 1 and (d > 0).mean() <= 0.01, (i, d.max(), (d > 0).mean())
    mask = torch.ones_like(big, dtype=torch.bool)
    mask[:, 4:-4, 16:1936] = False
    assert bool((big[mask] == 0xA5).all()), "canary bytes around the output were overwritten"
