"""Cat outputs byte for byte: SHA-256 digests of both outputs (centre zoom and cat view) of a fixed set of inputs,
recorded on a B200 from the kernels before the dedicated cat warp kernel replaced the shared one.  The set reaches
every branch of the Cat launch: 4K batches, 1080p, an odd width, unaligned row strides, frames whose maximum is <= 1
(the other normalisation branch, and the fixup launch without the warp), ENABLE_FOV_WARP = False, other blur radii,
and a full-rank colour matrix (three planes).

    python tests/test_gpu_cat_bytes.py --write tests/golden/cat_bytes_sha256.json    # re-record (changes the yardstick)
"""
import hashlib
import json
import os
import sys

import numpy as np
import pytest

import frames

DIGESTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cat_bytes_sha256.json")

# not rank 2: the cat kernel blurs three planes
FULL_RANK = np.array([[0.62, 0.31, 0.07], [0.18, 0.71, 0.11], [0.05, 0.22, 0.73]], np.float32)


def _batch(torch, fs):
    return torch.from_numpy(np.stack(fs)).cuda()


def _strided(torch, x, pad_rows=3, pad_cols=5):
    """x [N,H,W,3] copied into a view whose row stride is 3 (W + 2 pad_cols) bytes: neither 4- nor 16-byte aligned."""
    n, h, w, _ = x.shape
    big = torch.zeros((n + 1, h + 2 * pad_rows, (w + 2 * pad_cols) * 3), dtype=torch.uint8, device=x.device)
    view = big[1:, pad_rows:pad_rows + h, pad_cols * 3 + 1:pad_cols * 3 + 1 + 3 * w].unflatten(2, (w, 3))
    view.copy_(x)
    return view


def _run(sp, x, out=None):
    human, cat = sp.visualize_batch(x, out=out)
    return human.cpu().numpy(), cat.cpu().numpy()


def case_4k(torch, Cat):
    return _run(Cat(), _batch(torch, [frames.noise(2160, 3840, 0), frames.natural(2160, 3840), frames.noise(2160, 3840, 1)]))


def case_1080p(torch, Cat):
    return Cat().visualize(frames.natural(1080, 1920, seed=7))


def case_odd_width(torch, Cat):
    return _run(Cat(), _batch(torch, [frames.noise(301, 999, 2), frames.natural(301, 999)]))


def case_unaligned_strides(torch, Cat):
    x = _batch(torch, [frames.natural(270, 1283), frames.noise(270, 1283, 3)])
    outs = (_strided(torch, torch.zeros_like(x), 2, 3), _strided(torch, torch.zeros_like(x), 1, 7))
    return _run(Cat(), _strided(torch, x), out=outs)


def case_max_le1(torch, Cat):
    return _run(Cat(), _batch(torch, [frames.noise(540, 960, 4), frames.le1(540, 960), frames.le1(540, 960, seed=9)]))


def case_without_fov_warp(torch, Cat):
    NoWarp = type("NoWarp", (Cat,), {"ENABLE_FOV_WARP": False})
    return _run(NoWarp(), _batch(torch, [frames.natural(1080, 1920), frames.le1(1080, 1920)]))


def _sigma(sigma):
    def case(torch, Cat):
        Wide = type("Wide", (Cat,), {"SIGMA": sigma})
        return _run(Wide(), _batch(torch, [frames.natural(1080, 1920), frames.noise(1080, 1920, 5), frames.le1(1080, 1920)]))
    return case


def case_full_rank(torch, Cat):
    """avb_cat_u8 with a full-rank matrix (Cat.LM_ALPHA always gives rank 2), both normalisation branches."""
    from animal_vision_b200 import tables
    from animal_vision_b200.engine import get_engine
    c = Cat()
    x = _batch(torch, [frames.natural(1080, 1920), frames.le1(1080, 1920), frames.noise(1080, 1920, 6)])
    eng = get_engine(x.device)
    n, H, W, _ = x.shape
    warp = eng._dev(tables.cat_warp_device_table(W, c.CAMERA_HFOV_DEG, c.CAT_PER_EYE_HALF_FOV_DEG, c.CAT_OVERLAP_DEG))
    scale = tables.cat_zoom_scale(c.CAMERA_HFOV_DEG, c.CAT_PER_EYE_HALF_FOV_DEG, c.CAT_TO_HUMAN_RATIO)
    zoom = eng._dev(tables.center_zoom_tables(W, H, scale))
    human, cat = torch.empty_like(x), torch.empty_like(x)
    eng.cat(x, human, cat, FULL_RANK, tables.gaussian_taps(tables.gaussian_ksize(c.SIGMA), c.SIGMA), warp, zoom)
    torch.cuda.synchronize()
    return human.cpu().numpy(), cat.cpu().numpy()


CASES = {
    "4k_batch": case_4k,
    "1080p": case_1080p,
    "odd_width": case_odd_width,
    "unaligned_strides": case_unaligned_strides,
    "max_le1": case_max_le1,
    "without_fov_warp": case_without_fov_warp,
    "sigma_0.25": _sigma(0.25),      # ksize 3
    "sigma_2": _sigma(2.0),          # ksize 17
    "sigma_4": _sigma(4.0),          # ksize 33
    "full_rank": case_full_rank,
}


def digests(name):
    import torch
    from animal_vision_b200.animals import Cat
    human, cat = CASES[name](torch, Cat)
    return {"human": hashlib.sha256(np.ascontiguousarray(human).tobytes()).hexdigest(),
            "cat": hashlib.sha256(np.ascontiguousarray(cat).tobytes()).hexdigest()}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_cat_bytes_unchanged(name):
    with open(DIGESTS) as fh:
        want = json.load(fh)[name]
    assert digests(name) == want


if __name__ == "__main__":
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path[:0] = [root, os.path.dirname(os.path.abspath(__file__))]
    assert sys.argv[1] == "--write", __doc__
    out = {name: digests(name) for name in sorted(CASES)}
    with open(sys.argv[2], "w") as fh:
        json.dump(out, fh, indent=1, sort_keys=True)
        fh.write("\n")
    print(json.dumps(out, indent=1))
