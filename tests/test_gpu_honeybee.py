"""GPU parity for the UV path (HoneyBee, default opponent mapper): <= 1 LSB on the uint8 output,
<= 1e-5 relative on the float32 receptor catches (the spectral intermediates)."""
import numpy as np
import pytest

import frames
from oracle import uv

pytestmark = pytest.mark.gpu


def _cmp(got, ref, what, max_frac=0.02):
    assert got.shape == ref.shape and got.dtype == np.uint8
    d = np.abs(got.astype(np.int16) - ref.astype(np.int16))
    assert d.max() <= 1, f"{what}: max diff {d.max()} LSB at {np.unravel_index(d.argmax(), d.shape)}"
    assert (d > 0).mean() <= max_frac, f"{what}: {(d > 0).mean():.4f} of bytes differ"


@pytest.mark.parametrize("mode", ["collapsed", "bands"])
def test_bee_against_golden(golden, golden_meta, mode):
    from animal_vision_b200.animals import HoneyBee
    h, w = golden_meta["small_hw"]
    g = golden("honeybee")
    bee = HoneyBee(spectral_mode=mode)
    for name, f in frames.parity_set(h, w):
        base, out = bee.visualize(f)
        assert base is f
        _cmp(out, g[f"opponent/white_patch/{name}"], f"{mode}/{name}")
    gw = HoneyBee(adaptation="gray_world", spectral_mode=mode)
    for name in ("noise0", "natural"):
        f = dict(frames.parity_set(h, w))[name]
        _cmp(gw.visualize(f)[1], g[f"opponent/gray_world/{name}"], f"{mode}/gray_world/{name}")


@pytest.mark.parametrize("mode", ["collapsed", "bands"])
def test_receptor_catches_1e5(golden, golden_meta, mode):
    import torch
    from animal_vision_b200.animals import HoneyBee
    h, w = golden_meta["small_hw"]
    f = frames.natural(h, w)
    ref = golden("intermediates")["bee_ubg"]
    got = HoneyBee(spectral_mode=mode).receptor_catches(torch.from_numpy(f[None]).cuda())[0].cpu().numpy()
    rel = np.abs(got - ref).max() / np.abs(ref).max()
    assert rel <= 1e-5, f"{mode}: receptor catches off by {rel:.2e} (relative to max)"
    nz = ref > 1e-3 * ref.max()
    assert (np.abs(got - ref)[nz] / ref[nz]).max() <= 1e-5


@pytest.mark.parametrize("hw", [(61, 67), (270, 480), (16, 64), (17, 65), (1080, 1920)])
def test_bee_against_oracle(hw):
    from animal_vision_b200.animals import HoneyBee
    h, w = hw
    cases = list(frames.parity_set(h, w)) if h < 1000 else [("noise0", frames.noise(h, w, 0))]
    for name, f in cases:
        _, ref = uv.honeybee_visualize(f)
        _, out = HoneyBee().visualize(f)
        _cmp(out, ref, f"{name}/{h}x{w}")


def test_bee_options_and_batch():
    import torch
    from animal_vision_b200.animals import HoneyBee
    fs = [frames.noise(90, 150, s) for s in range(3)] + [frames.natural(90, 150)]
    batch = torch.from_numpy(np.stack(fs)).cuda()
    for kw in (dict(), dict(adaptation=None), dict(blur_sigma_px=0.0), dict(blur_sigma_px=0.5), dict(assume_hsi_is_reflectance=False)):
        base, out = HoneyBee(**kw).visualize_batch(batch)
        assert base is batch
        for i, f in enumerate(fs):
            U, B, G = uv.honeybee_receptors(f, reflectance=kw.get("assume_hsi_is_reflectance", True))
            U, B, G = uv.von_kries(U, B, G, kw.get("adaptation", "white_patch"))
            s = kw.get("blur_sigma_px", 0.2)
            if s > 0:
                U, B, G = (uv.uv_gaussian_blur(c, s) for c in (U, B, G))
            srgb = uv.encode_srgb_f32(np.clip(uv.map_opponent(U, B, G), 0.0, 1.0))
            ref = (srgb * 255.0 + 0.5).astype(np.uint8)
            _cmp(out[i].cpu().numpy(), ref, f"{kw}/batch[{i}]")


def test_bee_other_mappers_against_golden(golden, golden_meta):
    """uv_mappers.py falsecolor / purple-yellow / mixed / custom matrix (honeybee.py:150-164)."""
    from animal_vision_b200.animals import HoneyBee
    h, w = golden_meta["small_hw"]
    g = golden("honeybee")
    fr = dict(frames.parity_set(h, w))
    n = 0
    for key, ref in g.items():
        mode, adapt, case = key.split("/")
        if mode == "opponent":
            continue
        kw = {}
        if mode == "custom_matrix":
            kw["custom_matrix"] = np.array([[0.9, 0.1, 0.0], [0.0, 0.3, 0.8], [0.5, 0.5, 0.1]], np.float32)
        _, out = HoneyBee(mapping_mode=mode, adaptation=adapt, **kw).visualize(fr[case])
        _cmp(out, ref, key)
        n += 1
    assert n >= 10


@pytest.mark.parametrize("mode", ["falsecolor", "uv_purple_yellow", "falsecolor_uv_mixed", "custom_matrix"])
def test_bee_other_mappers_against_oracle(mode):
    from animal_vision_b200.animals import HoneyBee
    M = np.array([[0.6, 0.2, 0.1], [0.1, 0.5, 0.3], [0.3, 0.1, 0.6]], np.float32)
    kw = {"custom_matrix": M} if mode == "custom_matrix" else {}
    for (h, w) in ((61, 67), (270, 480)):
        for name, f in frames.parity_set(h, w):
            _, ref = uv.honeybee_visualize(f, mapping_mode=mode, **kw)
            _, out = HoneyBee(mapping_mode=mode, **kw).visualize(f)
            _cmp(out, ref, f"{mode}/{name}/{h}x{w}")


def test_bee_degenerate_frames_keep_exact_percentiles():
    """Constant / two-valued frames put every pixel into one histogram bin: the candidate list then
    holds the whole frame and the select step must still return numpy's order statistics."""
    from animal_vision_b200.animals import HoneyBee
    h, w = 96, 250
    f = frames.constant(h, w, 97)
    f[:, : w // 2, 1] = 180
    for fr in (frames.constant(h, w, 0), frames.constant(h, w, 255), frames.constant(h, w, 97), f):
        _, ref = uv.honeybee_visualize(fr)
        _, out = HoneyBee().visualize(fr)
        _cmp(out, ref, "degenerate")


def test_plane_route_equals_the_second_walk():
    """The map pass of a mapper with percentiles reads the planes of the hist pass when the output is 4-byte aligned and
    W % 4 == 0, and walks the frame a second time otherwise (map_from_planes in csrc/k3_uv.cu).  Both routes give identical
    bytes: every case runs once into a packed output and once into a view that starts one pixel (3 bytes) into a wider
    buffer, which always takes the walk."""
    import torch
    from animal_vision_b200.animals import HoneyBee
    g = torch.Generator().manual_seed(5)
    for n, h, w in ((3, 270, 480), (1, 123, 236), (2, 64, 1100), (1, 37, 50)):
        fr = torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, generator=g).cuda()
        fr[0, : h // 2] //= 3
        wide = torch.zeros((n, h, w + 24, 3), dtype=torch.uint8, device="cuda")
        wide[:, :, 8:8 + w] = fr
        cases = [(kw, fr) for kw in ({}, {"adaptation": "gray_world"}, {"blur_sigma_px": None}, {"blur_sigma_px": 0.6},
                                     {"adaptation": None}, {"mapping_mode": "falsecolor"}, {"mapping_mode": "uv_purple_yellow"},
                                     {"mapping_mode": "falsecolor_uv_mixed"},
                                     {"mapping_mode": "falsecolor", "adaptation": "gray_world", "blur_sigma_px": 0.6})]
        cases.append(({}, wide[:, :, 8:8 + w]))            # strided input rows
        for kw, src in cases:
            bee = HoneyBee(**kw)
            _, packed = bee.visualize_batch(src)
            shifted = torch.empty((n, h, w + 1, 3), dtype=torch.uint8, device="cuda")[:, :, 1:]
            bee.visualize_batch(src, shifted)
            assert torch.equal(packed, shifted), ((n, h, w), kw, src.is_contiguous())
