"""K10 device PNG encode (animal_vision_b200/png.py, csrc/k10_png.cu) and the server path that uses it: the gate is byte
identity with cv2.imencode(".png"), no tolerance."""
import base64

import cv2
import numpy as np
import pytest

import frames

pytestmark = pytest.mark.gpu

SHAPES = ((1, 1), (1, 2), (2, 1), (3, 7), (5, 5), (17, 33), (40, 41), (61, 89), (300, 1), (1, 5000), (1, 5461),
          (1, 5462), (129, 42), (5, 1637), (135, 241), (1080, 1920))


def _cv2(img):
    ok, enc = cv2.imencode(".png", img)
    assert ok
    return enc.tobytes()


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


@pytest.fixture(scope="module")
def encode():
    from animal_vision_b200.png import encode_png
    return encode_png


@pytest.mark.parametrize("hw", SHAPES)
def test_parity_set_equals_cv2(torch, encode, hw):
    named = list(frames.parity_set(*hw)) + [("noise1", frames.noise(*hw, 1))]
    batch = torch.from_numpy(np.stack([f for _, f in named])).cuda()
    got = encode(batch)
    for (name, img), g in zip(named, got):
        assert g == _cv2(img), f"{name} {hw}"


def test_4k_equals_cv2(torch, encode):
    for name, img in (("natural", frames.natural(2160, 3840)), ("noise", frames.noise(2160, 3840, 1)),
                      ("full", frames.constant(2160, 3840, 255)), ("zeros", frames.constant(2160, 3840, 0))):
        assert encode(torch.from_numpy(img[None]).cuda())[0] == _cv2(img), name


def test_block_and_chunk_edges(torch, encode):
    """Symbol counts that are multiples of 16383 (empty final block) and zlib streams of whole IDAT payloads."""
    for hw in ((129, 42), (258, 42), (6, 1820), (5, 1637), (20, 409), (80, 102)):
        img = frames.noise(*hw, 0)
        assert encode(torch.from_numpy(img[None]).cuda())[0] == _cv2(img), hw


def test_mixed_batch_equals_one_at_a_time(torch, encode):
    h, w = 72, 104
    imgs = [frames.natural(h, w, s) for s in range(3)] + [frames.noise(h, w, 4), frames.impulses(h, w), frames.bars(h, w),
                                                          frames.constant(h, w, 255), frames.checker(h, w)]
    batch = torch.from_numpy(np.stack(imgs)).cuda()
    together = encode(batch)
    assert len(together) == 8
    for k, img in enumerate(imgs):
        assert together[k] == encode(batch[k:k + 1])[0] == _cv2(img)


def test_side_stream_gives_the_same_bytes(torch, encode):
    img = frames.natural(240, 320)
    dev = torch.from_numpy(img[None]).cuda()
    ref = encode(dev)[0]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        got = encode(dev)[0]
    assert got == ref == _cv2(img)


def test_strided_crop(torch, encode):
    big = np.stack([frames.natural(300, 400, 1), frames.noise(300, 400, 2)])
    dev = torch.from_numpy(big).cuda()
    crop = dev[:, 17:17 + 123, 31:31 + 201]                 # rows and frames strided, pixels packed
    assert not crop.is_contiguous()
    got = encode(crop)
    for k in range(2):
        assert got[k] == _cv2(np.ascontiguousarray(big[k, 17:140, 31:232]))


def test_lengths_within_bound(torch, encode):
    from animal_vision_b200 import _abi
    lib = _abi.load()
    for hw in ((1, 1), (5, 5), (129, 42), (300, 400), (1080, 1920)):
        imgs = [f for _, f in frames.parity_set(*hw)]
        got = encode(torch.from_numpy(np.stack(imgs)).cuda())
        assert max(len(g) for g in got) <= lib.avb_png_bound_bytes(*hw)


def test_bad_arguments_raise(torch, encode):
    from animal_vision_b200 import _abi
    from animal_vision_b200._abi import AvbError
    dev = torch.zeros((1, 8, 8, 3), dtype=torch.uint8, device="cuda")
    for bad in (dev.cpu(), dev.float(), dev[..., :2], dev[0], np.zeros((1, 8, 8, 3), np.uint8)):
        with pytest.raises(AvbError):
            encode(bad)
    assert encode(dev[:0]) == []
    lib = _abi.load()
    assert lib.avb_png_bound_bytes(0, 8) < 0 and lib.avb_png_bound_bytes(8, 65536) < 0
    assert lib.avb_png_workspace_bytes(1, 65536, 8) < 0 and lib.avb_png_workspace_bytes(0, 8, 8) < 0
    from animal_vision_b200 import tables
    from animal_vision_b200.engine import _fptr
    hdr = np.frombuffer(tables.png_header(8, 8), np.uint8)
    slot = int(lib.avb_png_bound_bytes(8, 8))
    ws = torch.empty(int(lib.avb_png_workspace_bytes(1, 8, 8)) + 16, dtype=torch.uint8, device="cuda")
    out = torch.empty(slot, dtype=torch.uint8, device="cuda")
    lens = torch.empty(1, dtype=torch.int64, device="cuda")
    st = torch.cuda.current_stream().cuda_stream

    def call(n=1, H=8, W=8, hp=_fptr(hdr), hl=int(hdr.size), o=out.data_ptr(), sl=slot, lp=lens.data_ptr(),
             wp=ws.data_ptr(), rs=24, fs=192):
        return lib.avb_png_encode_u8(dev.data_ptr(), n, H, W, fs, rs, hp, hl, o, sl, lp, wp, st)
    assert call() == 0
    for kw in (dict(H=0), dict(W=65536), dict(n=0), dict(hp=None), dict(o=None), dict(lp=None), dict(wp=None),
               dict(sl=slot - 1), dict(wp=ws.data_ptr() + 8), dict(hl=_abi.AVB_PNG_HEADER_LEN - 1), dict(rs=23),
               dict(n=2, fs=100)):
        assert call(**kw) == -1, kw
        assert lib.avb_last_error()
    torch.cuda.synchronize()
    assert bytes(out[:int(lens.item())].cpu().numpy()) == _cv2(np.zeros((8, 8, 3), np.uint8))


SPECIES = ("dog", "cat", "honeybee", "reindeer")


@pytest.mark.parametrize("animal", SPECIES)
def test_process_image_png_through_the_device_batcher(animal):
    from animal_vision_b200 import animals as A
    from animal_vision_b200 import serving
    img = frames.natural(120, 176, 3)
    req = _cv2(img)
    decoded = cv2.imdecode(np.frombuffer(req, np.uint8), cv2.IMREAD_COLOR)
    view = getattr(A, serving.SERVER_KEYS[animal])().visualize(decoded)[1]
    with serving.FrameBatcher(max_delay_ms=50.0) as fb:
        uri = serving.process_image_png(req, animal, batcher=fb)
    assert uri == "data:image/png;base64," + base64.b64encode(_cv2(view)).decode("utf-8")


def test_pixel_jpeg_and_png_requests_share_a_batch():
    from animal_vision_b200 import animals as A
    from animal_vision_b200 import serving
    imgs = [frames.natural(64, 96, s) for s in range(6)]
    views = A.Dog().visualize_batch(__import__("torch").from_numpy(np.stack(imgs)).cuda())[1].cpu().numpy()
    kinds = ["pix", "png", "jpeg", "png", "pix", "jpeg"]
    with serving.FrameBatcher(max_batch=16, max_delay_ms=200.0) as fb:
        futs = [fb.submit(f, "dog") if k == "pix" else fb.submit_png(f, "dog") if k == "png" else fb.submit_jpeg(f, "dog")
                for k, f in zip(kinds, imgs)]
        res = [f.result(60) for f in futs]
        human = fb.submit_png(imgs[0], "human").result(5)
    assert fb.batches == [("dog", 6)]
    for k, r in zip(kinds, range(6)):
        got = res[r]
        if k == "pix":
            assert isinstance(got, np.ndarray) and np.array_equal(got, views[r])
        elif k == "png":
            assert got == _cv2(views[r])
        else:
            assert got == cv2.imencode(".jpg", views[r])[1].tobytes()
    assert human == _cv2(imgs[0])
