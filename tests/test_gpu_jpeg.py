"""K8 device JPEG encode (animal_vision_b200/jpeg.py, csrc/k8_jpeg.cu) and the server path that uses it: the gate is byte
identity with cv2.imencode(".jpg"), no tolerance."""
import base64

import cv2
import numpy as np
import pytest

import frames

pytestmark = pytest.mark.gpu

QUALITIES = (10, 50, 75, 95, 100)
SHAPES = ((1, 1), (7, 9), (8, 8), (16, 16), (17, 33), (37, 53), (135, 241), (1080, 1920))


def _cv2(img, q=95):
    ok, enc = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q])
    assert ok
    return enc.tobytes()


@pytest.fixture(scope="module")
def torch():
    import torch as t
    return t


@pytest.fixture(scope="module")
def encode():
    from animal_vision_b200.jpeg import encode_jpeg
    return encode_jpeg


@pytest.mark.parametrize("q", QUALITIES)
@pytest.mark.parametrize("hw", SHAPES)
def test_parity_set_equals_cv2(torch, encode, q, hw):
    named = list(frames.parity_set(*hw))
    batch = torch.from_numpy(np.stack([f for _, f in named])).cuda()
    got = encode(batch, q)
    for (name, img), g in zip(named, got):
        assert g == _cv2(img, q), f"{name} {hw} q={q}"


@pytest.mark.parametrize("q", (75, 95, 100))
def test_4k_equals_cv2(torch, encode, q):
    for name, img in (("natural", frames.natural(2160, 3840)), ("noise", frames.noise(2160, 3840, 1)),
                      ("full", frames.constant(2160, 3840, 255))):
        assert encode(torch.from_numpy(img[None]).cuda(), q)[0] == _cv2(img, q), f"{name} q={q}"


def test_mixed_batch_equals_one_at_a_time(torch, encode):
    h, w = 72, 104
    imgs = [frames.natural(h, w, s) for s in range(3)] + [frames.noise(h, w, 4), frames.impulses(h, w), frames.bars(h, w),
                                                          frames.constant(h, w, 255), frames.checker(h, w)]
    batch = torch.from_numpy(np.stack(imgs)).cuda()
    together = encode(batch, 90)
    assert len(together) == 8
    for k, img in enumerate(imgs):
        assert together[k] == encode(batch[k:k + 1], 90)[0] == _cv2(img, 90)


def test_side_stream_gives_the_same_bytes(torch, encode):
    img = frames.natural(240, 320)
    dev = torch.from_numpy(img[None]).cuda()
    ref = encode(dev, 95)[0]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        got = encode(dev, 95)[0]
    assert got == ref == _cv2(img)


def test_strided_crop(torch, encode):
    big = np.stack([frames.natural(300, 400, 1), frames.noise(300, 400, 2)])
    dev = torch.from_numpy(big).cuda()
    crop = dev[:, 17:17 + 123, 31:31 + 201]                 # rows and frames strided, pixels packed
    assert not crop.is_contiguous()
    got = encode(crop, 85)
    for k in range(2):
        assert got[k] == _cv2(np.ascontiguousarray(big[k, 17:140, 31:232]), 85)


def test_bad_arguments_raise(torch, encode):
    from animal_vision_b200 import _abi
    from animal_vision_b200._abi import AvbError
    dev = torch.zeros((1, 8, 8, 3), dtype=torch.uint8, device="cuda")
    for bad in (dict(frames=dev.cpu()), dict(frames=dev.float()), dict(frames=dev[..., :2]), dict(frames=dev[0]),
                dict(frames=dev, quality=0), dict(frames=dev, quality=101), dict(frames=dev, quality=9.5)):
        with pytest.raises(AvbError):
            encode(**{"quality": 95, **bad})
    lib = _abi.load()
    assert lib.avb_jpeg_bound_bytes(0, 8) < 0 and lib.avb_jpeg_bound_bytes(8, 65536) < 0
    assert lib.avb_jpeg_workspace_bytes(1, 65536, 8) < 0
    from animal_vision_b200 import tables
    from animal_vision_b200.engine import _fptr
    hdr = np.frombuffer(tables.jpeg_header(8, 8, 95), np.uint8)
    qt = np.ascontiguousarray(tables.jpeg_quant_tables(95))
    slot = int(lib.avb_jpeg_bound_bytes(8, 8))
    ws = torch.empty(int(lib.avb_jpeg_workspace_bytes(1, 8, 8)) + 16, dtype=torch.uint8, device="cuda")
    out = torch.empty(slot, dtype=torch.uint8, device="cuda")
    lens = torch.empty(1, dtype=torch.int64, device="cuda")
    st = torch.cuda.current_stream().cuda_stream

    def call(H=8, W=8, hp=_fptr(hdr), hl=int(hdr.size), qp=_fptr(qt), o=out.data_ptr(), sl=slot, wp=ws.data_ptr(), rs=24):
        return lib.avb_jpeg_encode_u8(dev.data_ptr(), 1, H, W, 192, rs, hp, hl, qp, o, sl, lens.data_ptr(), wp, st)
    assert call() == 0
    for kw in (dict(H=0), dict(W=65536), dict(hp=None), dict(qp=None), dict(o=None), dict(wp=None), dict(sl=slot - 1),
               dict(wp=ws.data_ptr() + 8), dict(hl=_abi.AVB_JPEG_HEADER_MAX + 1), dict(rs=23)):
        assert call(**kw) == -1, kw
        assert lib.avb_last_error()
    torch.cuda.synchronize()


SPECIES = ("dog", "cat", "honeybee", "reindeer")


@pytest.mark.parametrize("animal", SPECIES)
def test_process_image_through_the_device_batcher(animal):
    from animal_vision_b200 import animals as A
    from animal_vision_b200 import serving
    img = frames.natural(120, 176, 3)
    req = _cv2(img)
    decoded = cv2.imdecode(np.frombuffer(req, np.uint8), cv2.IMREAD_COLOR)
    view = getattr(A, serving.SERVER_KEYS[animal])().visualize(decoded)[1]
    with serving.FrameBatcher(max_delay_ms=50.0) as fb:
        uri = serving.process_image(req, animal, batcher=fb)
    assert uri == "data:image/jpeg;base64," + base64.b64encode(_cv2(view)).decode("utf-8")


def test_jpeg_and_pixel_requests_share_a_batch():
    from animal_vision_b200 import animals as A
    from animal_vision_b200 import serving
    imgs = [frames.natural(64, 96, s) for s in range(6)]
    views = A.Dog().visualize_batch(__import__("torch").from_numpy(np.stack(imgs)).cuda())[1].cpu().numpy()
    with serving.FrameBatcher(max_batch=16, max_delay_ms=200.0) as fb:
        futs = [fb.submit_jpeg(f, "dog") if k % 2 else fb.submit(f, "dog") for k, f in enumerate(imgs)]
        res = [f.result(60) for f in futs]
        human = fb.submit_jpeg(imgs[0], "human").result(5)
    assert len(fb.batches) == 1 and fb.batches[0] == ("dog", 6)
    for k, r in enumerate(res):
        if k % 2:
            assert r == _cv2(views[k])
        else:
            assert isinstance(r, np.ndarray) and np.array_equal(r, views[k])
    assert human == _cv2(imgs[0])
