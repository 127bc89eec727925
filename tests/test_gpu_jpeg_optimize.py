"""K8's optimized mode (encode_jpeg(..., optimize=True), avb_jpeg_opt_encode_u8 / avb_jpeg_opt_encode_rgb_u8) and the
server and video paths that offer it: the gate is byte identity with cv2.imencode(".jpg") with IMWRITE_JPEG_OPTIMIZE,
no tolerance."""
import base64

import cv2
import numpy as np
import pytest

import frames

pytestmark = pytest.mark.gpu

QUALITIES = (1, 10, 50, 75, 95, 100)
SHAPES = ((1, 1), (7, 9), (8, 8), (16, 16), (17, 33), (37, 53), (135, 241), (1080, 1920))


def _cv2(img, q=95, optimize=True):
    params = [cv2.IMWRITE_JPEG_QUALITY, q] + ([cv2.IMWRITE_JPEG_OPTIMIZE, 1] if optimize else [])
    ok, enc = cv2.imencode(".jpg", np.ascontiguousarray(img), params)
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
    got = encode(batch, q, optimize=True)
    rgb = encode(batch, q, rgb=True, optimize=True)
    for (name, img), g, r in zip(named, got, rgb):
        assert g == _cv2(img, q), f"{name} {hw} q={q}"
        assert r == _cv2(img[..., ::-1], q), f"rgb {name} {hw} q={q}"


@pytest.mark.parametrize("q", (75, 95, 100))
def test_4k_equals_cv2(torch, encode, q):
    for name, img in (("natural", frames.natural(2160, 3840)), ("noise", frames.noise(2160, 3840, 1)),
                      ("constant", frames.constant(2160, 3840, 255))):
        got = encode(torch.from_numpy(img[None]).cuda(), q, optimize=True)[0]
        assert got == _cv2(img, q), f"{name} q={q}"
        if name == "natural":
            assert len(got) < len(_cv2(img, q, optimize=False))


def test_code_length_limiting(torch, encode):
    """Codes longer than 16 bits are folded down (the oracle's host test asserts that this frame takes that branch)."""
    img = frames.natural(720, 1280, 4)
    assert encode(torch.from_numpy(img[None]).cuda(), 100, optimize=True)[0] == _cv2(img, 100)


def test_mixed_batch_gets_tables_per_frame(torch, encode):
    h, w = 72, 104
    imgs = [frames.natural(h, w, s) for s in range(3)] + [frames.noise(h, w, 4), frames.impulses(h, w), frames.bars(h, w),
                                                          frames.constant(h, w, 255), frames.checker(h, w)]
    batch = torch.from_numpy(np.stack(imgs)).cuda()
    together = encode(batch, 90, optimize=True)
    assert len(together) == 8 and len(set(together)) == 8
    for k, img in enumerate(imgs):
        assert together[k] == encode(batch[k:k + 1], 90, optimize=True)[0] == _cv2(img, 90)


def test_standard_mode_is_unchanged_beside_it(torch, encode):
    img = frames.natural(240, 320)
    dev = torch.from_numpy(img[None]).cuda()
    assert encode(dev, 95, optimize=True)[0] == _cv2(img)
    assert encode(dev, 95)[0] == _cv2(img, optimize=False)
    assert encode(dev, 95, optimize=True)[0] == _cv2(img)


def test_side_stream_gives_the_same_bytes(torch, encode):
    img = frames.natural(240, 320)
    dev = torch.from_numpy(img[None]).cuda()
    ref = encode(dev, 95, optimize=True)[0]
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        got = encode(dev, 95, optimize=True)[0]
    assert got == ref == _cv2(img)


def test_strided_crop(torch, encode):
    big = np.stack([frames.natural(300, 400, 1), frames.noise(300, 400, 2)])
    crop = torch.from_numpy(big).cuda()[:, 17:17 + 123, 31:31 + 201]
    assert not crop.is_contiguous()
    for k, g in enumerate(encode(crop, 85, optimize=True)):
        assert g == _cv2(big[k, 17:140, 31:232], 85)
    for k, g in enumerate(encode(crop, 85, rgb=True, optimize=True)):
        assert g == _cv2(big[k, 17:140, 31:232, ::-1], 85)


def test_bad_arguments_raise(torch, encode):
    from animal_vision_b200 import _abi, tables
    from animal_vision_b200._abi import AvbError
    from animal_vision_b200.engine import _fptr
    dev = torch.zeros((1, 8, 8, 3), dtype=torch.uint8, device="cuda")
    for bad in (dict(frames=dev.cpu()), dict(frames=dev[..., :2]), dict(frames=dev, quality=0)):
        with pytest.raises(AvbError):
            encode(**{"quality": 95, "optimize": True, **bad})
    lib = _abi.load()
    assert lib.avb_jpeg_opt_workspace_bytes(1, 65536, 8) < 0 and lib.avb_jpeg_opt_workspace_bytes(0, 8, 8) < 0
    assert lib.avb_jpeg_opt_workspace_bytes(4, 64, 64) > lib.avb_jpeg_workspace_bytes(4, 64, 64)
    pre = np.frombuffer(tables.jpeg_header_prefix(8, 8, 95), np.uint8)
    sos = np.frombuffer(tables.JPEG_SOS, np.uint8)
    qt = np.ascontiguousarray(tables.jpeg_quant_tables(95))
    slot = int(lib.avb_jpeg_bound_bytes(8, 8))
    ws = torch.empty(int(lib.avb_jpeg_opt_workspace_bytes(1, 8, 8)) + 16, dtype=torch.uint8, device="cuda")
    out = torch.empty(slot, dtype=torch.uint8, device="cuda")
    lens = torch.empty(1, dtype=torch.int64, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    top = _abi.AVB_JPEG_HEADER_MAX - 432                   # prefix + SOS room beside the largest four DHT segments

    for fn in (lib.avb_jpeg_opt_encode_u8, lib.avb_jpeg_opt_encode_rgb_u8):
        def call(H=8, W=8, pp=_fptr(pre), pl=int(pre.size), sp=_fptr(sos), sl=int(sos.size), qp=_fptr(qt),
                 o=out.data_ptr(), ss=slot, wp=ws.data_ptr(), rs=24):
            return fn(dev.data_ptr(), 1, H, W, 192, rs, pp, pl, sp, sl, qp, o, ss, lens.data_ptr(), wp, st)
        assert call() == 0
        torch.cuda.synchronize()
        assert bytes(out[:int(lens[0])].cpu().numpy()) == _cv2(np.zeros((8, 8, 3), np.uint8))
        for kw in (dict(H=0), dict(W=65536), dict(pp=None), dict(sp=None), dict(qp=None), dict(o=None), dict(wp=None),
                   dict(ss=slot - 1), dict(wp=ws.data_ptr() + 8), dict(pl=1), dict(sl=1), dict(rs=23),
                   dict(pl=top - int(sos.size) + 1)):
            assert call(**kw) == -1, kw
            assert lib.avb_last_error()
    torch.cuda.synchronize()


SPECIES = ("dog", "cat", "honeybee")


@pytest.mark.parametrize("animal", SPECIES)
def test_process_image_optimized(animal):
    from animal_vision_b200 import animals as A
    from animal_vision_b200 import serving
    img = frames.natural(120, 176, 3)
    req = _cv2(img, optimize=False)
    decoded = cv2.imdecode(np.frombuffer(req, np.uint8), cv2.IMREAD_COLOR)
    view = getattr(A, serving.SERVER_KEYS[animal])().visualize(decoded)[1]
    with serving.FrameBatcher(max_delay_ms=50.0) as fb:
        uri = serving.process_image(req, animal, batcher=fb, optimize=True)
        std = serving.process_image(req, animal, batcher=fb)
    assert uri == "data:image/jpeg;base64," + base64.b64encode(_cv2(view)).decode("utf-8")
    assert std == "data:image/jpeg;base64," + base64.b64encode(_cv2(view, optimize=False)).decode("utf-8")


def test_process_split_image_optimized():
    from animal_vision_b200 import animals as A
    from animal_vision_b200 import serving
    from test_gpu_split import host_route
    img = frames.natural(120, 176, 5)
    req = _cv2(img, optimize=False)
    decoded = cv2.imdecode(np.frombuffer(req, np.uint8), cv2.IMREAD_COLOR)
    view = A.Dog().visualize(decoded)[1]
    split = host_route(decoded[None], view[None], ("Original", "Dog"))[0]
    with serving.FrameBatcher(max_delay_ms=50.0) as fb:
        uri = serving.process_split_image(req, "dog", ("Original", "Dog"), batcher=fb, optimize=True)
    assert uri == "data:image/jpeg;base64," + base64.b64encode(_cv2(split)).decode("utf-8")


def test_standard_and_optimized_requests_share_a_batch():
    import torch
    from animal_vision_b200 import animals as A
    from animal_vision_b200 import serving
    from test_gpu_split import host_route
    imgs = [frames.natural(64, 96, s) for s in range(8)]
    views = A.Dog().visualize_batch(torch.from_numpy(np.stack(imgs)).cuda())[1].cpu().numpy()
    splits = host_route(np.stack(imgs), views, ("Original", "Transformed"))
    with serving.FrameBatcher(max_batch=16, max_delay_ms=200.0) as fb:
        kinds = ("jpeg", "opt", "split", "split_opt", "pix", "opt", "jpeg", "split_opt")
        futs = [fb.submit_jpeg(f, "dog") if k == "jpeg" else fb.submit_jpeg(f, "dog", optimize=True) if k == "opt"
                else fb.submit_split_jpeg(f, "dog", optimize=k == "split_opt") if k.startswith("split")
                else fb.submit(f, "dog") for k, f in zip(kinds, imgs)]
        res = [f.result(60) for f in futs]
    assert fb.batches == [("dog", 8)]
    for k, kind in enumerate(kinds):
        split = splits[k]
        want = {"jpeg": _cv2(views[k], optimize=False), "opt": _cv2(views[k]), "split": _cv2(split, optimize=False),
                "split_opt": _cv2(split), "pix": None}[kind]
        if kind == "pix":
            assert np.array_equal(res[k], views[k])
        else:
            assert res[k] == want, kind


def test_run_split_jpeg_optimized_writes_a_readable_avi(tmp_path):
    from test_gpu_mjpeg import Sink
    from test_gpu_split import host_route
    from test_gpu_split_pipeline import batch, pinned, views_of
    from test_mjpeg_host import read_opencv
    from animal_vision_b200 import animals as A
    from animal_vision_b200.pipeline import HostBatchPipeline
    from animal_vision_b200.renderers.mjpeg import MjpegAviWriter
    pipe = HostBatchPipeline(chunk_frames=2, depth=3)
    dog = A.Dog()
    a = batch(5, 135, 241)
    view = views_of(pipe, dog, a)
    ref = [np.ascontiguousarray(s[..., ::-1]) for s in host_route(a, view, ("Original", "Dog"))]
    f = pinned(a)
    sink, std = Sink(), Sink()
    pipe.run_split_jpeg([(dog, f)], labels=("Original", "Dog"), quality=90, optimize=True, out=sink)
    pipe.run_split_jpeg([(dog, f)], labels=("Original", "Dog"), quality=90, out=std)       # the standard mode on the same pipeline
    assert sink.jpegs == [_cv2(s, 90) for s in ref]
    assert std.jpegs == [_cv2(s, 90, optimize=False) for s in ref]
    assert np.array_equal(f.numpy(), a)
    path = tmp_path / "opt.avi"
    with MjpegAviWriter(str(path), 25, (241, 135)) as wr:
        pipe.run_split_jpeg([(dog, f)], labels=("Original", "Dog"), quality=90, optimize=True, out=wr)
    count, _, decoded = read_opencv(str(path))                 # OpenCV's own Motion-JPEG reader (libjpeg decode)
    assert count == 5 and len(decoded) == 5
    for frame, j in zip(decoded, sink.jpegs):
        assert np.array_equal(frame, cv2.imdecode(np.frombuffer(j, np.uint8), cv2.IMREAD_COLOR))
