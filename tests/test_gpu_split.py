"""K9 labelled split-compare compose (csrc/k9_split.cu, renderers/video.py split_compare_batch) and the server's split
requests: the gate is byte identity with the host route (slice copies + draw_split_labels, cv2.imencode), no tolerance."""
import base64

import cv2
import numpy as np
import pytest
import torch

import frames
from animal_vision_b200.renderers.video import draw_split_labels, split_compare_batch
from test_split_host import SWEEP, _host_split_jpeg, _inputs

pytestmark = pytest.mark.gpu


def host_route(a, b, labels, seam=True):
    """[N,H,W,3] uint8 host arrays -> the labelled split frames as the host draws them."""
    comp = split_compare_batch(torch.from_numpy(a), torch.from_numpy(b), draw_seam=seam).numpy()
    return np.stack([draw_split_labels(f.copy(), *labels) if labels is not None else f for f in comp])


def _pair(h, w):
    named = _inputs(h, w)
    a = np.stack([f for _, f in named])
    return a, a[:, ::-1, ::-1].copy()


@pytest.mark.parametrize("h,w,left,right", SWEEP, ids=[f"{h}x{w}-{i}" for i, (h, w, _, _) in enumerate(SWEEP)])
def test_labelled_split_equals_host_route(h, w, left, right):
    a, b = _pair(h, w)
    da, db = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
    for seam in (True, False):
        got = split_compare_batch(da, db, draw_seam=seam, labels=(left, right)).cpu().numpy()
        assert np.array_equal(got, host_route(a, b, (left, right), seam)), f"{h}x{w} seam={seam}"


@pytest.mark.parametrize("hw", [(1, 1), (2, 1), (17, 33), (64, 97), (1080, 1920), (2160, 3840)])
def test_unlabelled_split_is_the_slice_copy(hw):
    a, b = _pair(*hw)
    da, db = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
    for seam in (True, False):
        got = split_compare_batch(da, db, draw_seam=seam).cpu().numpy()
        assert np.array_equal(got, host_route(a, b, None, seam))


def test_mixed_batch_of_8_equals_one_at_a_time():
    h, w = 135, 241
    a = np.stack([frames.natural(h, w, s) for s in range(3)] + [frames.noise(h, w, 4), frames.impulses(h, w),
                                                               frames.bars(h, w), frames.constant(h, w, 255),
                                                               frames.checker(h, w)])
    b = np.ascontiguousarray(255 - a[::-1])
    da, db = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
    together = split_compare_batch(da, db, labels=("Original", "Dog")).cpu()
    for k in range(8):
        one = split_compare_batch(da[k:k + 1], db[k:k + 1], labels=("Original", "Dog")).cpu()
        assert torch.equal(together[k:k + 1], one)
    assert np.array_equal(together.numpy(), host_route(a, b, ("Original", "Dog")))


def test_side_stream_gives_the_same_bytes():
    a, b = _pair(240, 320)
    da, db = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
    ref = split_compare_batch(da, db, labels=("Original", "Transformed"))
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        got = split_compare_batch(da, db, labels=("Original", "Transformed"))
    torch.cuda.current_stream().wait_stream(s)
    assert torch.equal(got, ref)
    assert np.array_equal(got.cpu().numpy(), host_route(a, b, ("Original", "Transformed")))


@pytest.mark.parametrize("x,ox", [(31, 9), (32, 16), (4, 4)])          # byte-wise, 16-byte and 4-byte accesses
def test_strided_crops_in_and_out(x, ox):
    h, w = 123, 201
    big_a = torch.from_numpy(np.stack([frames.natural(300, 400, 1), frames.noise(300, 400, 2)])).cuda()
    big_b = torch.from_numpy(np.stack([frames.bars(300, 400), frames.checker(300, 400)])).cuda()
    canvas = torch.zeros((3, 310, 416, 3), dtype=torch.uint8, device="cuda")
    ca, cb = big_a[:, 17:17 + h, x:x + w], big_b[:, 22:22 + h, x:x + w]
    co = canvas[1:, 7:7 + h, ox:ox + w]
    assert not (ca.is_contiguous() or co.is_contiguous())
    split_compare_batch(ca, cb, out=co, labels=("Original", "Transformed"))
    ref = host_route(np.ascontiguousarray(ca.cpu().numpy()), np.ascontiguousarray(cb.cpu().numpy()),
                     ("Original", "Transformed"))
    assert np.array_equal(co.cpu().numpy(), ref)
    rest = canvas.clone()
    rest[1:, 7:7 + h, ox:ox + w] = 0
    assert int(rest.count_nonzero()) == 0                                           # nothing written outside the crop


def test_overlapping_out_and_host_labels_are_rejected():
    a = torch.zeros((2, 16, 16, 3), dtype=torch.uint8, device="cuda")
    b = torch.zeros_like(a)
    for out in (a, b[:, :8]):
        with pytest.raises((ValueError, AssertionError)):
            split_compare_batch(a, b, out=out)
    with pytest.raises(ValueError):
        split_compare_batch(a[:, :, 4:12], b[:, :, :8], out=a[:, :, :8])


def test_abi_rejects_bad_arguments():
    from animal_vision_b200 import _abi
    from animal_vision_b200.engine import get_engine
    lib = _abi.load()
    eng = get_engine()
    band, cls, lut = eng.split_stencil(32, 48, "Original", "Transformed")
    assert band > 0
    a = torch.zeros((2, 32, 48, 3), dtype=torch.uint8, device="cuda")
    b, o = torch.zeros_like(a), torch.zeros_like(a)
    st = torch.cuda.current_stream().cuda_stream
    fs, rs = 32 * 48 * 3, 48 * 3

    def call(l=a.data_ptr(), r=b.data_ptr(), out=o.data_ptr(), n=2, H=32, W=48, lrs=rs, rrs=rs, ors=rs, ofs=fs, band=band,
             c=cls.data_ptr(), t=lut.data_ptr(), lfs=fs):
        return lib.avb_split_compose_u8(l, r, out, n, H, W, lfs, lrs, fs, rrs, ofs, ors, 1, band, c, t, st)
    assert call() == 0
    assert call(band=0, c=None, t=None) == 0
    for kw in (dict(l=None), dict(r=None), dict(out=None), dict(n=0), dict(H=0), dict(W=0), dict(W=-3),
               dict(lrs=rs - 1), dict(rrs=rs - 1), dict(ors=rs - 1), dict(ofs=fs - 1), dict(lfs=-1),
               dict(band=-1), dict(band=33), dict(c=None), dict(t=None)):
        assert call(**kw) == -1, kw
        assert lib.avb_last_error()
    torch.cuda.synchronize()


SPECIES = ("dog", "cat", "honeybee", "reindeer")


@pytest.mark.parametrize("animal", SPECIES)
def test_process_split_image_through_the_device_batcher(animal):
    from animal_vision_b200 import animals as A
    from animal_vision_b200 import serving
    img = frames.natural(120, 176, 3)
    req = cv2.imencode(".jpg", img)[1].tobytes()
    decoded = cv2.imdecode(np.frombuffer(req, np.uint8), cv2.IMREAD_COLOR)
    view = getattr(A, serving.SERVER_KEYS[animal])().visualize(decoded)[1]
    with serving.FrameBatcher(max_delay_ms=50.0) as fb:
        uri = serving.process_split_image(req, animal, batcher=fb)
    assert uri == "data:image/jpeg;base64," + base64.b64encode(_host_split_jpeg(decoded, view)).decode("utf-8")


def test_pixel_jpeg_and_split_requests_share_one_launch():
    from animal_vision_b200 import animals as A
    from animal_vision_b200 import serving
    imgs = [frames.natural(64, 96, s) for s in range(8)]
    views = A.Dog().visualize_batch(torch.from_numpy(np.stack(imgs)).cuda())[1].cpu().numpy()
    kinds = ["pix", "jpeg", "split", "split2", "pix", "split", "jpeg", "split2"]
    with serving.FrameBatcher(max_batch=16, max_delay_ms=200.0) as fb:
        futs = []
        for k, f in zip(kinds, imgs):
            if k == "pix":
                futs.append(fb.submit(f, "dog"))
            elif k == "jpeg":
                futs.append(fb.submit_jpeg(f, "dog"))
            elif k == "split":
                futs.append(fb.submit_split_jpeg(f, "dog"))
            else:
                futs.append(fb.submit_split_jpeg(f, "dog", ("A", "Dog view"), draw_seam=False))
        res = [f.result(60) for f in futs]
    assert fb.batches == [("dog", 8)]
    for k, (kind, r) in enumerate(zip(kinds, res)):
        if kind == "pix":
            assert isinstance(r, np.ndarray) and np.array_equal(r, views[k])
        elif kind == "jpeg":
            assert r == cv2.imencode(".jpg", views[k])[1].tobytes()
        elif kind == "split":
            assert r == _host_split_jpeg(imgs[k], views[k])
        else:
            assert r == _host_split_jpeg(imgs[k], views[k], ("A", "Dog view"), seam=False)
