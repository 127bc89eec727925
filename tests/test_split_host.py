"""The label tables of the split-compare frame (tables.split_label_stencil) and the host route of split requests, on the
CPU: the tables applied in NumPy give the bytes draw_split_labels draws on the whole frame, no tolerance."""
import base64

import cv2
import numpy as np
import pytest
import torch

import frames
from animal_vision_b200 import serving, tables
from animal_vision_b200.renderers import video
from animal_vision_b200.renderers.video import draw_split_labels, split_compare_batch

# (H, W, left, right): small, overlapping long labels, odd sizes, 1080p, 4K, empty and non-ASCII text
SWEEP = [
    (1, 1, "Original", "Transformed"), (1, 2, "Original", "Transformed"), (2, 1, "Original", "Transformed"),
    (9, 13, "Original", "Transformed"), (17, 33, "Original", "Transformed"), (40, 60, "Original", "Dog view"),
    (120, 200, "Original", "Dog view"), (300, 161, "A", "Dog view"), (77, 90, "A very long left label", "Another long one"),
    (500, 700, "", "Überblick"), (1080, 1920, "Original", "HoneyBee"), (1079, 1921, "Original", "Transformed"),
    (2160, 3840, "Original", "Transformed"),
]


def apply_stencil(st, frame):
    out = frame.copy()
    if st.band_rows:
        out[:st.band_rows] = st.luts[st.classes.astype(np.intp)[:, :, None], frame[:st.band_rows]]
    return out


def _inputs(h, w):
    if h * w <= 400 * 400:
        named = list(frames.parity_set(h, w))
    else:
        named = [("natural", frames.natural(h, w))]
    return named + [("noise7", frames.noise(h, w, 7))]


@pytest.mark.parametrize("h,w,left,right", SWEEP, ids=[f"{h}x{w}-{i}" for i, (h, w, _, _) in enumerate(SWEEP)])
def test_stencil_equals_draw_split_labels(h, w, left, right):
    st = tables.split_label_stencil(h, w, left, right)
    assert 0 <= st.band_rows <= h and st.classes.shape == (st.band_rows, w) and st.classes.dtype == np.uint16
    assert st.luts.dtype == np.uint8 and st.luts.shape[1] == 256 and int(st.classes.max(initial=0)) < st.luts.shape[0]
    assert np.array_equal(st.luts[0], np.arange(256))
    named = _inputs(h, w)
    a = torch.from_numpy(np.stack([f for _, f in named]))
    b = torch.from_numpy(np.stack([f[::-1, ::-1].copy() for _, f in named]))
    for seam in (True, False):
        comp = split_compare_batch(a, b, draw_seam=seam).numpy()
        for k, (name, _) in enumerate(named):
            ref = draw_split_labels(comp[k].copy(), left, right)
            assert np.array_equal(apply_stencil(st, comp[k]), ref), f"{name} {h}x{w} seam={seam}"


def test_stencil_rows_below_the_band_are_untouched():
    st = tables.split_label_stencil(1080, 1920, "Original", "Transformed")
    assert 0 < st.band_rows < 120
    f = frames.noise(1080, 1920, 3)
    assert np.array_equal(draw_split_labels(f.copy())[st.band_rows:], f[st.band_rows:])


def test_stencil_is_cached_per_key_and_read_only():
    a = tables.split_label_stencil(64, 96, "Original", "Transformed")
    assert tables.split_label_stencil(64, 96, "Original", "Transformed") is a
    assert tables.split_label_stencil(64, 96, "Original", "Dog") is not a
    assert tables.split_label_stencil(65, 96, "Original", "Transformed") is not a
    with pytest.raises(ValueError):
        a.luts[0, 0] = 1


def test_stencil_rejects_a_label_colour_that_is_not_grey(monkeypatch):
    monkeypatch.setattr(video, "LABEL_FONT_COLOURS", ((0, 0, 0), (255, 255, 0)))
    with pytest.raises(ValueError, match="channels"):
        tables.split_label_stencil(71, 97, "Not", "grey")


def test_stencil_rejects_too_many_classes(monkeypatch):
    monkeypatch.setattr(tables, "SPLIT_CLASS_INDEX", np.uint8)                      # 1 249 tables at 1080p
    with pytest.raises(ValueError, match="do not fit"):
        tables.split_label_stencil(1080, 1921, "Too", "many")


def test_labels_on_host_tensors_and_overlapping_out_are_rejected():
    a = torch.from_numpy(frames.noise(8, 8, 0)[None].copy())
    b = torch.from_numpy(frames.noise(8, 8, 1)[None].copy())
    with pytest.raises(ValueError):
        split_compare_batch(a, b, labels=("Original", "Transformed"))
    with pytest.raises(ValueError):
        split_compare_batch(a, b, out=a)
    big = torch.zeros((1, 8, 16, 3), dtype=torch.uint8)
    with pytest.raises(ValueError):
        split_compare_batch(big[:, :, :8], b, out=big[:, :, 4:12])
    out = torch.empty((2, 8, 8, 3), dtype=torch.uint8)
    assert split_compare_batch(a, b, out=out[1:]).data_ptr() == out[1:].data_ptr()


def _host_split_jpeg(frame, view, labels=("Original", "Transformed"), seam=True):
    comp = split_compare_batch(torch.from_numpy(frame[None]), torch.from_numpy(view[None]), draw_seam=seam)[0].numpy()
    return cv2.imencode(".jpg", draw_split_labels(comp, *labels))[1].tobytes()


def test_process_split_image_with_a_numpy_runner():
    img = frames.natural(48, 64)
    req = cv2.imencode(".jpg", img)[1].tobytes()
    dec = cv2.imdecode(np.frombuffer(req, np.uint8), cv2.IMREAD_COLOR)
    with serving.FrameBatcher(lambda key, batch: 255 - batch, max_delay_ms=1.0) as fb:
        uri = serving.process_split_image(req, "dog", batcher=fb)
        uri2 = serving.process_split_image(req, "dog", labels=("A", "Dog view"), batcher=fb)
        human = serving.process_split_image(req, "human", batcher=fb)
    assert uri == "data:image/jpeg;base64," + base64.b64encode(_host_split_jpeg(dec, 255 - dec)).decode()
    assert uri2 == "data:image/jpeg;base64," + base64.b64encode(_host_split_jpeg(dec, 255 - dec, ("A", "Dog view"))).decode()
    assert human == "data:image/jpeg;base64," + base64.b64encode(_host_split_jpeg(dec, dec)).decode()


def test_split_requests_share_the_batch_on_the_host_route():
    imgs = [frames.natural(40, 56, s) for s in range(5)]
    with serving.FrameBatcher(lambda key, batch: 255 - batch, max_batch=16, max_delay_ms=200.0) as fb:
        futs = [fb.submit(imgs[0], "dog"), fb.submit_jpeg(imgs[1], "dog"),
                fb.submit_split_jpeg(imgs[2], "dog"), fb.submit_split_jpeg(imgs[3], "dog", ("L", "R"), draw_seam=False),
                fb.submit_split_jpeg(imgs[4], "dog")]
        res = [f.result(10) for f in futs]
        with pytest.raises(TypeError):
            fb.submit_split_jpeg(imgs[0], "dog", labels="Original").result(1)
    assert fb.batches == [("dog", 5)]
    assert np.array_equal(res[0], 255 - imgs[0])
    assert res[1] == cv2.imencode(".jpg", 255 - imgs[1])[1].tobytes()
    assert res[2] == _host_split_jpeg(imgs[2], 255 - imgs[2])
    assert res[3] == _host_split_jpeg(imgs[3], 255 - imgs[3], ("L", "R"), seam=False)
    assert res[4] == _host_split_jpeg(imgs[4], 255 - imgs[4])
