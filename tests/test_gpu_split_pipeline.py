"""HostBatchPipeline.run_split and the split-frame fetch (avb_split_fetch_u8, Engine.split_fetch) on the device: the
frames come back as the bytes of the host route built from run()'s views (slice copies + draw_split_labels), no
tolerance; the fetch writes exactly its byte set; bad arguments are refused before anything is enqueued."""
import numpy as np
import pytest
import torch

import frames
from animal_vision_b200 import animals as A
from animal_vision_b200 import tables
from animal_vision_b200._abi import AvbError
from animal_vision_b200.engine import get_engine, split_fetch_bytes
from animal_vision_b200.pipeline import HostBatchPipeline
from test_gpu_split import host_route
from test_split_fetch_host import fetch_mask

pytestmark = pytest.mark.gpu

DEFAULT = ("Original", "Transformed")
LABEL_CASES = [(DEFAULT, True), (("Left side", "Right view"), False), (None, True), (None, False)]


class Invert:
    """A one-output stand-in species (view = 255 - frame) for frames smaller than the species kernels are meant for."""
    N_OUTPUTS = 1

    def visualize_batch(self, frames, out):
        torch.bitwise_not(frames, out=out)


class InvertPair:
    """The two-output form: a baseline, then the view."""
    N_OUTPUTS = 2

    def visualize_batch(self, frames, out):
        out[0].fill_(7)
        torch.bitwise_not(frames, out=out[1])


def batch(n, h, w, seed=0):
    return np.stack([frames.natural(h, w, seed + k) if k % 2 else frames.noise(h, w, seed + k) for k in range(n)])


def pinned(a):
    return torch.from_numpy(a).pin_memory()


def views_of(pipe, species, a):
    """The species view of every frame of `a`, through run() on the same pipeline."""
    src = pinned(a)
    outs = pipe.pinned_like(src, pipe.n_outputs(species))
    pipe.run([(species, src, outs)])
    return outs[-1].numpy().copy()


def check_split(pipe, species, a, view, labels, seam):
    f = pinned(a)
    pipe.run_split([(species, f)], labels=labels, draw_seam=seam)
    assert np.array_equal(f.numpy(), host_route(a, view, labels, seam)), (type(species).__name__, a.shape, labels, seam)


@pytest.mark.parametrize("depth", [2, 3])
@pytest.mark.parametrize("hw", [(1080, 1920), (135, 241)], ids=["1080x1920", "135x241"])
@pytest.mark.parametrize("name", ["Dog", "Cat", "HoneyBee", "Goldfish"])
def test_run_split_equals_the_host_route(name, hw, depth):
    """N = 7 in chunks of 3: slots are reused and the last chunk is partial."""
    sp = getattr(A, name)()
    pipe = HostBatchPipeline(chunk_frames=3, depth=depth)
    a = batch(7, *hw)
    view = views_of(pipe, sp, a)
    for labels, seam in LABEL_CASES:
        check_split(pipe, sp, a, view, labels, seam)


@pytest.mark.parametrize("hw", [(5, 1), (20, 30), (1, 1)])
@pytest.mark.parametrize("species", [Invert(), InvertPair()], ids=["one_output", "two_outputs"])
def test_tiny_frames(species, hw):
    """W // 2 == 0 (the right piece is the whole row) and a label band covering every row."""
    h, w = hw
    assert tables.split_label_stencil(h, w, *DEFAULT).band_rows == h
    pipe = HostBatchPipeline(chunk_frames=3, depth=2)
    a = batch(7, h, w)
    view = views_of(pipe, species, a)
    assert np.array_equal(view, 255 - a)
    for labels, seam in LABEL_CASES:
        check_split(pipe, species, a, view, labels, seam)


def test_fetch_follows_the_upload_of_its_frames():
    """The fetch writes the very host frames its chunk uploads; one 4K frame per chunk puts each fetch as early in the
    stream order as the events allow, so a fetch that did not wait for its upload would corrupt the view's input."""
    sp = A.Dog()
    pipe = HostBatchPipeline(chunk_frames=1, depth=3)
    a = batch(6, 2160, 3840, seed=40)
    view = views_of(pipe, sp, a)
    check_split(pipe, sp, a, view, DEFAULT, True)


def test_two_shapes_and_species_in_one_call_and_run_between_calls():
    pipe = HostBatchPipeline(chunk_frames=3, depth=2)
    dog, cat = A.Dog(), A.Cat()
    a1, a2 = batch(7, 135, 241), batch(5, 64, 96, seed=20)
    v1, v2 = views_of(pipe, dog, a1), views_of(pipe, cat, a2)
    f1, f2 = pinned(a1), pinned(a2)
    pipe.run_split([(dog, f1), (cat, f2)], labels=("Original", "Dog"))
    assert np.array_equal(f1.numpy(), host_route(a1, v1, ("Original", "Dog")))
    assert np.array_equal(f2.numpy(), host_route(a2, v2, ("Original", "Dog")))
    assert np.array_equal(views_of(pipe, cat, a2), v2)          # run() on the slots run_split used for Cat at 64x96
    check_split(pipe, cat, a2, v2, DEFAULT, True)


def test_returned_byte_counts():
    h, w = 1080, 1920
    band = tables.split_label_stencil(h, w, *DEFAULT).band_rows
    pipe = HostBatchPipeline(chunk_frames=3)
    cat, dog = A.Cat(), A.Dog()
    a = batch(7, h, w)
    _, run_d2h = pipe.run([(cat, pinned(a), pipe.pinned_like(pinned(a), 2))])
    assert run_d2h == 2 * 7 * h * w * 3
    for labels, b in ((DEFAULT, band), (None, 0)):
        h2d, d2h = pipe.run_split([(cat, pinned(a)), (dog, pinned(a[:4]))], labels=labels)
        assert h2d == 11 * h * w * 3
        assert d2h == 11 * (b * 3 * w + (h - b) * (3 * w - 3 * (w // 2))) == split_fetch_bytes(11, h, w, b)
        _, cat_d2h = pipe.run_split([(cat, pinned(a))], labels=labels)
        # a quarter of run()'s two Cat frames, plus the left half of the label band
        assert cat_d2h == run_d2h // 4 + 7 * b * 3 * (w // 2)
        assert cat_d2h < 0.27 * run_d2h


def _host_frames(n, h, w, layout, pin):
    """(flat buffer, [n,h,w,3] view, frame stride, row stride) with the layout's byte strides."""
    rs = 3 * w + (15 if layout == "wide_rows" else 0)
    fs = h * rs + (16 if layout == "per_frame" else 0)
    flat = torch.zeros(n * fs, dtype=torch.uint8)
    if pin:
        flat = flat.pin_memory()
    return flat, flat.as_strided((n, h, w, 3), (fs, rs, 3, 1)), fs, rs


@pytest.mark.parametrize("n", [1, 3])
@pytest.mark.parametrize("layout", ["packed", "wide_rows", "per_frame"])
@pytest.mark.parametrize("h,w,band", [(37, 53, 11), (37, 53, 0), (37, 53, 37), (6, 1, 2), (64, 96, 41)])
def test_fetch_writes_exactly_its_byte_set(h, w, band, layout, n):
    """packed and wide_rows take one 3D copy per piece, per_frame (frame stride not a whole number of rows, on both
    sides) two 2D copies per frame."""
    eng = get_engine()
    sfs = h * 3 * w + (16 if layout == "per_frame" else 0)
    src = torch.full((n * sfs,), 0xAB, dtype=torch.uint8, device="cuda").as_strided((n, h, w, 3), (sfs, 3 * w, 3, 1))
    flat, dst, fs, rs = _host_frames(n, h, w, layout, pin=True)
    nbytes = eng.split_fetch(src, dst, band)
    torch.cuda.synchronize()
    want = torch.zeros_like(flat).numpy().astype(bool)
    y = np.arange(h)[:, None]
    x = np.arange(3 * w)[None, :]
    for f in range(n):
        want[f * fs + y * rs + x] = fetch_mask(h, w, band)
    got = flat.numpy()
    assert np.array_equal(got != 0, want)
    assert (got[want] == 0xAB).all()
    assert nbytes == int(want.sum()) == split_fetch_bytes(n, h, w, band)


def test_fetch_refuses_pageable_destination_and_host_source():
    eng = get_engine()
    lib = eng.lib
    n, h, w = 2, 16, 24
    src = torch.full((n, h, w, 3), 0xAB, dtype=torch.uint8, device="cuda")
    pageable = torch.zeros((n, h, w, 3), dtype=torch.uint8)
    with pytest.raises(AvbError, match="page-locked"):
        eng.split_fetch(src, pageable, 4)
    fs, rs = h * w * 3, w * 3
    st = torch.cuda.current_stream().cuda_stream
    assert lib.avb_split_fetch_u8(src.data_ptr(), pageable.data_ptr(), n, h, w, fs, rs, fs, rs, 4, st) == -1
    assert b"page-locked" in lib.avb_last_error()
    host_src = torch.full((n, h, w, 3), 0xAB, dtype=torch.uint8).pin_memory()
    dst = torch.zeros((n, h, w, 3), dtype=torch.uint8).pin_memory()
    assert lib.avb_split_fetch_u8(host_src.data_ptr(), dst.data_ptr(), n, h, w, fs, rs, fs, rs, 4, st) == -1
    assert b"device memory" in lib.avb_last_error()
    torch.cuda.synchronize()
    assert not pageable.any() and not dst.any()
    assert eng.split_fetch(src, dst, 4) == split_fetch_bytes(n, h, w, 4)   # the library stays usable
    torch.cuda.synchronize()


def test_run_split_refuses_bad_jobs_before_enqueueing_anything():
    pipe = HostBatchPipeline(chunk_frames=3)
    dog = A.Dog()
    a = batch(4, 32, 48)
    good = pinned(a)
    wide = pinned(batch(4, 32, 96, seed=9))
    bad_frames = [torch.from_numpy(a.copy()),                          # pageable
                  wide[:, :, :48],                                      # pinned, not contiguous
                  torch.from_numpy(a).cuda(),                           # on the device
                  pinned(a.astype(np.float32)),                         # not uint8
                  pinned(a[..., :2].copy())]                            # not 3 channels
    before = [x.cpu().clone() for x in bad_frames]
    for bad in bad_frames:
        with pytest.raises(ValueError, match="pinned, contiguous uint8"):
            pipe.run_split([(dog, good), (dog, bad)])
    for labels in ("Original", ("Only one",), ("A", 3), ("a", "b", "c")):
        with pytest.raises(TypeError, match="labels"):
            pipe.run_split([(dog, good)], labels=labels)
    torch.cuda.synchronize()
    assert np.array_equal(good.numpy(), a)
    for x, b in zip(bad_frames, before):
        assert torch.equal(x.cpu(), b)


def test_run_split_refuses_jobs_that_share_host_frames():
    pipe = HostBatchPipeline(chunk_frames=3)
    dog = A.Dog()
    a = batch(6, 32, 48)
    f = pinned(a)
    for jobs in ([(dog, f), (dog, f)], [(dog, f[:4]), (dog, f[3:])]):
        with pytest.raises(ValueError, match="share host frames"):
            pipe.run_split(jobs)
    torch.cuda.synchronize()
    assert np.array_equal(f.numpy(), a)
    pipe.run_split([(dog, f[:3]), (dog, f[3:])])                     # adjacent, disjoint views are fine
    assert np.array_equal(f.numpy(), host_route(a, views_of(pipe, dog, a), DEFAULT))


class Refuses:
    N_OUTPUTS = 1

    def visualize_batch(self, frames, out):
        raise RuntimeError("refused")


def test_a_failing_job_leaves_no_copy_in_flight():
    """run_split waits for what it enqueued before it raises: the earlier job's frames are finished split frames."""
    pipe = HostBatchPipeline(chunk_frames=2)
    a, c = batch(5, 64, 96), batch(2, 64, 96, seed=30)
    f, g = pinned(a), pinned(c)
    with pytest.raises(RuntimeError, match="refused"):
        pipe.run_split([(Invert(), f), (Refuses(), g)])
    assert np.array_equal(f.numpy(), host_route(a, 255 - a, DEFAULT))
    assert np.array_equal(g.numpy(), c)


def test_run_leaves_no_copy_in_flight_when_a_job_fails():
    """run waits for what it enqueued before it raises: the earlier job's views are already in its outputs (1080p
    frames, so a copy still in flight would be seen), and the pipeline stays usable."""
    pipe = HostBatchPipeline(chunk_frames=2)
    a, c = batch(5, 1080, 1920), batch(2, 1080, 1920, seed=30)
    f, g = pinned(a), pinned(c)
    outs_f, outs_g = pipe.pinned_like(f, 1), pipe.pinned_like(g, 1)
    with pytest.raises(RuntimeError, match="refused"):
        pipe.run([(Invert(), f, outs_f), (Refuses(), g, outs_g)])
    assert np.array_equal(outs_f[0].numpy(), 255 - a)
    assert np.array_equal(views_of(pipe, Invert(), c), 255 - c)
