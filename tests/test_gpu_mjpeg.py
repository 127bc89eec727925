"""Motion-JPEG video from the device: K8's RGB entry point (encode_jpeg(rgb=True)), the AVI record pack (K11,
avb_mjpeg_pack_u8) and HostBatchPipeline.run_split_jpeg into MjpegAviWriter.  The gate is byte identity with
cv2.imencode of the host route's split frames, no tolerance."""
import cv2
import numpy as np
import pytest
import torch

import frames
from animal_vision_b200 import animals as A
from animal_vision_b200._abi import AvbError
from animal_vision_b200.engine import get_engine
from animal_vision_b200.jpeg import encode_jpeg
from animal_vision_b200.pipeline import HostBatchPipeline
from animal_vision_b200.renderers.mjpeg import MjpegAviWriter
from test_gpu_split import host_route
from test_gpu_split_pipeline import Invert, InvertPair, batch, pinned, views_of
from test_mjpeg_host import pack_records

pytestmark = pytest.mark.gpu

DEFAULT = ("Original", "Transformed")


def _cv2(img, q):
    ok, enc = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_QUALITY, q])
    assert ok
    return enc.tobytes()


@pytest.mark.parametrize("q", [1, 50, 95, 100])
@pytest.mark.parametrize("hw", [(1, 1), (17, 33), (1080, 1920), (2160, 3840)])
def test_rgb_encode_equals_cv2_of_the_swapped_frame(hw, q):
    imgs = np.stack([frames.natural(*hw, 3), frames.noise(*hw, 4)])
    dev = torch.from_numpy(imgs).cuda()
    got = encode_jpeg(dev, q, rgb=True)
    for img, g in zip(imgs, got):
        assert g == _cv2(np.ascontiguousarray(img[..., ::-1]), q)
    assert encode_jpeg(dev, q) == [_cv2(img, q) for img in imgs]            # the default order is still BGR


def test_rgb_encode_of_a_strided_crop():
    big = np.stack([frames.natural(300, 400, 1), frames.noise(300, 400, 2)])
    crop = torch.from_numpy(big).cuda()[:, 17:17 + 123, 31:31 + 201]
    assert not crop.is_contiguous()
    for k, g in enumerate(encode_jpeg(crop, 85, rgb=True)):
        assert g == _cv2(np.ascontiguousarray(big[k, 17:140, 31:232, ::-1]), 85)


def pack_on_device(jpegs, slot):
    """K11 over `jpegs` placed in slots of `slot` bytes (garbage after each file): the packed bytes, the offsets and
    the untouched tail of the output buffer."""
    eng = get_engine()
    n = len(jpegs)
    rng = np.random.default_rng(n)
    host = rng.integers(0, 256, n * slot, dtype=np.uint8)
    for f, j in enumerate(jpegs):
        host[f * slot:f * slot + len(j)] = np.frombuffer(j, np.uint8)
    slots = torch.from_numpy(host).cuda()
    lengths = torch.tensor([len(j) for j in jpegs], dtype=torch.int64, device="cuda")
    cap = n * (8 + ((slot + 3) & ~3))
    out = torch.full((cap + 64,), 0xAB, dtype=torch.uint8, device="cuda")
    offsets = torch.empty(n + 1, dtype=torch.int64, device="cuda")
    rc = eng.lib.avb_mjpeg_pack_u8(slots.data_ptr(), slot, lengths.data_ptr(), n, out.data_ptr(), offsets.data_ptr(),
                                   eng.stream_ptr())
    assert rc == 0, eng.lib.avb_last_error()
    offs = offsets.cpu().numpy()
    return out.cpu().numpy(), offs


@pytest.mark.parametrize("slot", [4099, 4102, 4104])          # slot starts at every byte alignment
def test_pack_equals_numpy_records(slot):
    rng = np.random.default_rng(slot)
    for n in range(1, 18):
        lens = rng.integers(0, slot + 1, n)
        lens[: min(n, 4)] = [slot, 1, 0, slot - 1][: min(n, 4)]
        jpegs = [rng.integers(0, 256, int(k), dtype=np.uint8).tobytes() for k in lens]
        got, offs = pack_on_device(jpegs, slot)
        ref, ref_offs = pack_records(jpegs)
        assert np.array_equal(offs, ref_offs), n
        assert np.array_equal(got[:ref.size], ref), n
        assert (got[ref.size:] == 0xAB).all(), n


def test_pack_large_frames():
    """4K-sized files: the grid-stride copy across many CTAs per frame."""
    rng = np.random.default_rng(1)
    jpegs = [rng.integers(0, 256, k, dtype=np.uint8).tobytes() for k in (2_661_237, 2_500_000, 3_000_001)]
    got, offs = pack_on_device(jpegs, 3_000_003)
    ref, ref_offs = pack_records(jpegs)
    assert np.array_equal(offs, ref_offs) and np.array_equal(got[:ref.size], ref)


def test_pack_refuses_bad_arguments():
    eng = get_engine()
    lib = eng.lib
    slots = torch.zeros(64, dtype=torch.uint8, device="cuda")
    lengths = torch.tensor([5, 6], dtype=torch.int64, device="cuda")
    out = torch.zeros(128, dtype=torch.uint8, device="cuda")
    offs = torch.zeros(3, dtype=torch.int64, device="cuda")
    st = eng.stream_ptr()

    def call(s=slots.data_ptr(), stride=32, l=lengths.data_ptr(), n=2, o=out.data_ptr(), of=offs.data_ptr()):
        return lib.avb_mjpeg_pack_u8(s, stride, l, n, o, of, st)
    assert call() == 0
    for kw in (dict(s=None), dict(l=None), dict(o=None), dict(of=None), dict(n=0), dict(stride=0),
               dict(o=out.data_ptr() + 4), dict(s=slots.data_ptr() + 1)):
        assert call(**kw) == -1, kw
        assert lib.avb_last_error()
    torch.cuda.synchronize()


class Sink:
    """write_records target that keeps every frame's JPEG and checks the records."""

    def __init__(self):
        self.jpegs, self.record_bytes = [], 0

    def write_records(self, records, jpeg_lengths):
        buf = bytes(records)
        self.record_bytes += len(buf)
        off = 0
        for n in jpeg_lengths:
            size = (n + 3) & ~3
            assert buf[off:off + 4] == b"00dc" and int.from_bytes(buf[off + 4:off + 8], "little") == size
            assert not any(buf[off + 8 + n:off + 8 + size])
            self.jpegs.append(buf[off + 8:off + 8 + n])
            off += 8 + size
        assert off == len(buf)


def check_jpegs(pipe, species, a, view, labels, seam, q=95):
    f = pinned(a)
    sink = Sink()
    h2d, d2h = pipe.run_split_jpeg([(species, f)], labels=labels, draw_seam=seam, quality=q, out=sink)
    assert np.array_equal(f.numpy(), a)                                        # the input frames are unchanged
    ref = host_route(a, view, labels, seam)
    assert sink.jpegs == [_cv2(np.ascontiguousarray(s[..., ::-1]), q) for s in ref], (type(species).__name__, labels)
    chunks = -(-a.shape[0] // pipe.chunk)
    assert h2d == a.size and d2h == sink.record_bytes + 8 * (2 * a.shape[0] + chunks)
    return sink


LABEL_CASES = [(DEFAULT, True), (("Left side", "Right view"), False), (None, True), (None, False)]


@pytest.mark.parametrize("hw", [(20, 30), (1, 1), (64, 97)])
@pytest.mark.parametrize("species", [Invert(), InvertPair()], ids=["one_output", "two_outputs"])
def test_stand_ins_equal_the_host_route(species, hw):
    pipe = HostBatchPipeline(chunk_frames=3, depth=2)
    a = batch(7, *hw)
    for labels, seam in LABEL_CASES:
        check_jpegs(pipe, species, a, 255 - a, labels, seam, q=90)


@pytest.mark.parametrize("name", ["Dog", "Cat", "HoneyBee"])
def test_species_at_1080p_equal_the_host_route(name):
    """N = 5 in chunks of 2: slots are reused and the last chunk is partial."""
    sp = getattr(A, name)()
    pipe = HostBatchPipeline(chunk_frames=2, depth=3)
    a = batch(5, 1080, 1920)
    view = views_of(pipe, sp, a)
    for labels, seam in LABEL_CASES[:3]:
        check_jpegs(pipe, sp, a, view, labels, seam)


def test_two_shapes_in_one_call_written_to_a_file(tmp_path):
    """The file run_split_jpeg writes equals, byte for byte, the one write_jpeg writes from the host route's JPEGs."""
    pipe = HostBatchPipeline(chunk_frames=3, depth=2)
    dog, cat = A.Dog(), A.Cat()
    a1, a2 = batch(7, 135, 241), batch(4, 135, 241, seed=20)
    v1, v2 = views_of(pipe, dog, a1), views_of(pipe, cat, a2)
    f1, f2 = pinned(a1), pinned(a2)
    dev = tmp_path / "device.avi"
    with MjpegAviWriter(str(dev), 30, (241, 135)) as wr:
        pipe.run_split_jpeg([(dog, f1), (cat, f2)], labels=("Original", "Dog"), quality=80, out=wr)
    host = tmp_path / "host.avi"
    with MjpegAviWriter(str(host), 30, (241, 135)) as wr:
        for a, v in ((a1, v1), (a2, v2)):
            for s in host_route(a, v, ("Original", "Dog")):
                wr.write_jpeg(_cv2(np.ascontiguousarray(s[..., ::-1]), 80))
    assert dev.read_bytes() == host.read_bytes()
    assert np.array_equal(f1.numpy(), a1) and np.array_equal(f2.numpy(), a2)
    sink = Sink()                                                  # two shapes: the slot sets of both in one call
    a3 = batch(5, 64, 96, seed=30)
    v3 = views_of(pipe, dog, a3)
    pipe.run_split_jpeg([(dog, pinned(a1)), (dog, pinned(a3))], out=sink)
    ref = list(host_route(a1, v1, DEFAULT)) + list(host_route(a3, v3, DEFAULT))
    assert sink.jpegs == [_cv2(np.ascontiguousarray(s[..., ::-1]), 95) for s in ref]


def test_bad_arguments_raise_before_anything_is_enqueued():
    pipe = HostBatchPipeline(chunk_frames=3)
    dog = A.Dog()
    a = batch(4, 32, 48)
    good = pinned(a)
    sink = Sink()
    for bad in (torch.from_numpy(a.copy()), torch.from_numpy(a).cuda()):
        with pytest.raises(ValueError, match="pinned, contiguous uint8"):
            pipe.run_split_jpeg([(dog, good), (dog, bad)], out=sink)
    with pytest.raises(ValueError, match="share host frames"):
        pipe.run_split_jpeg([(dog, good[:3]), (dog, good[2:])], out=sink)
    for q in (0, 101, 9.5, True):
        with pytest.raises(AvbError, match="quality"):
            pipe.run_split_jpeg([(dog, good)], quality=q, out=sink)
    for labels in ("Original", ("Only one",), ("A", 3)):
        with pytest.raises(TypeError, match="labels"):
            pipe.run_split_jpeg([(dog, good)], labels=labels, out=sink)
    with pytest.raises(TypeError, match="write_records"):
        pipe.run_split_jpeg([(dog, good)], out=object())
    torch.cuda.synchronize()
    assert sink.jpegs == [] and np.array_equal(good.numpy(), a)


class Refuses:
    N_OUTPUTS = 1

    def visualize_batch(self, frames, out):
        raise RuntimeError("refused")


def test_a_failing_job_drains_the_streams():
    pipe = HostBatchPipeline(chunk_frames=2, depth=2)
    a = batch(5, 64, 96)
    sink = Sink()
    with pytest.raises(RuntimeError, match="refused"):
        pipe.run_split_jpeg([(Invert(), pinned(a)), (Refuses(), pinned(a[:2].copy()))], out=sink)
    ref = [_cv2(np.ascontiguousarray(s[..., ::-1]), 95) for s in host_route(a, 255 - a, DEFAULT)]
    assert sink.jpegs == ref[:len(sink.jpegs)]                        # what was handed over is in order and whole
    check_jpegs(pipe, Invert(), a, 255 - a, DEFAULT, True)              # the pipeline stays usable
