"""Motion-JPEG AVI writer (animal_vision_b200/renderers/mjpeg.py), host only: the container OpenCV's own MJPEG writer
produces, byte for byte up to the 'movi' list, sizes and index consistent with the chunks, read back by OpenCV's MJPEG
reader and by FFmpeg; the record layout of the pack kernel (K11) restated in NumPy; the size limit."""
import struct

import cv2
import numpy as np
import pytest

import frames
from animal_vision_b200.renderers import mjpeg
from animal_vision_b200.renderers.mjpeg import MjpegAviWriter, jpeg_record


def pack_records(jpegs):
    """NumPy statement of avb_mjpeg_pack_u8: the records of `jpegs` back to back, and the n + 1 record offsets."""
    sizes = np.array([(len(j) + 3) & ~3 for j in jpegs], np.int64)
    offsets = np.concatenate([[0], np.cumsum(8 + sizes)]).astype(np.int64)
    out = np.zeros(int(offsets[-1]), np.uint8)
    for j, o, s in zip(jpegs, offsets, sizes):
        out[o:o + 4] = np.frombuffer(b"00dc", np.uint8)
        out[o + 4:o + 8] = np.array([s], "<u4").view(np.uint8)
        out[o + 8:o + 8 + len(j)] = np.frombuffer(j, np.uint8)
    return out, offsets


def chunks(buf, start, end):
    """[(offset, fourcc, size)] of the RIFF chunks in buf[start:end]."""
    out = []
    while start + 8 <= end:
        cc, size = buf[start:start + 4], struct.unpack_from("<I", buf, start + 4)[0]
        out.append((start, cc, size))
        start += 8 + size + (size & 1)
    return out


def _frames(n, h, w):
    return [frames.natural(h, w, s) if s % 2 else frames.noise(h, w, s) for s in range(n)]


def _jpegs(imgs, q=95):
    return [cv2.imencode(".jpg", f, [cv2.IMWRITE_JPEG_QUALITY, q])[1].tobytes() for f in imgs]


def check_layout(buf, jpegs, fps, w, h):
    """RIFF and 'movi' sizes, the frame counts and idx1 agree with the '00dc' chunks, which hold `jpegs`."""
    assert buf[:4] == b"RIFF" and struct.unpack_from("<I", buf, 4)[0] == len(buf) - 8 and buf[8:12] == b"AVI "
    top = chunks(buf, 12, len(buf))
    assert [c[1] for c in top] == [b"LIST", b"JUNK", b"LIST", b"idx1"]
    (movi_at, _, movi_size), (idx_at, _, idx_size) = top[2], top[3]
    assert movi_at == 4096 and buf[movi_at + 8:movi_at + 12] == b"movi" and idx_at == movi_at + 8 + movi_size
    recs = chunks(buf, movi_at + 12, movi_at + 8 + movi_size)
    assert len(recs) == len(jpegs) and idx_size == 16 * len(jpegs)
    for k, ((at, cc, size), j) in enumerate(zip(recs, jpegs)):
        assert cc == b"00dc" and size == (len(j) + 3) & ~3
        assert buf[at + 8:at + 8 + len(j)] == j and not any(buf[at + 8 + len(j):at + 8 + size])
        assert struct.unpack_from("<4s3I", buf, idx_at + 8 + 16 * k) == (b"00dc", 0x10, at - movi_at - 8, size)
    for at in (48, 140, 232):                                   # avih, strh, dmlh frame counts
        assert struct.unpack_from("<I", buf, at)[0] == len(jpegs)
    assert struct.unpack_from("<2I", buf, 64) == (w, h) and struct.unpack_from("<I", buf, 132)[0] == round(fps)


SIZES = [(1, 1), (17, 33), (64, 96), (2160, 3840)]


@pytest.mark.parametrize("fps", [25, 29.97, 60])
@pytest.mark.parametrize("n", [0, 1, 5])
@pytest.mark.parametrize("hw", SIZES, ids=[f"{h}x{w}" for h, w in SIZES])
def test_container_matches_opencv_writer(tmp_path, hw, n, fps):
    h, w = hw
    imgs = _frames(n, h, w) if h * w < 10 ** 5 else [frames.constant(h, w, 40 * k) for k in range(n)]
    vw = cv2.VideoWriter(str(tmp_path / "cv.avi"), cv2.CAP_OPENCV_MJPEG, cv2.VideoWriter_fourcc(*"MJPG"), fps, (w, h))
    assert vw.isOpened()
    for f in imgs:
        vw.write(f)
    vw.release()
    jpegs = _jpegs(imgs)
    with MjpegAviWriter(str(tmp_path / "me.avi"), fps, (w, h)) as wr:
        for j in jpegs:
            wr.write_jpeg(j)
    ref, got = (tmp_path / "cv.avi").read_bytes(), (tmp_path / "me.avi").read_bytes()
    assert got[12:4096] == ref[12:4096]                         # hdrl and JUNK
    check_layout(got, jpegs, fps, w, h)
    if n:
        check_layout(ref, [ref[at + 8:at + 8 + s] for at, _, s in chunks(ref, 4108, len(ref) - 8 - 16 * n)], fps, w, h)


def read_opencv(path):
    cap = cv2.VideoCapture(path, cv2.CAP_OPENCV_MJPEG)
    assert cap.isOpened()
    count, fps, out = cap.get(cv2.CAP_PROP_FRAME_COUNT), cap.get(cv2.CAP_PROP_FPS), []
    while True:
        ok, f = cap.read()
        if not ok:
            return count, fps, out
        out.append(f)


@pytest.mark.parametrize("fps", [25, 29.97])
@pytest.mark.parametrize("hw", [(17, 33), (64, 96)])
def test_opencv_mjpeg_reader_plays_it(tmp_path, hw, fps):
    jpegs = _jpegs(_frames(5, *hw), 80)
    path = str(tmp_path / "v.avi")
    with MjpegAviWriter(path, fps, hw[::-1]) as wr:
        for j in jpegs:
            wr.write_jpeg(j)
    count, got_fps, decoded = read_opencv(path)
    assert count == 5 and got_fps == round(fps) and len(decoded) == 5
    for f, j in zip(decoded, jpegs):
        assert np.array_equal(f, cv2.imdecode(np.frombuffer(j, np.uint8), cv2.IMREAD_COLOR))


def test_ffmpeg_returns_the_jpegs_as_packets(tmp_path):
    jpegs = _jpegs(_frames(5, 64, 96))
    assert {len(j) % 4 for j in jpegs + _jpegs(_frames(5, 17, 33))} == {0, 1, 2, 3}
    path = str(tmp_path / "v.avi")
    with MjpegAviWriter(path, 30, (96, 64)) as wr:
        for j in jpegs:
            wr.write_jpeg(j)
    cap = cv2.VideoCapture(path, cv2.CAP_FFMPEG)
    if not cap.isOpened():
        pytest.skip("this OpenCV build has no FFmpeg backend")
    cap.set(cv2.CAP_PROP_FORMAT, -1)
    packets = []
    while True:
        ok, p = cap.read()
        if not ok:
            break
        packets.append(p.tobytes())
    assert len(packets) == 5
    for p, j in zip(packets, jpegs):
        assert p[:len(j)] == j and not any(p[len(j):])


def test_numpy_packing_is_what_write_jpeg_writes(tmp_path):
    jpegs = [j for n in (17, 18, 19, 20) for j in _jpegs(_frames(2, n, n + 3))]
    jpegs += [b"\xff\xd8\xff\xd9"[:k] for k in (1, 2, 3, 4)] + [b""]
    assert {len(j) % 4 for j in jpegs} == {0, 1, 2, 3}
    packed, offsets = pack_records(jpegs)
    assert all(packed[o:offsets[k + 1]].tobytes() == jpeg_record(j) for k, (o, j) in enumerate(zip(offsets, jpegs)))
    one = tmp_path / "one.avi"
    with MjpegAviWriter(str(one), 30, (8, 8)) as wr:
        for j in jpegs:
            wr.write_jpeg(j)
    buf = one.read_bytes()
    assert buf[4108:4108 + packed.size] == packed.tobytes()
    together = tmp_path / "together.avi"
    with MjpegAviWriter(str(together), 30, (8, 8)) as wr:
        wr.write_records(memoryview(packed[:offsets[5]]), [len(j) for j in jpegs[:5]])
        wr.write_records(packed[offsets[5]:].tobytes(), [len(j) for j in jpegs[5:]])
    assert together.read_bytes() == buf


def test_malformed_records_are_refused(tmp_path):
    j = _jpegs(_frames(2, 17, 33))
    packed, _ = pack_records(j)
    with MjpegAviWriter(str(tmp_path / "v.avi"), 30, (33, 17)) as wr:
        with pytest.raises(ValueError):
            wr.write_records(packed.tobytes(), [len(j[0])])             # lengths do not cover the records
        bad = packed.copy()
        bad[:4] = np.frombuffer(b"01wb", np.uint8)
        with pytest.raises(ValueError):
            wr.write_records(bad.tobytes(), [len(x) for x in j])
        assert wr.frames == 0
    for bad in (dict(fps=0.4), dict(size=(0, 8)), dict(size=(8, 70000))):
        with pytest.raises(ValueError):
            MjpegAviWriter(str(tmp_path / "w.avi"), **{"fps": 30, "size": (8, 8), **bad})


def test_a_record_past_the_riff_limit_raises_and_the_file_still_closes(tmp_path, monkeypatch):
    jpegs = _jpegs(_frames(6, 17, 33))
    sizes = [8 + ((len(j) + 3) & ~3) for j in jpegs]
    # room for exactly three frames and their index entries
    monkeypatch.setattr(mjpeg, "RIFF_MAX", 4108 + sum(sizes[:3]) + 8 + 16 * 3 - 8)
    path = str(tmp_path / "v.avi")
    wr = MjpegAviWriter(path, 30, (33, 17))
    wr.write_jpeg(jpegs[0])
    packed, _ = pack_records(jpegs[1:])
    with pytest.raises(ValueError, match="limit"):
        wr.write_records(packed.tobytes(), [len(j) for j in jpegs[1:]])     # the third record fits, the fourth does not
    with pytest.raises(ValueError, match="limit"):
        wr.write_jpeg(jpegs[3])
    assert wr.frames == 3
    wr.close()
    buf = open(path, "rb").read()
    assert len(buf) - 8 == mjpeg.RIFF_MAX
    check_layout(buf, jpegs[:3], 30, 33, 17)
    count, _, decoded = read_opencv(path)
    assert count == 3 and len(decoded) == 3
    for f, j in zip(decoded, jpegs):
        assert np.array_equal(f, cv2.imdecode(np.frombuffer(j, np.uint8), cv2.IMREAD_COLOR))
