"""Server-side batching beside the reference's `processimage` (utils.py:133-199) and its socket loop
(server/server.py:40-68), SURVEY.md 8f-4.

The reference handles one socket's frame at a time: JPEG bytes -> temp.jpg -> cv2.imread -> `filter.visualize(img)[1]` ->
tempexport.jpg -> base64 data URI, and the asyncio loop blocks on it.  Here every frame that is waiting -- from any
number of sockets -- is grouped by (species key, frame shape) and each group runs as ONE device batch through
`visualize_batch`; JPEG decode stays on the host and in memory (no temp files).  `FrameBatcher.submit` is thread
safe and returns a `concurrent.futures.Future`; `process_image` is the drop-in for `processimage` (same arguments, same
data-URI result, same string keys: "human", "cat", "cow", ... as utils.py:145-191, plus keys for the UV species).

`FrameBatcher.submit_jpeg` asks for the JPEG file of the species view instead of its pixels.  Where the batch result
lives decides the encoder: a view left on the device by the default runner is encoded there (K8, `jpeg.encode_jpeg`,
the bytes of cv2.imencode) and only the compressed bytes come back; a NumPy result is encoded with cv2.imencode.
`FrameBatcher.submit_png` does the same with PNG (K10, `png.encode_png`), and `process_image_png` wraps it as a data URI.
`optimize=True` on the JPEG requests asks for the bytes cv2.imencode gives with IMWRITE_JPEG_OPTIMIZE: Huffman tables
built from each file's own symbol counts, the same pixels in fewer bytes (on the device, K8's optimized mode).

`FrameBatcher.submit_split_jpeg` asks for the JPEG file of the labelled split-compare frame of the request's input and
its species view -- what the reference's CLI shows (main.py:41-48 `render_split_compare(img, out)`, with the defaults of
`make_split_frame`).  Split requests share the species launch of their (key, shape) group with pixel and JPEG requests;
on the device they are composed (K9, `split_compare_batch(..., labels=...)`) per distinct (labels, seam) from the input
the runner already uploaded, and encoded by K8.  `process_split_image` wraps it as a data URI.  The reference server's
`processsplitimage` (utils.py:202-336) is not restated here: this is the split frame defined above, not a drop-in."""
from __future__ import annotations

import base64
import threading
import time
from collections import OrderedDict, deque
from concurrent.futures import Future
from typing import Callable, Dict, List, Optional, Tuple

import numpy as np

from . import animals as A

# the reference's lower-case server keys (utils.py:145-191) and, beyond them, one key per remaining registry entry
SERVER_KEYS: Dict[str, str] = {
    "cat": "Cat", "cow": "Cow", "goat": "Goat", "pig": "Pig", "sheep": "Sheep", "dog": "Dog", "rat": "Rat", "horse": "Horse",
    "rabbit": "Rabbit", "panda": "Panda", "squirrel": "Squirrel", "elephant": "Elephant", "lion": "Lion", "wolf": "Wolf", "fox": "Fox",
    "bear": "Bear", "raccoon": "Raccoon", "deer": "Deer", "kangaroo": "Kangaroo", "tiger": "Tiger", "honeybee": "HoneyBee",
    "reindeer": "Reindeer", "ratuv": "RatUV", "goldfish": "Goldfish", "damselfish": "Damselfish", "anableps": "Anableps",
    "anchovy": "Anchovy", "guppy": "Guppy", "morpho": "Morpho", "heliconius": "Heliconius", "pieris": "Pieris",
    "mantisshrimp": "MantisShrimp", "kestrel": "Kestrel", "jumpingspider": "JumpingSpider", "dragonfly": "Dragonfly",
    "hummingbird": "Hummingbird",
}


class _DeviceRunner:
    """run(key, frames[k,H,W,3] uint8) -> the species view of every frame, a [k,H,W,3] uint8 CUDA tensor (index [1] of
    `visualize`), enqueued on the current stream.  `upload_and_run` also returns the uploaded input, so split requests
    compose from it without a second upload."""

    def __init__(self, device=None):
        self.device = device
        self.species: Dict[str, object] = {}

    def upload_and_run(self, key: str, frames: np.ndarray):
        from .engine import get_engine
        eng = get_engine(self.device)
        t = eng.torch
        sp = self.species.get(key)
        if sp is None:
            sp = self.species[key] = getattr(A, SERVER_KEYS[key])()
        with t.cuda.device(eng.device):
            pin = t.from_numpy(frames).pin_memory()
            dev = pin.to(eng.device, non_blocking=True)
            return dev, sp.visualize_batch(dev)[1]

    def __call__(self, key: str, frames: np.ndarray):
        return self.upload_and_run(key, frames)[1]


def _device_runner(device=None) -> _DeviceRunner:
    return _DeviceRunner(device)


def _rows(batch, idx: List[int]):
    """The frames `idx` of a device batch: the batch itself when that is all of them, else one gather."""
    import torch
    return batch if len(idx) == batch.shape[0] else batch[torch.tensor(idx, device=batch.device)]


def _pixels(view, idx: List[int]) -> List[np.ndarray]:
    """The frames `idx` of a batch result as host arrays (one D2H copy for a device result)."""
    if isinstance(view, np.ndarray):
        return [np.array(view[i], copy=True) for i in idx]
    import torch
    with torch.cuda.device(view.device):
        sel = _rows(view, idx)
        pin = torch.empty(tuple(sel.shape), dtype=torch.uint8).pin_memory()
        pin.copy_(sel, non_blocking=True)
        torch.cuda.current_stream(view.device).synchronize()
        return [pin[k].numpy() for k in range(len(idx))]


# encoded request kinds: cv2's extension for each, and whether it sets IMWRITE_JPEG_OPTIMIZE
_HOST_EXT = {"jpeg": (".jpg", False), "jpeg_opt": (".jpg", True), "png": (".png", False)}


def _encode_host(frame: np.ndarray, fmt: str = "jpeg") -> bytes:
    import cv2
    ext, optimize = _HOST_EXT[fmt]
    ok, enc = cv2.imencode(ext, frame, [cv2.IMWRITE_JPEG_OPTIMIZE, 1]) if optimize else cv2.imencode(ext, frame)
    if not ok:
        raise ValueError("could not encode the result")
    return enc.tobytes()


def _encoded(view, idx: List[int], fmt: str) -> List[bytes]:
    """Files of the frames `idx` of a batch result, the bytes cv2.imencode gives with its defaults: JPEG at quality 95
    (fmt "jpeg"; "jpeg_opt" with IMWRITE_JPEG_OPTIMIZE) or PNG (fmt "png")."""
    if isinstance(view, np.ndarray):
        return [_encode_host(view[i], fmt) for i in idx]
    import torch
    from .jpeg import encode_jpeg
    from .png import encode_png
    with torch.cuda.device(view.device):
        sel = _rows(view, idx)
        return encode_png(sel) if fmt == "png" else encode_jpeg(sel, 95, optimize=fmt == "jpeg_opt")


def _split_host(frame: np.ndarray, view: np.ndarray, labels: Tuple[str, str], seam: bool, optimize: bool = False) -> bytes:
    """The host route of a split request: slice copies, cv2 labels, cv2.imencode."""
    import torch
    from .renderers.video import draw_split_labels, split_compare_batch
    comp = split_compare_batch(torch.from_numpy(frame[None]), torch.from_numpy(np.ascontiguousarray(view)[None]),
                               draw_seam=seam)[0].numpy()
    return _encode_host(draw_split_labels(comp, *labels), "jpeg_opt" if optimize else "jpeg")


def _split_jpegs(frames: np.ndarray, dev_in, view, idx: List[int], labels: Tuple[str, str], seam: bool,
                 optimize: bool = False) -> List[bytes]:
    """JPEG files of the labelled split frames (input | species view) of the frames `idx` of a batch."""
    if isinstance(view, np.ndarray):
        return [_split_host(frames[i], view[i], labels, seam, optimize) for i in idx]
    import torch
    from .jpeg import encode_jpeg
    from .renderers.video import split_compare_batch
    with torch.cuda.device(view.device):
        if dev_in is None:
            dev_in = torch.from_numpy(frames).pin_memory().to(view.device, non_blocking=True)
        orig, sel = _rows(dev_in, idx), _rows(view, idx)
        return encode_jpeg(split_compare_batch(orig, sel, draw_seam=seam, labels=labels), 95, optimize=optimize)


def _check_labels(labels) -> Tuple[str, str]:
    if not (isinstance(labels, (tuple, list)) and len(labels) == 2 and all(isinstance(x, str) for x in labels)):
        raise TypeError(f"labels must be a pair of strings, got {labels!r}")
    return (labels[0], labels[1])


class FrameBatcher:
    """Collects (frame, species key) requests from any number of producers and runs them as device batches.

    A worker thread takes everything that is pending (waiting up to `max_delay_ms` for stragglers once a request is in,
    never beyond `max_batch` frames per launch), groups it by (key, shape) in arrival order and resolves every request's
    Future with its own output frame.  `run_batch` is injectable (tests run the host logic without a GPU)."""

    def __init__(self, run_batch: Optional[Callable[[str, np.ndarray], np.ndarray]] = None, *, max_batch: int = 16,
                 max_delay_ms: float = 2.0, device=None):
        self._run = run_batch if run_batch is not None else _device_runner(device)
        self.max_batch, self.max_delay = int(max_batch), float(max_delay_ms) * 1e-3
        self._q: deque = deque()
        self._cv = threading.Condition()
        self._stop = False
        self.batches: List[Tuple[str, int]] = []            # (key, frames) of every launch, for inspection
        self._worker = threading.Thread(target=self._loop, name="avb-batcher", daemon=True)
        self._worker.start()

    def submit(self, frame: np.ndarray, animal: str) -> Future:
        """Future of the species view of `frame`, an HxWx3 uint8 array."""
        return self._submit(frame, animal, None)

    def submit_jpeg(self, frame: np.ndarray, animal: str, optimize: bool = False) -> Future:
        """Future of the JPEG file (bytes) of the species view, the bytes cv2.imencode(".jpg", view) gives; with
        `optimize`, the bytes of cv2.imencode(".jpg", view, [cv2.IMWRITE_JPEG_OPTIMIZE, 1])."""
        return self._submit(frame, animal, "jpeg_opt" if optimize else "jpeg")

    def submit_png(self, frame: np.ndarray, animal: str) -> Future:
        """Future of the PNG file (bytes) of the species view, the bytes cv2.imencode(".png", view) gives."""
        return self._submit(frame, animal, "png")

    def submit_split_jpeg(self, frame: np.ndarray, animal: str, labels: Tuple[str, str] = ("Original", "Transformed"),
                          draw_seam: bool = True, optimize: bool = False) -> Future:
        """Future of the JPEG file (bytes) of the split-compare frame of `frame` and its species view: left half of
        the input, right half of the view, the seam, and the two corner labels -- the bytes of
        cv2.imencode(".jpg", draw_split_labels(split frame, *labels)), with IMWRITE_JPEG_OPTIMIZE if `optimize`."""
        try:
            kind = ("split", _check_labels(labels), bool(draw_seam), bool(optimize))
        except TypeError as e:
            fut: Future = Future()
            fut.set_exception(e)
            return fut
        return self._submit(frame, animal, kind)

    def _submit(self, frame: np.ndarray, animal: str, kind) -> Future:
        """kind: None (pixels), "jpeg", "jpeg_opt", "png", or ("split", labels, seam, optimize)."""
        fut: Future = Future()
        if animal != "human" and animal not in SERVER_KEYS:
            fut.set_exception(KeyError(f"no case implemented for {animal!r}"))             # utils.py:192-193 prints and fails later
            return fut
        if not (isinstance(frame, np.ndarray) and frame.ndim == 3 and frame.shape[2] == 3 and frame.dtype == np.uint8):
            fut.set_exception(AssertionError("frame must be a HxWx3 uint8 array"))
            return fut
        if animal == "human":                                                               # utils.py:146-147
            if kind is None:
                fut.set_result(frame)
                return fut
            try:
                fut.set_result(_encode_host(frame, kind) if kind in _HOST_EXT else _split_host(frame, frame, *kind[1:]))
            except Exception as e:          # noqa: BLE001
                fut.set_exception(e)
            return fut
        with self._cv:
            if self._stop:
                raise RuntimeError("FrameBatcher is closed")
            self._q.append((animal, frame, fut, kind))
            self._cv.notify()
        return fut

    def _loop(self):
        while True:
            with self._cv:
                while not self._q and not self._stop:
                    self._cv.wait()
                if self._stop and not self._q:
                    return
                deadline = time.monotonic() + self.max_delay
                while len(self._q) < self.max_batch and not self._stop:
                    left = deadline - time.monotonic()
                    if left <= 0:
                        break
                    self._cv.wait(left)
                pending = list(self._q)
                self._q.clear()
            groups: "OrderedDict[Tuple[str, Tuple[int, ...]], list]" = OrderedDict()
            for animal, frame, fut, kind in pending:
                groups.setdefault((animal, frame.shape), []).append((frame, fut, kind))
            for (animal, _shape), items in groups.items():
                for a in range(0, len(items), self.max_batch):
                    part = items[a:a + self.max_batch]
                    try:
                        self._run_part(animal, part)
                    except Exception as e:          # noqa: BLE001  (a failed batch fails its own requests, the loop lives on)
                        for _, fut, _ in part:
                            if not fut.done():
                                fut.set_exception(e)

    def _run_part(self, animal: str, part: list):
        """One species launch for the requests `part` of one (key, shape) group, then each request's own result."""
        batch = np.stack([f for f, _, _ in part])
        splits: "OrderedDict[tuple, List[int]]" = OrderedDict()
        for i, (_, _, kind) in enumerate(part):
            if kind is not None and kind not in _HOST_EXT:
                splits.setdefault(kind[1:], []).append(i)
        upload_and_run = getattr(self._run, "upload_and_run", None)
        if splits and upload_and_run is not None:
            dev_in, out = upload_and_run(animal, batch)
        else:
            dev_in, out = None, self._run(animal, batch)
        self.batches.append((animal, len(part)))
        pix = [i for i, (_, _, kind) in enumerate(part) if kind is None]
        res = dict(zip(pix, _pixels(out, pix))) if pix else {}
        for fmt in _HOST_EXT:
            idx = [i for i, (_, _, kind) in enumerate(part) if kind == fmt]
            if idx:
                res.update(zip(idx, _encoded(out, idx, fmt)))
        for (labels, seam, optimize), idx in splits.items():
            res.update(zip(idx, _split_jpegs(batch, dev_in, out, idx, labels, seam, optimize)))
        for i, (_, fut, _) in enumerate(part):
            fut.set_result(res[i])

    def close(self):
        with self._cv:
            self._stop = True
            self._cv.notify_all()
        self._worker.join(timeout=10)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


_default: Optional[FrameBatcher] = None
_default_lock = threading.Lock()


def default_batcher() -> FrameBatcher:
    global _default
    with _default_lock:
        if _default is None:
            _default = FrameBatcher()
        return _default


def _data_uri(imagedata: bytes, submit: Callable[[np.ndarray], Future], mime: str) -> str:
    """Decodes `imagedata` BGR as cv2.imread gives it, submits the frame and returns the encoded result as a base64
    data URI of type `mime`."""
    import cv2
    img = cv2.imdecode(np.frombuffer(imagedata, np.uint8), cv2.IMREAD_COLOR)
    if img is None:
        raise ValueError("could not decode the image")
    return f"data:{mime};base64," + base64.b64encode(submit(img).result()).decode("utf-8")


def process_image(imagedata: bytes, animal: str, batcher: Optional[FrameBatcher] = None, *, optimize: bool = False) -> str:
    """Drop-in for utils.py:133-199 `processimage`: JPEG bytes in, JPEG data URI out; decoded BGR as cv2.imread gives it
    (the species index channels 0/1/2, never "R/G/B" -- the reference feeds BGR here too, utils.py:141-142).
    `optimize=True` answers with the smaller file of IMWRITE_JPEG_OPTIMIZE (same pixels)."""
    return _data_uri(imagedata, lambda img: (batcher or default_batcher()).submit_jpeg(img, animal, optimize),
                     "image/jpeg")


def process_image_png(imagedata: bytes, animal: str, batcher: Optional[FrameBatcher] = None) -> str:
    """`process_image` with a lossless result: image bytes in, data URI of the PNG of the species view out
    (`FrameBatcher.submit_png`, the bytes of cv2.imencode(".png", view))."""
    return _data_uri(imagedata, lambda img: (batcher or default_batcher()).submit_png(img, animal), "image/png")


def process_split_image(imagedata: bytes, animal: str, labels: Tuple[str, str] = ("Original", "Transformed"),
                        batcher: Optional[FrameBatcher] = None, *, optimize: bool = False) -> str:
    """JPEG bytes in, data URI of the JPEG of the labelled split-compare frame out (input on the left, species view on
    the right, seam, corner labels; `FrameBatcher.submit_split_jpeg`).  Decoded BGR as cv2.imread gives it, like
    `process_image`; `optimize` as there."""
    return _data_uri(imagedata, lambda img: (batcher or default_batcher()).submit_split_jpeg(
        img, animal, labels, optimize=optimize), "image/jpeg")
