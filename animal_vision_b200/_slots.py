"""Shared tail of the device encoders (K8 JPEG, K10 PNG): each frame's file is written into a fixed-size slot of a
device buffer with its length in a device array, so only the lengths and then the used bytes cross to the host."""
from __future__ import annotations

import threading
from typing import Callable, Dict, List

import numpy as np

from ._abi import check

_locks: Dict[tuple, threading.Lock] = {}
_locks_guard = threading.Lock()


def _lock_for(key: tuple) -> threading.Lock:
    with _locks_guard:
        return _locks.setdefault(key, threading.Lock())


def encode_slots(eng, name: str, n: int, slot: int, need: int, launch: Callable[[int, int, int, int], int],
                 launches: int) -> List[bytes]:
    """Run `launch(workspace_ptr, out_ptr, slot, lengths_ptr) -> rc` with `need` bytes of workspace and n slots of `slot`
    bytes, on the engine's current stream; return the n files.  Buffers are cached per stream, so encodes on
    different streams may overlap; host threads encoding on the same stream take turns on one lock per buffer set, so
    one cannot overwrite another's slots before they are copied back.  Call with the engine's device current."""
    if slot <= 0 or need <= 0:
        check(min(slot, need), f"avb_{name}_workspace_bytes")
    key = (name, eng.stream_ptr())
    with _lock_for((id(eng), key)):
        return _encode_locked(eng, key, n, slot, need, launch, launches)


def _encode_locked(eng, key, n, slot, need, launch, launches) -> List[bytes]:
    import torch
    name = key[0]
    bufs = eng._cache.get(key)
    if bufs is None or bufs[0].numel() < need or bufs[1].numel() < n * slot or bufs[2].numel() < n:
        eng._cache[key] = None
        bufs = eng._cache[key] = (torch.empty(need, dtype=torch.uint8, device=eng.device),
                                  torch.empty(n * slot, dtype=torch.uint8, device=eng.device),
                                  torch.empty(n, dtype=torch.int64, device=eng.device))
    ws, out, lengths = bufs
    check(launch(ws.data_ptr(), out.data_ptr(), slot, lengths.data_ptr()), f"avb_{name}_encode_u8")
    eng.launches += launches
    lens = lengths[:n].cpu().tolist()                   # waits for the encode
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    host = torch.empty(int(offs[-1]), dtype=torch.uint8).pin_memory()
    for f in range(n):
        host[int(offs[f]):int(offs[f + 1])].copy_(out[f * slot:f * slot + lens[f]], non_blocking=True)
    torch.cuda.current_stream(eng.device).synchronize()
    buf = host.numpy().tobytes()
    return [buf[int(offs[f]):int(offs[f + 1])] for f in range(n)]
