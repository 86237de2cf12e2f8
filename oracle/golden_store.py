"""Compact storage of golden inputs that are seeded `torch.randn` draws (tests/golden/*.npz).

A stored array `<key>` may instead appear as `<key>__seed`, `<key>__shape`, `<key>__idx`, `<key>__val` and
`<key>__sha256`: the array is `torch.randn(shape, generator=torch.Generator().manual_seed(seed))` with the flat
positions `idx` overwritten by `val`.  `expand` rebuilds it and checks the SHA-256 of its bytes, so a torch whose
generator draws other numbers fails loudly instead of comparing against different inputs.  Random float32 data does
not compress; this keeps every golden file well under 1 MB.
"""
import hashlib

import numpy as np
import torch

SUFFIXES = ("__seed", "__shape", "__idx", "__val", "__sha256")


def pack_seeded_randn(key, arr, seed):
    """The compact entries of `arr`, which must be a seeded randn draw with some positions overwritten."""
    arr = np.ascontiguousarray(arr, dtype=np.float32)
    base = torch.randn(arr.shape, generator=torch.Generator().manual_seed(int(seed))).numpy().reshape(-1)
    idx = np.flatnonzero(base != arr.reshape(-1))
    return {key + "__seed": np.array(int(seed), dtype=np.int64), key + "__shape": np.array(arr.shape, dtype=np.int64),
            key + "__idx": idx.astype(np.int64), key + "__val": arr.reshape(-1)[idx],
            key + "__sha256": np.array(hashlib.sha256(arr.tobytes()).hexdigest())}


def expand(npz):
    """A dict of the golden file's arrays, compact entries rebuilt."""
    out = {k: npz[k] for k in npz.files if not k.endswith(SUFFIXES)}
    for k in npz.files:
        if k.endswith("__seed"):
            key = k[:-len("__seed")]
            shape = tuple(int(v) for v in npz[key + "__shape"])
            a = torch.randn(shape, generator=torch.Generator().manual_seed(int(npz[k]))).numpy()
            a.reshape(-1)[npz[key + "__idx"]] = npz[key + "__val"]
            if hashlib.sha256(a.tobytes()).hexdigest() != str(npz[key + "__sha256"]):
                raise RuntimeError(f"golden {key}: torch.randn with seed {int(npz[k])} no longer draws the stored input")
            out[key] = a
    return out
