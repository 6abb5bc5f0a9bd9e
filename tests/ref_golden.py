"""Results of the unmodified reference implementation (neonbjb/tortoise-tts) that the oracle tests compare against,
stored in tests/golden/reference_v1.pt so that the comparisons run without the reference tree.

A test asks for a result by key and passes the reference computation that produces it. Normally the stored result is
returned and the computation is not run. With TTB_RECORD_REFERENCE=1, where the reference is importable
(oracle/ref_shims.py), the computation runs, its result is stored under the key, and the test compares against it:

    TTB_RECORD_REFERENCE=1 python -m pytest tests/test_oracle_vs_reference.py tests/test_oracle_conditioning.py \\
        tests/test_cleaners.py tests/test_text_split.py

Tensors larger than the file should hold are stored as a fixed, seeded sample of their elements; results that a test
compares for exact equality are stored as a digest.
"""
import hashlib
import os

import torch

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_v1.pt")
RECORD = os.environ.get("TTB_RECORD_REFERENCE") == "1"
_store = None


def _get(key, compute, encode):
    global _store
    if _store is None:
        _store = torch.load(PATH) if os.path.exists(PATH) else {}
    if RECORD:
        _store[key] = encode(compute())
        torch.save(_store, PATH)
    return _store[key]


def _own(v):
    """Tensors copied out of the storage they may be a view of: only their own elements are saved."""
    if isinstance(v, torch.Tensor):
        return v.detach().clone()
    if isinstance(v, dict):
        return {k: _own(x) for k, x in v.items()}
    return v


def value(key, compute):
    """The reference result itself (a tensor, a dict of tensors, or a string)."""
    return _get(key, compute, _own)


def sampled(key, compute, k=2048):
    """(idx, values, shape) of a large reference tensor: `values` are its flattened elements at the positions `idx`,
    a seeded sample of k of them."""
    def encode(t):
        t = t.detach().float()
        idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:k].sort().values
        return {"idx": idx.int(), "val": t.reshape(-1)[idx].clone(), "shape": list(t.shape)}
    d = _get(key, compute, encode)
    return d["idx"].long(), d["val"], torch.Size(d["shape"])


def hexdigest(obj):
    """Digest of a result compared for exact equality: tensors by dtype, shape and bytes; lists, tuples, strings,
    numbers and None by value."""
    h = hashlib.sha256()

    def feed(o):
        if isinstance(o, torch.Tensor):
            h.update(("T%s%s" % (o.dtype, tuple(o.shape))).encode())
            h.update(o.detach().cpu().contiguous().numpy().tobytes())
        elif isinstance(o, (list, tuple)):
            h.update(b"[%d" % len(o))
            for x in o:
                feed(x)
        else:
            h.update(repr(o).encode())
    feed(obj)
    return h.hexdigest()[:16]


def digest(key, compute):
    """The digest (hexdigest) of the reference result."""
    return _get(key, compute, hexdigest)
