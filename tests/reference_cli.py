"""The reference csdr CLI's outputs on the CLI tests' seeded inputs, for machines where oracle/_ref/csdr_ref is not built.

The CLI tests run every command graph through the helpers decorated with @recorded.  With the compiled reference present they run it; with
CSDRB_RECORD_REF=1 as well, each of its results is kept and written to tests/golden/ref_cli.npz at exit:

    CSDR_REFERENCE=<csdr sources> python -c "import __graft_entry__ as g; g.build()"
    CSDRB_RECORD_REF=1 python -m pytest tests/test_cli_emulated.py

Without the reference the tests get REFERENCE in its place, and the helpers return the recorded result: a `Recorded` output keeps the length,
the SHA-256, the first HEAD bytes and CHUNKS seeded 8-byte pieces of what the reference wrote.  Whole outputs compare by length and digest,
values (`arr`, `rel`) at the kept positions.
"""
import atexit
import functools
import hashlib
import os
from pathlib import Path

import numpy as np

STORE = Path(__file__).resolve().parent / "golden" / "ref_cli.npz"
HEAD, CHUNKS = 64, 128
RECORD = os.environ.get("CSDRB_RECORD_REF") == "1"


class _Reference:
    """stands for the reference CLI in a test's (ours, ref) pair when only its recorded outputs are available"""

    def __repr__(self):
        return "reference-cli(recorded)"


REFERENCE = _Reference()


def _positions(n: int) -> np.ndarray:
    """byte offsets of the kept 8-byte pieces of an n-byte output (a function of n alone, so they are not stored)"""
    pieces = n // 8
    return np.sort(np.random.default_rng(n).choice(pieces, min(CHUNKS, pieces), replace=False)) * 8


class Recorded:
    """a sampled stand-in for the bytes a reference run wrote; sha is None for a part of an output"""

    def __init__(self, n, sha, head, pos, chunks):
        self.n, self.sha, self.head, self.pos, self.chunks = n, sha, head, pos, chunks

    @classmethod
    def of(cls, data: bytes):
        pos = _positions(len(data))
        return cls(len(data), hashlib.sha256(data).hexdigest(), data[:HEAD], pos, [data[p:p + 8] for p in pos])

    def encode(self) -> np.ndarray:
        return np.frombuffer(np.int64(self.n).tobytes() + bytes.fromhex(self.sha) + self.head + b"".join(self.chunks), np.uint8)

    @classmethod
    def decode(cls, a: np.ndarray):
        b = a.tobytes(); n = int(np.frombuffer(b[:8], np.int64)[0]); h = min(HEAD, n); pos = _positions(n); c = b[40 + h:]
        return cls(n, b[8:40].hex(), b[40:40 + h], pos, [c[8 * k:8 * k + 8] for k in range(pos.size)])

    def __len__(self):
        return self.n

    def __getitem__(self, s):
        start, stop, step = s.indices(self.n)
        assert step == 1, "only contiguous slices of a recorded output"
        keep = [(p - start, c) for p, c in zip(self.pos, self.chunks) if p >= start and p + 8 <= stop]
        whole = start == 0 and stop == self.n
        return Recorded(stop - start, self.sha if whole else None, self.head[start:min(stop, HEAD)] if start < HEAD else b"",
                        np.array([p for p, _ in keep], np.int64), [c for _, c in keep])

    def __eq__(self, other):
        if isinstance(other, Recorded):
            return self.n == other.n and self.sha is not None and self.sha == other.sha
        other = bytes(other)
        if len(other) != self.n:
            return False
        if self.sha is not None:
            return hashlib.sha256(other).hexdigest() == self.sha
        return other[:len(self.head)] == self.head and all(other[p:p + 8] == c for p, c in zip(self.pos, self.chunks))

    __hash__ = None

    def array(self, dtype):
        dt = np.dtype(dtype); s = dt.itemsize
        idx = [np.arange(len(self.head) // s)] + [p // s + np.arange(8 // s) for p in self.pos]
        vals = np.frombuffer(self.head[:len(self.head) // s * s] + b"".join(self.chunks), dt)
        return RecordedArray(self.n // s, np.concatenate(idx).astype(np.int64), vals)


class RecordedArray:
    """the values of a recorded output at known indices; comparisons with a full array happen at those indices"""
    __array_ufunc__ = None                                                  # make numpy hand `full == rec`, `full - rec` to the methods below

    def __init__(self, size, idx, vals):
        self.size, self.idx, self.vals = size, idx, vals

    def at(self, full):
        full = np.asarray(full)
        assert full.size >= self.size, (full.size, self.size)
        return full.reshape(-1)[self.idx]

    def __getitem__(self, s):
        start, stop, step = s.indices(self.size)
        assert step == 1
        m = (self.idx >= start) & (self.idx < stop)
        return RecordedArray(stop - start, self.idx[m] - start, self.vals[m])

    def astype(self, dtype):
        return RecordedArray(self.size, self.idx, self.vals.astype(dtype))

    def __eq__(self, other):
        return self.at(other) == self.vals

    def __sub__(self, other):
        return self.vals - self.at(other)

    def __rsub__(self, other):
        return self.at(other) - self.vals


def arr(out, dtype):
    """np.frombuffer for a run's output, recorded or not"""
    return out.array(dtype) if isinstance(out, Recorded) else np.frombuffer(out, dtype)


def rel_rms(a, b):
    from oracle.pyoracle import rel_rms as full
    if isinstance(b, RecordedArray):
        return full(b.at(a), b.vals)
    if isinstance(a, RecordedArray):
        return full(a.vals, a.at(b))
    return full(a, b)


def _key(name, args) -> str:
    h = hashlib.sha256(name.encode())
    for a in args:
        if isinstance(a, os.PathLike):                                      # per-run temporary paths do not change what the program computes
            continue
        if isinstance(a, Recorded):
            h.update(a.sha.encode())
        elif isinstance(a, (bytes, bytearray)):
            h.update(hashlib.sha256(a).hexdigest().encode())
        elif isinstance(a, list) and a and isinstance(a[0], (bytes, bytearray)):
            h.update(hashlib.sha256(b"".join(a)).hexdigest().encode())
        else:
            h.update(repr(a).encode())
    return h.hexdigest()[:24]


_store = None
_taken = {}


def _load():
    global _store
    if _store is None:
        _store = dict(np.load(STORE)) if STORE.exists() else {}
    return _store


@atexit.register
def _save():
    if _taken:
        np.savez_compressed(STORE, **_taken)


def recorded(fn):
    """run `fn(cli, ...)` for a real program; for REFERENCE return what the reference CLI gave on the same arguments"""
    @functools.wraps(fn)
    def run(cli, *args, **kw):
        k = _key(fn.__name__, args + tuple(v for _, v in sorted(kw.items())))
        if cli is REFERENCE:
            a = _load().get(k)
            assert a is not None, f"{fn.__name__}: no recorded reference output for these arguments (tests/reference_cli.py says how to record them)"
            return bool(a[0]) if a.dtype == np.bool_ else Recorded.decode(a)
        out = fn(cli, *args, **kw)
        if RECORD and str(cli).endswith("csdr_ref"):
            _taken[k] = np.array([out]) if isinstance(out, bool) else Recorded.of(bytes(out)).encode()
        return out
    return run
