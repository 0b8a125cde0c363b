"""Shared helpers for the test-suite: fixtures, synthetic inputs, native bindings."""
import bz2
import ctypes as C
import functools
import hashlib
import json
import lzma
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


@functools.lru_cache(maxsize=None)
def fixture(name):
    """The reference's test fixture `name` (its test/sample*.ref, *.bz2, *.bzt and block files), rebuilt from
    tests/golden/fixtures as tests/golden/fixtures.json describes: the .ref texts are stored xz-compressed and the
    .bzt tables as they are; every .bz2 of the reference is libbz2's stream of its .ref at the level in its header, and
    a block file is a slice of its .ref.  The result must have the size and SHA-256 of the reference's file."""
    with open(os.path.join(GOLDEN, "fixtures.json")) as f:
        spec = json.load(f)[name]
    path = os.path.join(GOLDEN, "fixtures", name)
    if "bzip2_level" in spec:
        data = bz2.compress(fixture(spec["from"]), spec["bzip2_level"])
    elif "offset" in spec:
        data = fixture(spec["from"])[spec["offset"]:spec["offset"] + spec["size"]]
    elif os.path.exists(path + ".xz"):
        with open(path + ".xz", "rb") as f:
            data = lzma.decompress(f.read())
    else:
        with open(path, "rb") as f:
            data = f.read()
    got = (len(data), hashlib.sha256(data).hexdigest())
    assert got == (spec["size"], spec["sha256"]), "fixture %s rebuilt as %r, not the reference's file" % (name, got)
    return data


def rng(seed):
    return np.random.Generator(np.random.PCG64(seed))


def ascii_random(n, seed=20260923):
    """BASELINE config 2 generator: uniform over 94 printable bytes + newline."""
    a = rng(seed).integers(32, 127, size=n, dtype=np.uint8)
    a[a == 126] = 10
    return a.tobytes()


def texty(n, seed=1):
    """Cheap text-like data with long repeats (word soup from a small vocabulary)."""
    g = rng(seed)
    vocab = [bytes(g.integers(97, 123, size=int(l), dtype=np.uint8)) for l in g.integers(2, 9, size=200)]
    out = bytearray()
    while len(out) < n:
        k = int(g.integers(0, 200))
        out += vocab[k] + (b" " if g.random() < 0.9 else b".\n")
        if g.random() < 0.01 and len(out) > 5000:
            s = int(g.integers(0, len(out) - 3000))
            out += out[s:s + int(g.integers(200, 3000))]
    return bytes(out[:n])


def runs(n, seed=2):
    """Run-heavy data exercising RLE1 (runs of 1..600 bytes)."""
    g = rng(seed)
    out = bytearray()
    while len(out) < n:
        out += bytes([int(g.integers(0, 256))]) * int(g.choice([1, 2, 3, 4, 5, 6, 7, 100, 255, 256, 259, 260, 600, 1000]))
    return bytes(out[:n])


def native():
    from compressjs_b200 import _native
    return _native


def native_bwt(data):
    N = native()
    L = N.lib()
    a = np.frombuffer(data, dtype=np.uint8)
    u = np.zeros(max(a.size, 1), dtype=np.uint8)
    p = L.b2_bwt_cyclic(a.ctypes.data if a.size else None, u.ctypes.data, a.size)
    assert p >= 0, N.last_error()
    return u[:a.size].tobytes(), p


def native_bwt_batch(blocks):
    N = native()
    L = N.lib()
    lens = np.array([len(b) for b in blocks], dtype=np.int32)
    offs = np.zeros(len(blocks), dtype=np.uint64)
    offs[1:] = np.cumsum(lens[:-1].astype(np.uint64))
    cat = np.frombuffer(b"".join(blocks), dtype=np.uint8)
    u = np.zeros(max(cat.size, 1), dtype=np.uint8)
    pidx = np.zeros(len(blocks), dtype=np.int32)
    rc = L.b2_bwt_cyclic_batch(cat.ctypes.data, u.ctypes.data, offs.ctypes.data, lens.ctypes.data, pidx.ctypes.data, len(blocks))
    assert rc == 0, N.last_error()
    res = []
    for o, l, p in zip(offs, lens, pidx):
        res.append((u[int(o):int(o) + int(l)].tobytes(), int(p)))
    return res


def golden():
    import json
    p = os.path.join(ROOT, "tests", "golden", "golden.json")
    with open(p) as f:
        return json.load(f)
