"""Synthetic workloads of BASELINE.json / SURVEY.md section 8d.

config 2: uniform ASCII (bench.py gen_ascii).
config 3: "enwik8-shaped" text: order-3 byte Markov chain trained on the reference's test/sample5.ref
          (HTML/wikitext, 201 symbols), PCG64 seed 20260923, plus ~1 % injected long repeats
          (copy 200-5000 bytes from >= 64 KiB back).  Vectorised: many independent chains are advanced in
          lock-step and concatenated, which keeps the order-3 statistics and is fast enough for 100 MB.
"""
import lzma
import os
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _train_bytes():
    # the reference's test/sample5.ref, kept xz-compressed with the test fixtures
    with open(os.path.join(ROOT, "tests", "golden", "fixtures", "sample5.ref.xz"), "rb") as f:
        return np.frombuffer(lzma.decompress(f.read()), dtype=np.uint8)


def enwik_like(nbytes, seed=20260923, chains=4096):
    g = np.random.Generator(np.random.PCG64(seed))
    t = _train_bytes().astype(np.int64)
    n = t.size
    # successor table of every order-3 context: contexts sorted, successors grouped
    ctx = (t[:-3] << 16) | (t[1:-2] << 8) | t[2:-1]
    nxt = t[3:]
    order = np.argsort(ctx, kind="stable")
    ctx_s, nxt_s = ctx[order], nxt[order].astype(np.uint8)
    uniq, start, count = np.unique(ctx_s, return_index=True, return_counts=True)
    per = (nbytes + chains - 1) // chains
    out = np.empty((chains, per), dtype=np.uint8)
    pos0 = g.integers(0, n - 4, size=chains)
    cur = ctx[np.minimum(pos0, ctx.size - 1)]
    for j in range(per):
        k = np.searchsorted(uniq, cur)
        k = np.minimum(k, uniq.size - 1)
        miss = uniq[k] != cur
        if miss.any():  # unseen context (chain boundary effects): restart from a random training position
            cur[miss] = ctx[g.integers(0, ctx.size, size=int(miss.sum()))]
            k = np.searchsorted(uniq, cur)
        r = (g.random(chains) * count[k]).astype(np.int64)
        b = nxt_s[start[k] + r]
        out[:, j] = b
        cur = ((cur << 8) & 0xFFFFFF) | b
    data = out.reshape(-1)[:nbytes].copy()
    # ~1 % of the bytes are long repeats copied from at least 64 KiB back
    budget, i = nbytes // 100, 1 << 17
    while budget > 0 and i < nbytes - 6000:
        ln = int(g.integers(200, 5001))
        src = int(g.integers(0, i - 65536))
        data[i:i + ln] = data[src:src + ln]
        budget -= ln
        i += int(g.integers(ln + 1, max(ln + 2, 2 * nbytes // max(nbytes // 100 // 2600, 1))))
    return data
