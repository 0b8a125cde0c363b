"""Generates tests/golden/golden.json: outputs of the CPU oracle (oracle/bz2_oracle.c) on the
reference's own test inputs (its test/sample*.ref, stored under tests/golden/fixtures).  These are the
pinned outputs of the oracle, the C restatement of the reference's JavaScript; sizes in legacy-sort
mode equal README.md:42,45 of the reference.  Run:  python tests/golden/make_golden.py
"""
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import oracle as O  # noqa: E402
from tests.util import fixture  # noqa: E402

out = {}
for k in range(6):
    name = "sample%d" % k
    data = fixture(name + ".ref")
    out["ref_%s" % name] = {"size": len(data), "sha256": hashlib.sha256(data).hexdigest()}
    for lv in (1, 9):
        z, tr = O.bzip2_compress(data, lv, trace=True)
        out["bzip2_%s_-%d" % (name, lv)] = {
            "size": len(z), "sha256": hashlib.sha256(z).hexdigest(),
            "blocks": [{"n": t.n, "pidx": t.pidx, "m": t.m, "alpha": t.alpha, "ngroups": t.ngroups, "nsel": t.nsel,
                        "crc": t.crc, "bit_start": t.bit_start, "bit_len": t.bit_len} for t in tr]}
    for lv in (1, 6, 9):   # BWTC container (oracle/bwtc_oracle.c); -9 and sample5 -1 equal SURVEY.md section 8c / README.md:41,46
        z = O.bwtc_compress(data, lv)
        out["bwtc_%s_-%d" % (name, lv)] = {"size": len(z), "sha256": hashlib.sha256(z).hexdigest()}
for lv in (1, 9):
    z = O.bzip2_compress(fixture("sample5.ref"), lv, legacy_sort=True)
    out["bzip2_sample5_-%d_legacy_v8_sort" % lv] = {"size": len(z), "sha256": hashlib.sha256(z).hexdigest()}
json.dump(out, open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden.json"), "w"), indent=1, sort_keys=True)
print("wrote", len(out), "entries")
