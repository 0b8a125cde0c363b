"""bench.py -- headline benchmark of the bzip2 block pipeline (BASELINE.json).

  python bench.py --gpus 1 --steps K --warmup W            our arm (CUDA, libb2bz.so)
  python bench.py --impl reference --gpus 1 ...            the reference's CPU path (oracle port)
  torchrun ... bench.py --gpus N ...                       one rank per GPU, weak scaling

A step = one bzip2 -9 encode of the workload (BASELINE configs[1]: 1 GiB synthetic ASCII per GPU,
numpy PCG64 seed 20260923, 94 printable bytes + newline).  `value` = whole-job MB/s (10^6 raw bytes
per second) with the input resident in HBM; `e2e` = the same through the host-buffer C ABI call
(b2_bzip2_compress: H2D + all kernels + D2H inside the timed region).  The roofline entry is for the
dominant kernel of the forward BWT (k_msd_bucket, the shared-memory bucket sort that follows the MSD
scatter pass): algorithmic bytes per launch over its CUDA-event time, against the measured HBM copy
bandwidth; `roofline.bwt_stage` is the whole forward BWT.  Further objects on the same line:
`parity` (oracle vs the first blocks of the benchmarked stream), `decode` (resident + end to end +
roofline), `config3` (100 MB enwik-shaped text, encode + decode), `bwtc` (BASELINE configs[3]),
`cpu_baseline`.

--dump-outputs DIR writes what the last timed step returned (the .bz2 stream, sampled) as .npy files under DIR, so
that the streams of two builds can be compared; see dump_outputs().
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from, which may be read-only

import numpy as np  # noqa: E402

SEED = 20260923
LEVEL = 9
METRIC = "bzip2_-9_encode_MBps"
BS9 = LEVEL * 100000 - 19
DUMP_HEAD, DUMP_TAIL, DUMP_SAMPLE = 1 << 20, 1 << 16, 4 << 20   # stream bytes --dump-outputs keeps


def gen_ascii(nbytes, seed):
    g = np.random.Generator(np.random.PCG64(seed))
    out = np.empty(nbytes, dtype=np.uint8)
    step = 1 << 26
    for o in range(0, nbytes, step):
        k = min(step, nbytes - o)
        a = g.integers(32, 127, size=k, dtype=np.uint8)
        a[a == 126] = 10
        out[o:o + k] = a
    return out


class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self, t0=None, t1=None):
        """Samples taken inside [t0, t1] (perf_counter) -- the sampler is started before the warm-up because
        nvidia-smi needs about a second to deliver its first line."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        inside = [r for (t, r) in self.rows if (t0 is None or t >= t0) and (t1 is None or t <= t1)]
        window = "timed region"
        if not inside:
            inside, window = [r for (_, r) in self.rows], "whole run (no sample fell into the timed region)"
        self.rows = inside
        self.window = window
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) > 8 and r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in self.rows if len(r) > 8 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) > 8:
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(self.rows), "window": self.window}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def traffic_from_profiles():
    """DRAM bytes per record of the BWT kernels from the committed `ncu --set full` captures."""
    p = os.path.join(ROOT, "profiles", "bwt_kernel_traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            return None
    return None


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference(args):
    """The reference's own CPU implementation of the path (its JavaScript cannot run here: no node in the
    image; this is the C restatement in oracle/, all host threads), on a bounded sample per step.  Encode is the
    line's metric; a decode leg of the same sample follows (`decode`)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    O.build()
    cores = max(1, min(host_cores(), 32))  # one 900k block (~60 MB of working set) per thread; more threads only thrash the host caches
    per_step_blocks = max(2, cores)        # one 900k block per core and step keeps the run in minutes
    data = gen_ascii(min(args.mb << 20, per_step_blocks * 900000 + 1000), SEED)
    sample = np.ascontiguousarray(data[: min(len(data), per_step_blocks * BS9)])
    for _ in range(args.warmup):
        O.bzip2_compress(sample[: 2 * 900000], LEVEL, threads=cores)
    t0 = time.perf_counter()
    z = None
    for _ in range(args.steps):
        z = O.bzip2_compress(sample, LEVEL, threads=cores)
    dt = time.perf_counter() - t0
    val = sample.size * args.steps / dt / 1e6
    # decode leg: the reference's decoder is single threaded per stream (lib/Bzip2.js:454-481)
    dsteps = max(1, min(args.steps, 2))
    td = time.perf_counter()
    for _ in range(dsteps):
        back = O.bzip2_decompress(z)
    ddt = time.perf_counter() - td
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "MB/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic",
        "config": {"workload": "1 GiB synthetic ASCII (PCG64 seed %d), bzip2 -9 (900k blocks) encode" % SEED, "level": LEVEL,
                   "sample": "first %d blocks (%d bytes) per step" % (per_step_blocks, sample.size)},
        "cpu_baseline": {"value": val, "unit": "MB/s", "cores": cores, "kind": "port",
                         "sample": "%d x 900k blocks per step, %d threads (oracle/bz2_oracle.c, one block per thread)" % (per_step_blocks, cores)},
        "e2e": {"value": val, "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "decode": {"metric": "bzip2_-9_decode_MBps", "value": sample.size * dsteps / ddt / 1e6, "unit": "MB/s", "cores": 1, "steps": dsteps,
                   "roundtrip_ok": bool(back == sample.tobytes()), "sample": "the stream of the encode sample, oracle decoder, 1 thread"},
        "note": "reference JS cannot execute in this image (no node); C restatement of its algorithm timed instead",
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------
def _check(rc, what, _native):
    if rc:
        raise SystemExit("%s failed: %s" % (what, _native.last_error()))


def prefix_parity(L, _native, host, d_out, comp_bytes, trace, nblocks_check, threads):
    """Oracle (CPU restatement of the reference) on the first blocks of the workload against the benchmarked
    stream: the bits in front of block K must be identical."""
    import torch
    from oracle import oracle as O
    O.build()
    K = min(nblocks_check, len(trace) - 1)
    if K < 1:
        return {"blocks": 0, "ok": None, "note": "stream has fewer than two blocks"}
    raw_end = int(trace[K].raw_start)  # first raw byte of block K
    sample = np.ascontiguousarray(host[: min(len(host), raw_end + BS9 // 2)])
    t0 = time.perf_counter()
    z = O.bzip2_compress(sample, LEVEL, threads=threads)
    dt = time.perf_counter() - t0
    bits = int(trace[K].bit_start)
    nbytes, rem = bits // 8, bits % 8
    got = d_out[: nbytes + 1].cpu().numpy()
    exp = np.frombuffer(z, dtype=np.uint8)[: nbytes + 1]
    ok = bool(np.array_equal(got[:nbytes], exp[:nbytes]))
    if rem and ok:
        mask = (0xFF << (8 - rem)) & 0xFF
        ok = (int(got[nbytes]) & mask) == (int(exp[nbytes]) & mask)
    return {"blocks": K, "bits": bits, "ok": ok, "oracle_s": round(dt, 2), "oracle_threads": threads,
            "what": "oracle/bz2_oracle.c output on the first %d raw bytes vs the first %d bits of the benchmarked stream" % (sample.size, bits)}


def decode_arm(L, _native, torch, d_comp, comp, d_ref, nbytes, steps, pinned_comp=None):
    """Decode of a stream: resident (b2_bzip2_decompress_dev) and end to end (b2_bzip2_decompress, pinned host in,
    library-pinned out), round trip checked against d_ref."""
    d_dec = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    dn = C.c_size_t()
    _check(L.b2_bzip2_decompress_dev(d_comp.data_ptr(), comp, 0, d_dec.data_ptr(), nbytes, C.byref(dn)), "decompress_dev", _native)
    dms, dst = 0.0, None
    for _ in range(steps):
        _check(L.b2_bzip2_decompress_dev(d_comp.data_ptr(), comp, 0, d_dec.data_ptr(), nbytes, C.byref(dn)), "decompress_dev", _native)
        dst = _native.stats()
        dms += dst["ms_total"]
    ok = dn.value == nbytes and bool(torch.equal(d_dec[: dn.value], d_ref))
    res = {"metric": "bzip2_-9_decode_MBps", "value": nbytes * steps / (dms / 1e3) / 1e6, "unit": "MB/s", "steps": steps,
           "roundtrip_ok": ok, "ms_per_step": dms / steps,
           "stages_ms": {k: dst[k] for k in ("ms_scan", "ms_hdec", "ms_unmtf", "ms_ibwt", "ms_unrle")}}
    # SURVEY.md 8(d): c + 4n (dbuf) + 8n (T-vector build) + 4n (chase) + N_raw out
    alg = comp + 16 * nbytes + nbytes
    peak, _ = peaks()
    dom = max(res["stages_ms"].items(), key=lambda kv: kv[1])
    res["roofline"] = {"bound": "hbm", "achieved": alg / 1e9 / (dms / steps / 1e3), "peak": peak, "unit": "GB/s",
                       "frac": alg / 1e9 / (dms / steps / 1e3) / peak, "algorithmic_bytes": alg, "dominant_stage": dom[0],
                       "dominant_stage_ms": dom[1], "note": "whole decode, algorithmic bytes of SURVEY.md 8(d): c + 16 n + N"}
    if pinned_comp is not None:
        out, n = C.POINTER(C.c_uint8)(), C.c_size_t()
        _check(L.b2_bzip2_decompress(pinned_comp.data_ptr(), comp, 0, C.byref(out), C.byref(n)), "decompress", _native)
        L.b2_free(out)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            _check(L.b2_bzip2_decompress(pinned_comp.data_ptr(), comp, 0, C.byref(out), C.byref(n)), "decompress", _native)
            if n.value != nbytes:
                raise SystemExit("e2e decode returned %d bytes" % n.value)
            L.b2_free(out)
        dt = time.perf_counter() - t0
        res["e2e"] = {"value": nbytes * steps / dt / 1e6, "unit": "MB/s", "h2d_bytes_per_step": comp, "d2h_bytes_per_step": nbytes,
                      "api": "b2_bzip2_decompress (host pinned in, library-pinned out)"}
    return res


def config3_leg(L, _native, torch, steps):
    """BASELINE configs[2]: 100 MB enwik-shaped text, bzip2 -9 encode + decode on this GPU."""
    from tools.workloads import enwik_like
    t0 = time.perf_counter()
    data = enwik_like(100000000)
    gen_s = time.perf_counter() - t0
    n = data.size
    pinned = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    pinned.numpy()[:] = data
    d_in = pinned.cuda()
    cap = L.b2_bzip2_bound(n)
    d_out = torch.empty(cap, dtype=torch.uint8, device="cuda")
    out_n = C.c_size_t()
    for _ in range(2):
        _check(L.b2_bzip2_compress_dev(d_in.data_ptr(), n, LEVEL, d_out.data_ptr(), cap, C.byref(out_n)), "compress_dev", _native)
    ems, st, agg = 0.0, None, {}
    for _ in range(steps):
        _check(L.b2_bzip2_compress_dev(d_in.data_ptr(), n, LEVEL, d_out.data_ptr(), cap, C.byref(out_n)), "compress_dev", _native)
        st = _native.stats()
        ems += st["ms_total"]
        for k, v in st.items():
            agg[k] = agg.get(k, 0) + v
    comp = out_n.value
    # end to end encode
    out, nn = C.POINTER(C.c_uint8)(), C.c_size_t()
    _check(L.b2_bzip2_compress(pinned.data_ptr(), n, LEVEL, C.byref(out), C.byref(nn)), "compress", _native)
    pinned_comp = torch.empty(nn.value, dtype=torch.uint8, pin_memory=True)
    pinned_comp.numpy()[:] = np.ctypeslib.as_array(out, (nn.value,))
    L.b2_free(out)
    t1 = time.perf_counter()
    for _ in range(steps):
        _check(L.b2_bzip2_compress(pinned.data_ptr(), n, LEVEL, C.byref(out), C.byref(nn)), "compress", _native)
        L.b2_free(out)
    e2e_s = (time.perf_counter() - t1) / steps
    dec = decode_arm(L, _native, torch, d_out, comp, d_in, n, steps, pinned_comp)
    peak, _ = peaks()
    bwt_gbs = (agg["bwt_bytes"] / 1e9) / (agg["ms_bwt"] / 1e3) if agg.get("ms_bwt") else 0.0
    enc_ms, dec_ms = ems / steps, dec["ms_per_step"]
    return {"workload": "100 000 000 B enwik-shaped text (order-3 chain trained on the reference's test/sample5.ref + 1 %% long repeats, seed %d), bzip2 -9" % SEED,
            "encode_MBps": n / (enc_ms / 1e3) / 1e6, "decode_MBps": dec["value"], "encode_plus_decode_MBps": n / ((enc_ms + dec_ms) / 1e3) / 1e6,
            "encode_e2e_MBps": n / e2e_s / 1e6, "decode_e2e_MBps": (dec.get("e2e") or {}).get("value"),
            "encode_ms": enc_ms, "decode_ms": dec_ms, "compressed_bytes": comp, "blocks": int(agg["blocks"] // steps), "roundtrip_ok": dec["roundtrip_ok"],
            "bwt_stage": {"achieved": bwt_gbs, "frac": bwt_gbs / peak, "rounds": int(st["bwt_rounds"]), "ms_per_step": agg["ms_bwt"] / steps,
                          "path": "LSD radix passes + prefix doubling (text mode)"},
            "encode_stages_ms": {k: agg[k] / steps for k in ("ms_rle1", "ms_bwt", "ms_mtf", "ms_huff", "ms_pack")},
            "decode_stages_ms": dec["stages_ms"], "generator_s": round(gen_s, 1)}


def bwtc_leg(L, _native, torch, host, mb, check_blocks):
    """BASELINE configs[3]: BWTC -9 (range-coder back end) on the config-2 buffer, one GPU."""
    n = min(len(host), mb << 20)
    src = np.ascontiguousarray(host[:n])
    out, nn = C.POINTER(C.c_uint8)(), C.c_size_t()
    t0 = time.perf_counter()
    _check(L.b2_bwtc_compress(src.ctypes.data, n, 9, C.byref(out), C.byref(nn)), "bwtc_compress", _native)
    dt = time.perf_counter() - t0
    st = _native.stats()
    z = bytes(np.ctypeslib.as_array(out, (nn.value,)))
    L.b2_free(out)
    res = {"workload": "BWTC -9 on the first %d MiB of the config-2 buffer (b2_bwtc_compress, host buffers)" % (n >> 20), "bytes": n,
           "encode_MBps": n / dt / 1e6, "wall_s": round(dt, 3), "compressed_bytes": nn.value, "ms_total_gpu": st["ms_total"],
           "stages_ms": {"bwt": st["ms_bwt"], "mtf": st["ms_mtf"], "model": st["ms_huff"], "coder": st["ms_pack"]},
           "note": "model = one warp per block (Fenwick tree in shared memory; blocks in parallel); coder = ONE serial recurrence per file (one warp, lane 0 carries it): stages_ms.coder bounds the path"}
    if check_blocks:
        from oracle import oracle as O
        k = min(n, check_blocks * 900000)
        exp = O.bwtc_compress(src[:k].tobytes(), 9)
        o2, n2 = C.POINTER(C.c_uint8)(), C.c_size_t()
        _check(L.b2_bwtc_compress(src.ctypes.data, k, 9, C.byref(o2), C.byref(n2)), "bwtc_compress", _native)
        res["parity_blocks"] = check_blocks
        res["parity_ok"] = bytes(np.ctypeslib.as_array(o2, (n2.value,))) == exp
        L.b2_free(o2)
    # decode (one serial thread: model and coder cannot be separated) on a small sample of the same buffer
    dn = min(n, 2 << 20)
    _check(L.b2_bwtc_compress(src.ctypes.data, dn, 9, C.byref(out), C.byref(nn)), "bwtc_compress", _native)
    zs = np.ctypeslib.as_array(out, (nn.value,)).copy()
    L.b2_free(out)
    t1 = time.perf_counter()
    _check(L.b2_bwtc_decompress(zs.ctypes.data, zs.size, C.byref(out), C.byref(nn)), "bwtc_decompress", _native)
    res["decode_MBps"] = dn / (time.perf_counter() - t1) / 1e6
    res["decode_sample_bytes"] = dn
    res["roundtrip_ok"] = bool(nn.value == dn and np.array_equal(np.ctypeslib.as_array(out, (nn.value,)), src[:dn]))
    L.b2_free(out)
    return res


def dump_outputs(path, d_stream, n):
    """The .bz2 stream of the last timed step (first n bytes of the CUDA tensor d_stream) as .npy files under `path`:
    its length, its first MiB and last 64 KiB (header, first blocks, last block, stream CRC) and its bytes at up to
    4 Mi positions drawn with PCG64(SEED) (every position of a shorter stream), with those positions.  Byte values are
    float32, the length and positions float64 (exact below 2**53): about 52 MB in all.  The same arguments give the
    same input, so two builds are compared file by file."""
    import torch
    os.makedirs(path, exist_ok=True)
    s = d_stream[:n]
    if n <= DUMP_SAMPLE:
        idx = np.arange(n)
    else:
        idx = np.unique(np.random.Generator(np.random.PCG64(SEED)).integers(0, n, size=DUMP_SAMPLE))
    arrays = {
        "stream_length": np.array([n], dtype=np.float64),
        "stream_head": s[:DUMP_HEAD].cpu().numpy().astype(np.float32),
        "stream_tail": s[max(0, n - DUMP_TAIL):].cpu().numpy().astype(np.float32),
        "stream_sample_index": idx.astype(np.float64),
        "stream_sample": s[torch.from_numpy(idx).to(s.device)].cpu().numpy().astype(np.float32),
    }
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--mb", type=int, default=int(os.environ.get("B2_BENCH_MB", "1024")), help="MiB of input per GPU and step")
    ap.add_argument("--no-cpu", action="store_true", help="skip every leg that runs the CPU oracle (cpu_baseline, parity)")
    ap.add_argument("--no-extra", action="store_true", help="skip the config3 and bwtc legs")
    ap.add_argument("--bwtc-mb", type=int, default=int(os.environ.get("B2_BENCH_BWTC_MB", "64")), help="MiB of the config-2 buffer for the BWTC leg (config 4 = 1024)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the stream of the last timed step (sampled) to DIR/*.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from compressjs_b200 import _native

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        import datetime
        # a mismatched collective must fail fast, not sit out the default 10 minute watchdog on N GPUs
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=180))
    L = _native.lib()
    rc = L.b2_init(local)
    if rc:
        raise SystemExit("b2_init: " + _native.last_error())

    shard = args.mb << 20
    nbytes = shard * world
    HALO = 4 << 20
    # weak scaling: the job is ONE stream of world x shard bytes.  One GPU: the whole input.  Several: every rank
    # holds (and uploads) only its own share plus a halo of the next share; the ranks exchange share summaries, cut
    # and encode their blocks; the finished fragments stay on their GPUs at their final bit positions (value), travel
    # over NCCL straight into place on rank 0 (gathered) or into one shared host buffer (e2e) -- sharded.py.
    if world == 1:
        host = gen_ascii(shard, SEED)
    else:
        own = gen_ascii(shard, SEED + rank)
        host = np.concatenate([own, gen_ascii(min(HALO, shard), SEED + rank + 1)]) if rank + 1 < world else own  # the generator is prefix consistent
    pinned = torch.empty(host.size, dtype=torch.uint8, pin_memory=True)
    pinned.numpy()[:] = host
    d_in = pinned.cuda(non_blocking=False)
    cap = L.b2_bzip2_bound(nbytes)
    d_out = torch.empty(cap, dtype=torch.uint8, device="cuda") if world == 1 else None
    out_n = C.c_size_t()
    from compressjs_b200 import sharded as SH
    state = {"comp": 0, "out": None}

    def step_resident():
        if world == 1:
            _check(L.b2_bzip2_compress_dev(d_in.data_ptr(), nbytes, LEVEL, d_out.data_ptr(), cap, C.byref(out_n)), "compress_dev", _native)
            state["comp"] = out_n.value
            return _native.stats()
        # the stream stays sharded like the input: every rank ends with its fragment at its final bit position
        ss = SH.compress_shares(d_in, shard, LEVEL, keep_sharded=True)
        st = _native.stats()
        state["ss"] = ss
        state["comp"] = ss.total_bytes
        return st

    def step_gathered():
        # the same step followed by the NVLink gather of the pieces into one buffer on rank 0
        out = SH.compress_shares(d_in, shard, LEVEL, keep_sharded=True).gather()
        if out is not None:
            state["out"] = out

    def step_e2e(check=False):
        if world == 1:
            out, n = C.POINTER(C.c_uint8)(), C.c_size_t()
            _check(L.b2_bzip2_compress(pinned.data_ptr(), nbytes, LEVEL, C.byref(out), C.byref(n)), "compress", _native)
            st = _native.stats()
            if check:  # untimed warm-up call: the host-buffer path must produce the resident path's stream
                got = torch.from_numpy(np.ctypeslib.as_array(out, (n.value,))).cuda()
                if n.value != state["comp"] or not torch.equal(got, d_out[:n.value]):
                    raise SystemExit("e2e stream differs from the HBM-resident stream")
            L.b2_free(out)
            return st, n.value
        if state.get("shm") is None:                # once: a pinned host buffer mapped by all ranks of the box
            state["shm"] = SH.SharedHostBuffer(cap)
        d = pinned.cuda(non_blocking=True)          # H2D of the step's input: the own share + halo only
        torch.cuda.current_stream().synchronize()   # the library works on its own stream
        # every rank downloads its fragment over its own PCIe link straight into place in the shared host buffer
        nn = SH.compress_shares(d, shard, LEVEL, host_out=state["shm"].tensor) or 0
        if check and rank == 0:
            got = state["shm"].tensor[:nn].cuda()
            if nn != state["comp"] or not torch.equal(got, state["out"][:nn]):
                raise SystemExit("e2e stream (host buffer) differs from the HBM-resident stream")
        return _native.stats(), nn

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident (HBM) arm ----
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step_resident()
    barrier()
    t0 = time.perf_counter()
    agg = {}
    dev_ms = 0.0
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        st = step_resident()
        dev_ms += st["ms_total"]
        for k, v in st.items():
            agg[k] = agg.get(k, 0) + v
    ev1.record()
    barrier()
    wall = time.perf_counter() - t0
    if world > 1:
        dev_ms = ev0.elapsed_time(ev1)  # includes the summary / size exchanges and the shift to the final bit position
    clocks = sampler.stop(t0, t0 + wall) if rank == 0 else None
    comp_bytes = state["comp"]
    trace = _native.last_trace() if world == 1 else []
    if args.dump_outputs:
        if world == 1:
            dump_outputs(args.dump_outputs, d_out, comp_bytes)
        else:
            full = state["ss"].gather()   # collective: the last timed step's stream, assembled on rank 0
            if rank == 0:
                dump_outputs(args.dump_outputs, full, full.numel())
            del full

    # device time: max over ranks (events on the library's launching stream)
    t = torch.tensor([dev_ms, wall * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max, wall_ms_max = t.tolist()

    # ---- the same step with the pieces gathered on rank 0 (secondary figure; also feeds the parity check below) ----
    gathered_ms = None
    if world > 1:
        step_gathered()
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        gsteps = max(1, min(args.steps, 3))
        for _ in range(gsteps):
            step_gathered()
        g1.record()
        barrier()
        tg = torch.tensor([g0.elapsed_time(g1) / gsteps], dtype=torch.float64, device="cuda")
        dist.all_reduce(tg, op=dist.ReduceOp.MAX)
        gathered_ms = float(tg.item())

    # ---- multi-rank parity: the stream assembled from the ranks' fragments == the one-GPU stream of the same input ----
    sharded_parity = None
    d_full = None
    if world > 1 and rank == 0:
        full = np.concatenate([gen_ascii(shard, SEED + r) for r in range(world)])
        d_full = torch.from_numpy(full).cuda()
        del full
        one = torch.empty(cap, dtype=torch.uint8, device="cuda")
        _check(L.b2_bzip2_compress_dev(d_full.data_ptr(), nbytes, LEVEL, one.data_ptr(), cap, C.byref(out_n)), "compress_dev", _native)
        same = out_n.value == state["out"].numel() and bool(torch.equal(one[: out_n.value], state["out"]))
        sharded_parity = {"ok": same, "bytes": int(out_n.value),
                          "sha256_16": hashlib.sha256(state["out"].cpu().numpy().tobytes()).hexdigest()[:16],
                          "what": "%d-rank stream (sharded input, fragments placed over NCCL) vs b2_bzip2_compress_dev of the whole input on rank 0" % world}
        del one
        if not same:
            print(json.dumps({"error": "sharded stream differs from the single-GPU stream", "sharded_parity": sharded_parity}))
            raise SystemExit(3)

    # ---- e2e arm: host buffers through the C ABI ----
    e2e_steps = max(1, min(args.steps, 3))
    step_e2e(check=True)
    barrier()
    t1 = time.perf_counter()
    e2e_comp = 0
    for _ in range(e2e_steps):
        _, e2e_comp = step_e2e()
    barrier()
    e2e_wall = time.perf_counter() - t1
    t = torch.tensor([e2e_wall], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_wall = t.item()

    # ---- several GPUs: sharded decode of the stream just produced (BASELINE configs[4] style: every rank holds the
    # compressed stream, decodes its share of the blocks, the decoded shards meet on rank 0) ----
    sharded_decode = None
    if world > 1:
        szt = torch.tensor([state["comp"] if rank == 0 else 0], dtype=torch.int64, device="cuda")
        dist.broadcast(szt, 0)
        comp = int(szt.item())
        d_comp = state["out"][:comp].contiguous() if rank == 0 else torch.empty(comp, dtype=torch.uint8, device="cuda")
        dist.broadcast(d_comp, 0)
        torch.cuda.synchronize()
        dsteps = max(1, min(args.steps, 3))
        res = SH.decompress_file_sharded(d_comp)      # warm-up + round trip
        ok = None
        if rank == 0:
            ok = res.numel() == nbytes and bool(torch.equal(res, d_full))
        del res
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(dsteps):
            res = SH.decompress_file_sharded(d_comp)
            del res
        e1.record()
        barrier()
        tt = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        sharded_decode = {"metric": "bzip2_-9_decode_MBps", "value": nbytes * dsteps / (tt.item() / 1e3) / 1e6, "unit": "MB/s", "steps": dsteps,
                          "ms_per_step": tt.item() / dsteps, "roundtrip_ok": ok, "compressed_bytes": comp,
                          "what": "decompress_file_sharded: %d ranks, %d MiB raw per rank, decoded stream assembled on rank 0" % (world, args.mb)}
        del d_comp
    if rank == 0:
        total_raw = nbytes
        value = total_raw * args.steps / (dev_ms_max / 1e3) / 1e6
        peak, peak_src = peaks()
        bwt_gbs = (agg["bwt_bytes"] / 1e9) / (agg["ms_bwt"] / 1e3) if agg.get("ms_bwt") else 0.0
        tr = traffic_from_profiles() or {}
        msd = agg.get("msd_launches", 0) > 0
        if msd:
            nl = agg["msd_launches"]
            kb, ks = agg["msd_bucket_bytes"] / nl, agg["msd_scatter_bytes"] / nl
            mb_ms, ms_ms = agg["ms_msd_bucket"] / nl, agg["ms_msd_scatter"] / nl
            bucket_gbs, scatter_gbs = kb / 1e9 / (mb_ms / 1e3), ks / 1e9 / (ms_ms / 1e3)
            recs = kb / 9.0
            roof = {"bound": "hbm", "kernel": "k_msd_bucket (shared-memory bucket sort of the forward BWT: records in, BWT column out)",
                    "achieved": bucket_gbs, "peak": peak, "unit": "GB/s", "frac": bucket_gbs / peak,
                    "traffic": (tr.get("k_msd_bucket_dram_bytes_per_record") or 0) * recs or None, "traffic_source": tr.get("source"),
                    "peak_source": peak_src, "launches": int(nl), "algorithmic_bytes_per_launch": kb, "avg_launch_ms": mb_ms,
                    "algorithmic_bytes_per_unit": "9 per text byte (8-byte record read, 1 byte of the column written)",
                    "k_msd_scatter": {"achieved": scatter_gbs, "frac": scatter_gbs / peak, "algorithmic_bytes_per_launch": ks, "avg_launch_ms": ms_ms,
                                      "traffic": (tr.get("k_msd_scatter_dram_bytes_per_record") or 0) * recs or None,
                                      "algorithmic_bytes_per_unit": "9 per text byte (1 read, 8-byte record written)"}}
        else:
            radix_gbs = (agg["radix_bytes"] / 1e9) / (agg["ms_radix"] / 1e3) if agg.get("ms_radix") else 0.0
            roof = {"bound": "hbm", "kernel": "k_radix_pass (BWT onesweep pass)", "achieved": radix_gbs, "peak": peak, "unit": "GB/s",
                    "frac": radix_gbs / peak if peak else None, "traffic": None, "peak_source": peak_src, "launches": int(agg["radix_launches"]),
                    "algorithmic_bytes_per_launch": agg["radix_bytes"] / max(agg["radix_launches"], 1),
                    "avg_launch_ms": agg["ms_radix"] / max(agg["radix_launches"], 1)}
        # the survey's formula for an LSD prefix-doubling sort, B = N (91 + 224 R), as an equivalent rate next to the executed bytes
        rounds = int(agg["bwt_rounds"] // max(args.steps, 1))
        lsd_equiv = total_raw / world * args.steps * (91 + 224 * rounds) / 1e9 / (agg["ms_bwt"] / 1e3) if agg.get("ms_bwt") else 0.0
        roof["bwt_stage"] = {"achieved": bwt_gbs, "frac": bwt_gbs / peak if peak else None, "rounds": rounds, "ms_per_step": agg["ms_bwt"] / args.steps,
                             "algorithmic_bytes_per_step": agg["bwt_bytes"] / args.steps,
                             "bytes_per_text_byte": agg["bwt_bytes"] / args.steps / (total_raw / world),
                             "lsd_formula_equivalent_gbs": lsd_equiv, "lsd_formula_equivalent_frac": lsd_equiv / peak,
                             "note": "achieved counts the bytes of the passes actually executed (SURVEY.md 8d); the *_equivalent figures apply the survey's "
                                     "91 N + 224 N R formula of a 4-pass LSD sort to the same time"}
        line = {
            "metric": METRIC, "value": value, "unit": "MB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "config": {"workload": "%d MiB synthetic ASCII per GPU (PCG64 seed %d+rank), bzip2 -9 (900k blocks) encode" % (args.mb, SEED),
                       "level": LEVEL, "bytes_per_gpu": shard, "total_bytes": nbytes, "blocks_per_gpu": int(agg["blocks"] // max(args.steps, 1)),
                       "l2": "inputs (%d MiB) larger than L2 (126 MB); no flush needed" % args.mb, "bwt_batch_blocks": int(os.environ.get("B2_BWT_BATCH", "296")),
                       "compressed_bytes": comp_bytes, "wall_ms_per_step": wall_ms_max / args.steps},
            "e2e": {"value": total_raw * e2e_steps / e2e_wall / 1e6, "unit": "MB/s", "h2d_bytes_per_step": nbytes if world == 1 else nbytes + (world - 1) * HALO, "d2h_bytes_per_step": e2e_comp,
                    "steps": e2e_steps, "api": "b2_bzip2_compress (host pinned in, library-pinned out; upload in 64 MiB chunks and download per batch overlapped with the encode)" if world == 1 else
                    "sharded.compress_shares (every rank uploads its share + a 4 MiB halo from pinned host memory and downloads its fragment into its place in one page-locked host buffer shared by the ranks)"},
            "gpu_launches": int(agg["kernel_launches"]),
            "roofline": roof,
            "stages_ms_per_step": {k: agg[k] / args.steps for k in ("ms_rle1", "ms_bwt", "ms_mtf", "ms_huff", "ms_pack", "ms_radix", "ms_msd_scatter", "ms_msd_bucket")},
            "clocks": clocks,
        }
        if world > 1:
            line["sharded_phases_ms_last_step_rank0"] = {k: round(v, 2) for k, v in SH.PHASES.items()}
            line["sharded_parity"] = sharded_parity
            line["config"]["output"] = ("the finished stream stays sharded in HBM like the input: every rank holds its fragment at its final bit "
                                        "position (sharded.ShardedStream); 'gathered' repeats the step with the pieces moved to rank 0 over NVLink, "
                                        "e2e assembles them in one host buffer")
            line["gathered"] = {"value": total_raw / (gathered_ms / 1e3) / 1e6, "unit": "MB/s", "ms_per_step": gathered_ms,
                                "what": "value's step + ShardedStream.gather(): one contiguous .bz2 in rank 0's HBM"}
            line["decode"] = sharded_decode
        if world == 1:
            if not args.no_cpu:
                line["parity"] = prefix_parity(L, _native, host, d_out, comp_bytes, trace, 32, max(1, min(host_cores(), 32)))
                if line["parity"]["ok"] is False:
                    print(json.dumps({"error": "benchmarked stream differs from the oracle", "parity": line["parity"]}))
                    raise SystemExit(3)
            # decode leg: the stream just produced -- the second half of the metric
            pinned_comp = torch.empty(comp_bytes, dtype=torch.uint8, pin_memory=True)
            pinned_comp.copy_(d_out[:comp_bytes])
            line["decode"] = decode_arm(L, _native, torch, d_out, comp_bytes, d_in, nbytes, max(1, min(args.steps, 3)), pinned_comp)
            del pinned_comp
            if not args.no_extra:
                del d_out
                torch.cuda.empty_cache()
                # the extra legs must never cost the headline line: a failure is reported in place
                try:
                    line["config3"] = config3_leg(L, _native, torch, max(1, min(args.steps, 3)))
                except (Exception, SystemExit) as e:
                    line["config3"] = {"error": repr(e)}
                try:
                    line["bwtc"] = bwtc_leg(L, _native, torch, host, args.bwtc_mb, 0 if args.no_cpu else 2)
                except (Exception, SystemExit) as e:
                    line["bwtc"] = {"error": repr(e)}
        if not args.no_cpu and world == 1:
            from oracle import oracle as O
            O.build()
            sample = np.ascontiguousarray(host[: min(len(host), 8 * BS9)])
            tc = time.perf_counter()
            zc = O.bzip2_compress(sample, LEVEL)
            dtc = time.perf_counter() - tc
            line["cpu_baseline"] = {"value": sample.size / dtc / 1e6, "unit": "MB/s", "cores": 1, "kind": "port",
                                    "sample": "first 8 x 900k blocks (%d bytes) of the same workload, oracle/bz2_oracle.c, 1 thread" % sample.size,
                                    "compressed_bytes": len(zc)}
            # yardsticks SURVEY.md section 8(d) asks for next to the port: libbz2 1.0.8 on one core (a different, much
            # cheaper table search: NOT bit-compatible) and the reference's own published single-thread figure
            import bz2
            tl = time.perf_counter()
            zl = bz2.compress(sample.tobytes(), LEVEL)
            line["cpu_baseline"]["libbz2_1thread_MBps"] = sample.size / (time.perf_counter() - tl) / 1e6
            line["cpu_baseline"]["libbz2_compressed_bytes"] = len(zl)
            line["cpu_baseline"]["reference_js_published_MBps"] = 0.0936   # README.md:70 of the reference (enwik8, node 0.8, 2013 laptop)
        print(json.dumps(line))
    if state.get("shm") is not None:
        state["shm"].close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
