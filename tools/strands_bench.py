#!/usr/bin/env python3
"""Both strands on one GPU: the strand-doubling kernel and the BWA-SMEM run_ascii step with strands=1 and strands=2.

    python tools/strands_bench.py [--ref-bases N] [--reads N] [--steps 5] [--parity 20000] [--out FILE]

Workload: bench.py's configs[3] reference (1 Gbp, numpy PCG64(1000)) and 50 M reads of 151 bp with 1 % substitutions. The odd
reads are drawn from the reverse strand: the window is reverse-complemented before it is mutated.

Reported, all from one run:
  (a) gsm_reads_both_strands_device alone on the device-packed batch: ms and GB/s of packed bytes moved (in + 2 x in);
  (b) PipelinedEngine.run_ascii (raw ASCII in pinned memory, BWA-SMEM, min_len 1) with strands=1 and with strands=2, timed
      alternately in the same process: ms per step and reads/s;
  counts (not timed): of the reverse-drawn reads, the fraction whose longest record is at least 100 bases, and the fraction
      whose longest record has a hit at the read's true origin, for both settings;
  parity: both slots of the first --parity reads against the C oracle (the reference's get_SMEMS restated), dict semantics.
Times: CUDA events, mean of --steps runs after one warm-up.  The card's name and power limit are printed beside the numbers.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

L = 151


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:        # the numbers still stand; say that the card could not be read
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def make_reads(ref_dev, n_reads, seed, sub_rate=0.01, chunk=1_000_000):
    """(n_reads, L) ASCII bytes on the device and the 0-based origin of each read; odd reads from the reverse strand."""
    import torch
    dev = ref_dev.device
    gen = torch.Generator(device=dev).manual_seed(seed)
    asc = torch.empty((n_reads, L), dtype=torch.uint8, device=dev)
    starts = torch.randint(0, ref_dev.numel() - L + 1, (n_reads,), generator=gen, device=dev)
    ar = torch.arange(L, device=dev)
    lut = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device=dev)
    for a in range(0, n_reads, chunk):
        b = min(n_reads, a + chunk)
        r = ref_dev[starts[a:b, None] + ar[None, :]]
        rev = (torch.arange(a, b, device=dev) & 1).bool()
        r[rev] = 3 - r[rev].flip(1)
        mut = torch.rand(r.shape, generator=gen, device=dev) < sub_rate
        shift = torch.randint(1, 4, r.shape, generator=gen, device=dev, dtype=torch.uint8)
        r = torch.where(mut, (r + shift) & 3, r)
        asc[a:b] = lut[r.long()]
    return asc, starts


def longest(res, per_read_slots):
    """Per read: (index of its longest record -- the first one on ties --, that record's length)."""
    import numpy as np
    offs = res.offsets[::per_read_slots]
    ln = res.records["qend"].astype(np.int32) - res.records["qstart"].astype(np.int32)
    cnt = np.diff(offs)
    assert (cnt > 0).all(), "every read has a record with min_len 1"
    mx = np.maximum.reduceat(ln, offs[:-1])
    read = np.repeat(np.arange(len(cnt)), cnt)
    cand = np.flatnonzero(ln == mx[read])
    _, first = np.unique(read[cand], return_index=True)
    return cand[first], mx


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref-bases", type=int, default=1_000_000_000)
    ap.add_argument("--reads", type=int, default=50_000_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--chunks", type=int, default=8, help="chunks of the pipelined path")
    ap.add_argument("--parity", type=int, default=20_000, help="reads whose two slots are checked against the C oracle")
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()

    import numpy as np
    import torch
    import bench
    import genie_smem_b200 as g
    from genie_smem_b200 import _capi as capi
    assert torch.cuda.is_available(), "strands_bench.py needs a CUDA device (no CPU fallback)"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    stream = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)      # noqa: E731

    def timed(fn, steps):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    # ---- workload
    t0 = time.time()
    ref = bench.make_reference(args.ref_bases, 1000)
    ref_dev = torch.from_numpy(ref).to(dev)
    index = g.DeviceIndex.build_on_device(ref_dev, dev).build_seed_table()
    asc_dev, starts_dev = make_reads(ref_dev, args.reads, 1001)
    del ref_dev
    n = args.reads
    log(f"index + reads: {time.time() - t0:.1f} s")

    # ---- (a) the doubling kernel alone, on the device-packed batch
    batch = g.ReadBatch.from_device_bases(asc_dev, ascii=True)
    cpr = (L + 63) // 64
    in_bytes = n * cpr * 16
    out_p = torch.empty(2 * in_bytes + 16, dtype=torch.uint8, device=dev)
    out_c = torch.empty(2 * n + 1, dtype=torch.int32, device=dev)
    out_l = torch.empty(2 * n, dtype=torch.int32, device=dev)
    rc_ = batch.cstruct()

    def double():
        capi.check(capi.lib.gsm_reads_both_strands_device(C.byref(rc_), out_p.data_ptr(), out_c.data_ptr(), out_l.data_ptr(), stream()))
    ms_double = timed(double, max(args.steps, 20))
    moved = 3 * in_bytes
    # the doubled batch equals what both_strands() builds (same entry point) and its first read pair equals the host packer
    pair = g.ReadBatch.from_strings([bytes(asc_dev[0].cpu().numpy()).decode(),
                                     bytes(asc_dev[0].cpu().numpy()).decode()[::-1].translate(str.maketrans("ACGT", "TGCA"))])
    assert np.array_equal(out_p[: 2 * cpr * 16].cpu().numpy(), pair.packed_host[: 2 * cpr * 16]), "doubled batch != host packer"
    del batch, out_p, out_c, out_l
    torch.cuda.empty_cache()

    # ---- (b) run_ascii with strands=1 and strands=2, alternating
    asc = torch.empty((n, L), dtype=torch.uint8, pin_memory=True)
    asc.copy_(asc_dev)
    starts = starts_dev.cpu().numpy()
    del asc_dev, starts_dev
    torch.cuda.empty_cache()
    caps = dict(mems_per_read=64, recs_per_read=32)            # per slot; a reverse-complement slot of a forward read
    pipes = {s: g.PipelinedEngine(index, n, L, n_chunks=args.chunks, strands=s, **caps) for s in (1, 2)}      # holds chance matches

    def step(s):
        return pipes[s].run_ascii(g.METHOD_BWA, asc, L, min_len=1, reuse_host_buffers=True)
    for s in (1, 2):
        step(s)
    ev = {s: [] for s in (1, 2)}
    wall = {s: [] for s in (1, 2)}
    res = {}
    for _ in range(args.steps):
        for s in (1, 2):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t = time.perf_counter()
            e0.record()
            res[s] = step(s)
            e1.record()
            torch.cuda.synchronize()
            wall[s].append((time.perf_counter() - t) * 1e3)
            ev[s].append(e0.elapsed_time(e1))
    ms = {s: float(np.mean(ev[s])) for s in (1, 2)}
    log(f"doubling {ms_double:.3f} ms; run_ascii strands=1 {ms[1]:.1f} ms, strands=2 {ms[2]:.1f} ms")

    # ---- counts: reverse-drawn reads, longest record >= 100 bases, and its hit at the true origin
    rev = np.arange(n) % 2 == 1
    counts = {}
    for s in (1, 2):
        r = res[s]
        k, mx = longest(r, s)
        sel = k[rev]
        recs = r.records[sel].copy()
        hits = g.locate_hits(index, recs, max_occ=500)
        want = starts[rev].astype(np.int64) + recs["qstart"].astype(np.int64)     # in the searched string's coordinates
        hr = hits.hits["record"].astype(np.int64)
        ok = np.zeros(len(sel), bool)
        ok[hr[hits.hits["offset"].astype(np.int64) == want[hr]]] = True
        counts[f"strands{s}"] = {"reverse_reads": int(rev.sum()), "longest_ge_100": float((mx[rev] >= 100).mean()),
                                 "longest_hit_at_origin": float(ok.mean()),
                                 "longest_on_strand1": float((recs["read_id"] & 1).mean()) if s == 2 else 0.0,
                                 "records": int(len(r.records))}
    log(json.dumps(counts))

    # ---- parity: both slots of the first --parity reads against the C oracle
    from oracle.c_oracle import COracle
    m = min(args.parity, n)
    codes = np.frombuffer(asc[:m].numpy().tobytes(), np.uint8).reshape(m, L)
    lut = np.zeros(256, np.uint8)
    lut[list(b"ACGT")] = [0, 1, 2, 3]
    codes = lut[codes]
    inter = np.empty((2 * m, L), np.uint8)
    inter[0::2], inter[1::2] = codes, 3 - codes[:, ::-1]
    text = np.frombuffer(b"ACGT", np.uint8)[ref].tobytes()
    o = COracle(text, index.suffix_array_host())
    out, cnt = o.smems(0, None, min_len=1, joined=np.frombuffer(b"ACGT", np.uint8)[inter.reshape(-1)].tobytes(),
                       lens=np.full(2 * m, L, np.uint32))
    r2 = res[2]
    mism, raises = bench.compare_with_oracle(inter, (r2.records, r2.offsets, r2.status), out, cnt, 2 * m)
    r1 = res[1]
    same = all(np.array_equal(r1.records[r1.offsets[i]:r1.offsets[i + 1]][f], r2.for_read(i, 0)[f])
               for i in range(m) for f in ("qstart", "qend", "sa_lo", "sa_hi"))
    log(f"parity: {mism} mismatching slots of {2 * m}; strand 0 == strands=1: {same}")

    result = {
        "card": card(),
        "workload": {"reference": f"bench.py configs[3] generator, {args.ref_bases} bases, PCG64(1000)",
                     "reads": n, "read_len": L, "substitutions": 0.01, "reverse_strand_reads": "every odd read (window reverse-complemented, then mutated)",
                     "method": "BWA-SMEM, min_len 1", "pipeline": f"PipelinedEngine.run_ascii, {args.chunks} chunks, caps {caps} per slot"},
        "a_doubling_kernel": {"ms": round(ms_double, 4), "packed_bytes_in": in_bytes, "bytes_moved": moved,
                              "GBs": round(moved / (ms_double * 1e-3) / 1e9, 1),
                              "share_of_strands2_step": round(ms_double / ms[2], 5)},
        "b_run_ascii": {f"strands{s}": {"ms": round(ms[s], 2), "ms_each": [round(x, 2) for x in ev[s]], "wall_ms": round(float(np.mean(wall[s])), 2),
                                        "reads_per_s": round(n / (ms[s] * 1e-3)), "slots_per_s": round(s * n / (ms[s] * 1e-3)),
                                        "records": int(len(res[s].records))} for s in (1, 2)},
        "strands2_over_strands1_rate": round(ms[1] / ms[2], 4),
        "counts": counts,
        "parity": {"reads": m, "slots": 2 * m, "mismatching_slots": int(mism), "slots_where_reference_raises": int(raises),
                   "strand0_equals_strands1": bool(same)},
        "steps": args.steps,
    }
    txt = json.dumps(result, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")
    if mism or not same:
        sys.exit(1)


if __name__ == "__main__":
    main()
