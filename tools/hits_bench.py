#!/usr/bin/env python3
"""Hit expansion on one GPU: gsm_hits_count + gsm_hits_locate over the BWA-SMEM records of the configs[3] workload.

    python tools/hits_bench.py [--ref-bases N] [--reads N] [--max-occ 500] [--steps 3] [--out FILE]

Setup: bench.py's synthetic reference (1 Gbp, numpy PCG64(1000)) cut into 25 sequences of 40 Mbp, and the same text as
3,000 sequences and as 20,000 sequences (a start table too large for shared memory); 50 M reads of 151 bp with 1 %
substitutions (bench.py's generator); BWA-SMEM records with min_len 1; max_occ 500, min_len 0.

Reported, all from one run: records, hits, gsm_hits_count ms, gsm_hits_locate ms and hits/s with the full suffix array and
with the sampled one (S = 32, full array unbound), and as the baseline gsm_locate_sampled_batch on the identical row set
(the row of every hit, one thread per row).  Every hit of the full-SA run is checked against positions computed with torch
from the full suffix array, and the sampled-SA hits must equal the full-SA hits.  Times: CUDA events, mean of --steps runs
after one warm-up.  The card's name and power limit are printed beside the numbers.
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref-bases", type=int, default=1_000_000_000)
    ap.add_argument("--reads", type=int, default=50_000_000)
    ap.add_argument("--max-occ", type=int, default=500)
    ap.add_argument("--sample", type=int, default=32)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--tables", default="25,3000,20000", help="sequence counts of the start tables timed")
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()

    import numpy as np
    import torch
    import bench
    import genie_smem_b200 as g
    from genie_smem_b200 import _capi as capi
    assert torch.cuda.is_available(), "hits_bench.py needs a CUDA device (no CPU fallback)"
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

    # ---- workload: bench.py's reference and reads
    t0 = time.time()
    ref = bench.make_reference(args.ref_bases, 1000)
    ref_dev = torch.from_numpy(ref).to(dev)
    index = g.DeviceIndex.build_on_device(ref_dev, dev).build_seed_table()
    codes = torch.empty((args.reads, bench.READ_LEN), dtype=torch.uint8, device=dev)
    bench.device_reads(ref_dev, args.reads, bench.READ_LEN, 1001, codes)
    batch = g.ReadBatch.from_device_bases(codes, bench.READ_LEN)
    del codes, ref_dev
    engine = g.Engine(index, args.reads, bench.READ_LEN, mems_per_read=24, recs_per_read=8)
    engine.launch(g.METHOD_BWA, batch, min_len=1)
    _, n_rec = engine.check_overflow()
    del batch
    engine.mem_pool = engine.rec_tmp = engine.scratch = None
    torch.cuda.empty_cache()
    recs = engine.records[: n_rec * 16]
    log(f"setup {time.time() - t0:.1f} s: {n_rec} records from {args.reads} reads on {args.ref_bases} bases")

    n_bases = index.n_bases
    tables = {}
    for n in (int(x) for x in args.tables.split(",")):
        ct = g.Contigs.from_lengths([f"seq{i}" for i in range(n)], [n_bases // n + (1 if i < n_bases % n else 0) for i in range(n)])
        t = torch.from_numpy(ct.start.view(np.int32).copy()).to(dev)
        tables[n] = (ct, t, capi.DevContigs(n, t.data_ptr()))

    # ---- phase 1
    counts = torch.empty(n_rec, dtype=torch.int32, device=dev)
    off = torch.empty(n_rec + 1, dtype=torch.int64, device=dev)
    tb = C.c_uint64()
    capi.check(capi.lib.gsm_hits_workspace_info(n_rec, C.byref(tb)))
    tmp = torch.empty(int(tb.value), dtype=torch.uint8, device=dev)

    def count():
        capi.check(capi.lib.gsm_hits_count(recs.data_ptr(), n_rec, args.max_occ, 0, counts.data_ptr(), off.data_ptr(), tmp.data_ptr(), int(tb.value), stream()))
    ms_count = timed(count, args.steps)
    total = int(off[-1].item())
    log(f"{total} hits; gsm_hits_count {ms_count:.3f} ms")
    out = torch.empty(total * 4, dtype=torch.int32, device=dev)
    status = torch.zeros(1, dtype=torch.int64, device=dev)

    def locate(table, ssa=None, sample=0):
        capi.check(capi.lib.gsm_hits_locate(C.byref(index.c), C.c_void_p(ssa.data_ptr() if ssa is not None else 0), sample,
                                            C.byref(table[2]), recs.data_ptr(), off.data_ptr(), 0, n_rec, args.max_occ, 0,
                                            out.data_ptr(), total, status.data_ptr(), stream()))

    # ---- expected hits from the full suffix array (torch), and the row of every hit (the baseline's input)
    r32 = recs.view(torch.int32).view(-1, 4)
    lo = r32[:, 2].long() & 0xFFFFFFFF
    cnt = (r32[:, 3].long() & 0xFFFFFFFF) - lo + 1
    ln = ((r32[:, 1].long() & 0xFFFFFFFF) >> 16) - (r32[:, 1].long() & 0xFFFF)
    samp = cnt > args.max_occ
    step = torch.where(samp, cnt // args.max_occ, torch.ones_like(cnt))
    rec_of = torch.repeat_interleave(torch.arange(n_rec, device=dev), counts.long())
    k = torch.arange(total, device=dev) - off[rec_of]
    rows = (lo[rec_of] + k * step[rec_of])
    del k
    pos = (index.sa[rows].long() & 0xFFFFFFFF) - 1
    rows32 = rows.to(torch.int32)
    del rows

    def expect(n_seq):
        st = tables[n_seq][1].long()
        c = torch.searchsorted(st, pos, right=True) - 1
        o = pos - st[c]
        fl = (o + ln[rec_of] > st[c + 1] - st[c]).long() | (samp[rec_of].long() << 1)
        return torch.stack([rec_of, c, o, fl], 1).to(torch.int32).view(-1)

    result = {"card": card(), "workload": {"ref_bases": args.ref_bases, "reads": args.reads, "read_len": bench.READ_LEN, "sub_rate": bench.SUB_RATE,
                                           "records": "BWA-SMEM, min_len 1", "max_occ": args.max_occ, "min_len": 0, "sample": args.sample},
              "records": n_rec, "hits": total, "sampled_records": int(samp.sum().item()), "gsm_hits_count_ms": round(ms_count, 3),
              "steps": args.steps, "full_sa": {}, "sampled_sa": {}}
    checked = 0
    for n_seq, table in tables.items():
        ms = timed(lambda: locate(table), args.steps)
        assert int(status.item()) == 0
        ok = bool(torch.equal(out, expect(n_seq)))
        assert ok, f"full-SA hits differ from the suffix array ({n_seq} sequences)"
        checked = total
        result["full_sa"][f"{n_seq}_sequences"] = {"gsm_hits_locate_ms": round(ms, 3), "hits_per_s": total / (ms * 1e-3)}
        log(f"full SA, {n_seq} sequences: {ms:.3f} ms, {total / (ms * 1e-3) / 1e9:.3f} G hits/s")
    want = {n: expect(n) for n in tables}
    del pos

    # ---- sampled suffix array: the full one unbound
    index.build_sampled_sa(args.sample)
    full_sa = index.sa
    index.sa = None
    index._bind()
    pos_out = torch.empty_like(rows32)

    def baseline():
        capi.check(capi.lib.gsm_locate_sampled_batch(C.byref(index.c), C.c_void_p(index.ssa.data_ptr()), args.sample, total, C.c_void_p(rows32.data_ptr()),
                                                      C.c_void_p(pos_out.data_ptr()), stream()))
    for n_seq, table in tables.items():
        ms_base = timed(baseline, args.steps)
        ms = timed(lambda: locate(table, index.ssa, args.sample), args.steps)
        ms_base2 = timed(baseline, args.steps)                  # before and after: the baseline's spread in this run
        assert int(status.item()) == 0
        assert bool(torch.equal(out, want[n_seq])), f"sampled-SA hits differ from the full-SA hits ({n_seq} sequences)"
        base = min(ms_base, ms_base2)
        result["sampled_sa"][f"{n_seq}_sequences"] = {
            "gsm_hits_locate_ms": round(ms, 3), "hits_per_s": total / (ms * 1e-3),
            "gsm_locate_sampled_batch_ms": [round(ms_base, 3), round(ms_base2, 3)], "baseline_rows_per_s": total / (base * 1e-3),
            "ratio_vs_baseline": round(base / ms, 4)}
        log(f"sampled SA, {n_seq} sequences: {ms:.3f} ms ({total / (ms * 1e-3) / 1e9:.3f} G hits/s); gsm_locate_sampled_batch "
            f"{ms_base:.3f} / {ms_base2:.3f} ms; ratio {base / ms:.3f}")
    ok_base = bool(torch.equal(pos_out, (full_sa[rows32.long()])))
    assert ok_base, "gsm_locate_sampled_batch positions differ from the full suffix array"
    index.sa = full_sa
    index._bind()
    result["hits_checked_against_full_sa"] = checked
    result["note"] = ("hits/s = hits / kernel time; the baseline locates the row of every hit (one 4-byte position per row), "
                      "gsm_hits_locate also finds the hit's record and sequence and writes 16 bytes")
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
