#!/usr/bin/env python3
"""Seed chaining on one GPU: gsm_chain_seeds + gsm_chains_collect over the hits of BWA-SMEM records of both strands.

    python tools/chains_bench.py [--ref-bases N] [--reads N] [--chunk-reads N] [--steps 5] [--out FILE]

Workload: bench.py's synthetic reference (1 Gbp, numpy PCG64(1000)) as 25 sequences of 40 Mbp; 50 M reads of 151 bp with
1 % substitutions drawn with torch on the device, every odd read reverse-complemented (drawn from the reverse strand);
Engine(strands=2) in chunks of --chunk-reads reads, BWA-SMEM records with min_len 1, hits with max_occ 500 and min_len 19
from the full suffix array, chains with w 100 and max_gap 10000.

Timed with CUDA events, per chunk and summed over the batch, mean of --steps passes after one warm-up pass: the device step
(strand doubling + sweep + select + scan + ordered write, gsm_hits_count, gsm_hits_locate) and the chaining kernels
(gsm_chain_seeds + gsm_chains_collect).  Host syncs between the phases (to size buffers) fall outside every timed interval.
Reported: hits, chains, slots on the slow path, chaining ms and hits/s, algorithmic bytes/s (hits read 16 B, chain ids
written 4 B per hit, chains written 32 B each) against the 7.7 TB/s data-sheet HBM bandwidth, chaining's share of the
device step, and the best() placement rate (true strand, sequence and offset) of forward- and reverse-drawn reads that lie
inside one sequence.  The card's name, power limit and max SM clock are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True

HBM_BYTES_PER_S = 7.7e12          # B200 data sheet
FAST_CAP = 8                      # chains per slot on the fast path (csrc/chains.cu)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref-bases", type=int, default=1_000_000_000)
    ap.add_argument("--sequences", type=int, default=25)
    ap.add_argument("--reads", type=int, default=50_000_000)
    ap.add_argument("--chunk-reads", type=int, default=6_250_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    args = ap.parse_args()

    import torch
    import bench
    import genie_smem_b200 as g
    from genie_smem_b200 import _capi as capi
    from hits_bench import card
    assert torch.cuda.is_available(), "chains_bench.py needs a CUDA device (no CPU fallback)"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    stream = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)      # noqa: E731
    P = lambda t: C.c_void_p(t.data_ptr())                                     # noqa: E731
    L = bench.READ_LEN

    # ---- workload
    t0 = time.time()
    ref = bench.make_reference(args.ref_bases, 1000)
    ref_dev = torch.from_numpy(ref).to(dev)
    index = g.DeviceIndex.build_on_device(ref_dev, dev).build_seed_table()
    n_seq = args.sequences
    seq_len = args.ref_bases // n_seq
    lengths = [seq_len] * (n_seq - 1) + [args.ref_bases - seq_len * (n_seq - 1)]
    index.set_contigs(g.Contigs.from_lengths([f"seq{i}" for i in range(n_seq)], lengths))
    gen = torch.Generator(device=dev)
    gen.manual_seed(1001)
    n = args.reads
    starts = torch.randint(0, args.ref_bases - L + 1, (n,), generator=gen, device=dev, dtype=torch.int64)
    ar = torch.arange(L, device=dev, dtype=torch.int64)[None, :]
    batches = []
    for lo in range(0, n, args.chunk_reads):
        hi = min(n, lo + args.chunk_reads)
        r = ref_dev[(starts[lo:hi, None] + ar).view(-1)].view(hi - lo, L)
        mut = torch.rand(r.shape, generator=gen, device=dev) < bench.SUB_RATE
        add = torch.randint(1, 4, r.shape, generator=gen, device=dev, dtype=torch.uint8)
        r = torch.where(mut, (r + add) & 3, r)
        odd = torch.arange(lo, hi, device=dev) % 2 == 1
        r[odd] = 3 - r[odd].flip(1)                                          # every odd read from the reverse strand
        batches.append((lo, hi, g.ReadBatch.from_device_bases(r.contiguous(), L, read_id_base=lo)))
        del r, mut, add
    del ref_dev
    torch.cuda.empty_cache()
    eng = g.Engine(index, args.chunk_reads, L, mems_per_read=64, recs_per_read=32, strands=2)     # per slot: chance matches on the other strand
    log(f"setup {time.time() - t0:.1f} s: {n} reads in {len(batches)} chunks on {args.ref_bases} bases, {n_seq} sequences")

    buf = {}

    def grow(name, nbytes):
        b = buf.get(name)
        if b is None or b.numel() < nbytes:
            b = buf[name] = torch.empty(max(nbytes, 256), dtype=torch.uint8, device=dev)
        return b

    def ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    stats = {"records": 0, "hits": 0, "chains": 0, "slow_slots": 0, "placed": [0, 0], "placeable": [0, 0]}

    def one_pass(collect):
        ms = {"smem": 0.0, "hits": 0.0, "chain": 0.0}
        for lo, hi, batch in batches:
            e0 = ev()
            view = eng._both_strands(batch)
            eng.launch(g.METHOD_BWA, view, min_len=1)
            e1 = ev()
            _, n_rec = eng.check_overflow()
            slots = view.n
            counts = grow("counts", 4 * max(n_rec, 1))
            off = grow("hit_off", 8 * (n_rec + 1))
            tb = C.c_uint64()
            capi.check(capi.lib.gsm_hits_workspace_info(n_rec, C.byref(tb)))
            tmp = grow("tmp", int(tb.value))
            e2 = ev()
            capi.check(capi.lib.gsm_hits_count(P(eng.records), n_rec, 500, 19, P(counts), P(off), P(tmp), int(tb.value), stream()))
            e3 = ev()
            total = int(off[: 8 * (n_rec + 1)].view(torch.int64)[-1].item())
            hits = grow("hits", 16 * max(total, 1))
            status = grow("status", 8)
            status.zero_()
            e4 = ev()
            capi.check(capi.lib.gsm_hits_locate(C.byref(index.c), None, 0, C.byref(index._contigs_c), P(eng.records), P(off), 0, n_rec, 500, 19,
                                                P(hits), total, P(status), stream()))
            e5 = ev()
            ids = grow("ids", 4 * max(total, 1))
            cnt = grow("cnt", 4 * slots)
            coff = grow("coff", 8 * (slots + 1))
            need = C.c_uint64()
            capi.check(capi.lib.gsm_chains_workspace_info(slots, total, C.byref(need)))
            ws = grow("ws", int(need.value))
            e6 = ev()
            capi.check(capi.lib.gsm_chain_seeds(P(eng.records), P(eng.rec_off), slots, P(hits), P(off), total, 100, 10000, P(ids), P(cnt), P(coff),
                                                P(ws), int(need.value), stream()))
            e7 = ev()
            chain_off = coff[: 8 * (slots + 1)].view(torch.int64)
            n_ch = int(chain_off[-1].item())
            out = grow("chains", 32 * max(n_ch, 1))
            e8 = ev()
            capi.check(capi.lib.gsm_chains_collect(P(eng.rec_off), slots, P(off), total, P(coff), P(ws), int(need.value), P(out), n_ch, P(status),
                                                   stream()))
            e9 = ev()
            torch.cuda.synchronize()
            assert int(status[:8].view(torch.int64).item()) == 0
            ms["smem"] += e0.elapsed_time(e1)
            ms["hits"] += e2.elapsed_time(e3) + e4.elapsed_time(e5)
            ms["chain"] += e6.elapsed_time(e7) + e8.elapsed_time(e9)
            if collect:
                stats["records"] += n_rec
                stats["hits"] += total
                stats["chains"] += n_ch
                stats["slow_slots"] += int((chain_off.diff() > FAST_CAP).sum().item())
                ch = out[: 32 * n_ch].view(torch.int32).view(-1, 8).long() & 0xFFFFFFFF
                read = ch[:, 0] >> 1
                m = hi - lo
                wmax = torch.full((m,), -1, dtype=torch.int64, device=dev).scatter_reduce(0, read, ch[:, 5], "amax")
                idx = torch.arange(n_ch, device=dev)
                cand = torch.where(ch[:, 5] == wmax[read], idx, torch.full_like(idx, n_ch))
                best = torch.full((m,), n_ch, dtype=torch.int64, device=dev).scatter_reduce(0, read, cand, "amin")
                p = starts[lo:hi]
                c_true, o_true = p // seq_len, p % seq_len
                c_true = torch.clamp(c_true, max=n_seq - 1)
                o_true = p - c_true * seq_len
                inside = o_true + L <= torch.as_tensor(lengths, device=dev)[c_true]
                strand = torch.arange(lo, hi, device=dev) % 2
                has = best < n_ch
                b = ch[torch.clamp(best, max=max(n_ch - 1, 0))]
                ok = has & ((b[:, 0] & 1) == strand) & (b[:, 1] == c_true) & (b[:, 2] - (b[:, 4] & 0xFFFF) == o_true)
                for s in (0, 1):
                    sel = inside & (strand == s)
                    stats["placeable"][s] += int(sel.sum().item())
                    stats["placed"][s] += int((ok & sel).sum().item())
        return ms

    one_pass(True)                                   # warm-up, and the counts
    runs = [one_pass(False) for _ in range(args.steps)]
    mean = {k: sum(r[k] for r in runs) / len(runs) for k in runs[0]}
    step = mean["smem"] + mean["hits"] + mean["chain"]
    hits, chains = stats["hits"], stats["chains"]
    alg_bytes = 16 * hits + 4 * hits + 32 * chains
    result = {
        "card": card(),
        "workload": {"ref_bases": args.ref_bases, "sequences": n_seq, "reads": n, "read_len": L, "sub_rate": bench.SUB_RATE,
                     "odd_reads": "reverse strand", "engine": f"Engine(strands=2), chunks of {args.chunk_reads} reads",
                     "records": "BWA-SMEM, min_len 1", "max_occ": 500, "min_len": 19, "w": 100, "max_gap": 10000, "suffix_array": "full"},
        "steps": args.steps, "records": stats["records"], "hits": hits, "chains": chains, "slow_path_slots": stats["slow_slots"],
        "fast_path_capacity": FAST_CAP,
        "ms": {"smem_step": round(mean["smem"], 3), "hits_count_locate": round(mean["hits"], 3), "chaining": round(mean["chain"], 3),
               "device_step": round(step, 3)},
        "chaining_hits_per_s": hits / (mean["chain"] * 1e-3),
        "chaining_algorithmic_bytes": alg_bytes,
        "chaining_bytes_per_s": alg_bytes / (mean["chain"] * 1e-3),
        "chaining_fraction_of_hbm_peak": round(alg_bytes / (mean["chain"] * 1e-3) / HBM_BYTES_PER_S, 4),
        "chaining_share_of_device_step": round(mean["chain"] / step, 4),
        "best_placement_rate": {"forward_drawn": stats["placed"][0] / max(stats["placeable"][0], 1),
                                "reverse_drawn": stats["placed"][1] / max(stats["placeable"][1], 1),
                                "reads_inside_one_sequence": stats["placeable"]},
        "per_step_ms": [{k: round(v, 3) for k, v in r.items()} for r in runs],
    }
    log(json.dumps(result["ms"]), "share", result["chaining_share_of_device_step"])
    print(json.dumps(result))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
