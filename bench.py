#!/usr/bin/env python3
"""bench.py -- SMEM reads/s on B200 (BASELINE.json metric) for the B200-native engine.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c4|c3|c5] [--scaling strong|weak] [--impl reference]
                    [--dump-outputs DIR] ...

Workload = BASELINE.json configs[3] (`--config c4`, the configuration the metric is quoted on): synthetic 1 Gbp random ACGT
reference (numpy PCG64(1000)), 50 M reads of 151 bp (exact substrings with i.i.d. 1 % substitutions, SURVEY 8d), all three
SMEM methods.  `--config c3` = configs[2] (100 Mbp, 10 M reads), `--config c5` = configs[4] (3 Gbp, 100 M reads, RMI- vs
BWA-SMEM).  The index (suffix array, both BWT bucket arrays, seed table, LUT) is built ON THE GPU in about a second.

Multi-GPU (torchrun, one rank per GPU): the index is replicated, the config's reads are sharded by rank -- STRONG scaling, as
configs[3] states ("50M reads sharded across 1/2/4/8"); `--scaling weak` gives every GPU the config's full read count instead.
The one collective of the path -- per-rank records to rank 0 -- is INSIDE every timed region at N > 1: each rank's ordered
write kernel stores its records straight into its region of a buffer in rank 0's HBM through a peer mapping (NVLink /
NVSwitch), and one 8-byte-per-rank NCCL all-gather of the counts is the completion fence (sharding.RecordGatherer).

A "step" is one pass of the hot path over the read batch.
  value   BWA-SMEM reads/s, packed reads already resident in HBM: sweep + select + scan + ordered write (+ the gather at N > 1)
  e2e     the same through the public API from HOST buffers: 2-bit packed reads in pinned host memory -> H2D -> kernels ->
          records to pinned host memory (N = 1) / gathered into rank 0's HBM with offsets + status D2H per rank (N > 1);
          e2e.ascii_input = from raw ASCII read bytes (packed on the GPU), e2e.from_fastq = from FASTQ file bytes
  methods LUT- and RMI-SMEM throughputs; roofline / roofline_methods: algorithmic bytes (SURVEY 8d) over time vs the HBM peak
  parity  GPU records of the first reads of THIS batch against oracle/smem_oracle.c (the reference restated), all methods;
          any mismatch fails the run
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from, which may be read-only

READ_LEN = 151
SUB_RATE = 0.01
LUT_K = 12
RMI_K = 15
_B = np.frombuffer(b"ACGT", dtype=np.uint8)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# stdout carries exactly ONE JSON line: keep a private copy of it and point fd 1 at stderr, so that nothing a library
# prints (NCCL's version banner under NCCL_DEBUG, torch warnings) can land next to the result
_RESULT_OUT = None


def _claim_stdout():
    global _RESULT_OUT
    if _RESULT_OUT is None:
        sys.stdout.flush()
        _RESULT_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit_result(obj):
    _claim_stdout()
    print(json.dumps(obj), file=_RESULT_OUT, flush=True)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def make_reference(n_bases, seed=100):
    rng = np.random.Generator(np.random.PCG64(seed))
    return rng.integers(0, 4, n_bases, dtype=np.uint8)


def make_reads_host(ref_codes, n_reads, L, seed, sub_rate=SUB_RATE, chunk=1_000_000):
    """(n_reads, L) uint8 codes: exact substrings with i.i.d. substitutions (seed = config seed + 1)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    out = np.empty((n_reads, L), np.uint8)
    ar = np.arange(L, dtype=np.int64)[None, :]
    for a in range(0, n_reads, chunk):
        b = min(n_reads, a + chunk)
        starts = rng.integers(0, len(ref_codes) - L + 1, b - a)
        r = ref_codes[starts[:, None] + ar]
        mut = rng.random(r.shape) < sub_rate
        r[mut] = (r[mut] + rng.integers(1, 4, int(mut.sum()), dtype=np.uint8)) & 3
        out[a:b] = r
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1 + 0.2] or [r for _, r in self.rows]
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for k, nm in enumerate(names):
                    if r[5 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ CPU arm (oracle = checker / baseline only)
def cpu_arm(o, reads_codes, method, threads, budget_s, K=0, rmi=None, n_min=0):
    """Run the oracle port (oracle/smem_oracle.c, the reference algorithm restated in C) on the host cores over a bounded
    sample of the same reads.  Returns (reads/s, n_sample, threads, out, counts): the outputs are what `parity` compares
    the GPU records with."""
    threads = threads or o.max_threads
    L = reads_codes.shape[1]

    def run(n):
        sub = reads_codes[:n]
        joined = _B[sub.reshape(-1)].tobytes()
        lens = np.full(n, L, np.uint32)
        t0 = time.perf_counter()
        out, counts = o.smems(method, None, min_len=1, K=K, rmi=rmi, threads=threads, joined=joined, lens=lens)
        return time.perf_counter() - t0, out, counts

    n = min(max(64 * threads, n_min), len(reads_codes))
    if method == 1:
        o.lib.orc_build_lut(o.h, K)          # table build is index construction, not search
    dt, out, counts = run(n)
    rate = n / dt
    n2 = int(max(n, min(len(reads_codes), rate * budget_s)))
    if n2 > 2 * n:
        dt, out, counts = run(n2)
        n = n2
    return n / dt, n, threads, out, counts


def rmi_dict(params):
    return {"K": params.K, "level_sizes": [int(x) for x in params.level_sizes], "coef": params.coef_host, "intercept": params.intercept_host}


def compare_with_oracle(reads_codes, snap, out, counts, n):
    """GPU records of the first n reads (snap = (records, offsets, status) host arrays) against the oracle's output for the
    same reads, after the reference's dict semantics (duplicate SMEM strings collapse: first insertion keeps its place,
    last value wins).  Returns (#mismatching reads, #reads where the reference raises)."""
    recs, offs, status = snap
    mism = raises = 0
    for r in range(n):
        q = reads_codes[r]
        if counts[r] == -1:                       # the reference raises on this read: the kernel must flag it
            raises += 1
            mism += int(status[r] != 1)
            continue
        d = {}
        for rec in recs[offs[r]:offs[r + 1]]:
            d[q[int(rec["qstart"]):int(rec["qend"])].tobytes()] = (int(rec["sa_lo"]), int(rec["sa_hi"]))
        got = [(k, v[0], v[1]) for k, v in d.items()]
        exp = [(q[int(o[0]):int(o[1])].tobytes(), int(o[2]), int(o[3])) for o in out[r, :max(int(counts[r]), 0)]]
        mism += int(got != exp or status[r] != 0)
    return mism, raises


# ------------------------------------------------------------------------------------------ configuration
CONFIGS = {"c4": dict(ref_bases=1_000_000_000, reads=50_000_000, seed=1000, experts=(2048, 1048576), name="BASELINE.json configs[3]"),
           "c3": dict(ref_bases=100_000_000, reads=10_000_000, seed=100, experts=(512, 131072), name="BASELINE.json configs[2]"),
           "c5": dict(ref_bases=3_000_000_000, reads=100_000_000, seed=3000, experts=(4096, 4194304), name="BASELINE.json configs[4]")}
HOST_READS = 600_000      # the first reads of every batch come from numpy so the CPU arms can regenerate exactly them
PARITY_READS = 20_000     # reads per method compared with the oracle at N = 1 (2,048 at N > 1)
# --dump-outputs: reads sampled with a fixed seed.  A read has at most READ_LEN records (their ends strictly increase), so
# 10,000 reads x 151 records x 40 bytes (5 float64 fields) keeps the dump under 64 MB whatever the workload.
DUMP_READS = 10_000
DUMP_SEED = 20261020
DUMP_MAX_BYTES = 64_000_000


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--config", default="c4", choices=sorted(CONFIGS))
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"], help="N > 1: shard the config's reads (strong) or give every GPU all of them (weak)")
    ap.add_argument("--reads", type=int, default=0, help="total reads per step (default: the config's)")
    ap.add_argument("--ref-bases", type=int, default=0, help="reference size (default: the config's)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="CPU baseline budget per method")
    ap.add_argument("--skip-rmi", action="store_true")
    ap.add_argument("--skip-extras", action="store_true", help="skip the ascii / fastq / locate / probe-search legs")
    ap.add_argument("--e2e-chunks", type=int, default=8, help="chunks of the pipelined end-to-end path")
    ap.add_argument("--seed-k", type=int, default=-1, help="K of the sweep kernel's seed table (-1 = auto, 0 = none)")
    ap.add_argument("--sub-rate", type=float, default=SUB_RATE, help="substitution rate of the synthetic reads (SURVEY 8d extremes: 0)")
    ap.add_argument("--random-reads", action="store_true", help="uniform random reads instead of reference substrings (SURVEY 8d extreme)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed BWA-SMEM step returned in its last step (a fixed sample of reads) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the outputs of the native path")
    cfg = dict(CONFIGS[args.config])
    if args.ref_bases:
        cfg["ref_bases"] = args.ref_bases
        cfg["name"] = "custom size"
        # leaves scale with the reference: about one leaf per 1,000 rows
        leaves = 1 << max(10, int(np.log2(max(args.ref_bases // 1000, 1024))))
        cfg["experts"] = (max(16, leaves >> 9), leaves)
    if args.reads:
        cfg["reads"] = args.reads
        if cfg["name"] != "custom size":
            cfg["name"] += f" shape, {args.reads/1e6:g} M reads"
    args.ref_bases, args.total_reads, args.seed, args.experts, args.cfg_name = cfg["ref_bases"], cfg["reads"], cfg["seed"], cfg["experts"], cfg["name"]
    return args


def workload_dict(args, world, reads_rank):
    bucket_mb = 2 * (args.ref_bases // 192 + 1) * 64 / 1e6
    total = args.total_reads if args.scaling == "strong" else args.total_reads * world
    return {"workload": f"synthetic {args.ref_bases/1e6:g} Mbp random ACGT reference (PCG64 seed {args.seed}), "
                        f"{total/1e6:g} M reads x {READ_LEN} bp per step"
                        + (f" sharded over {world} GPUs ({reads_rank/1e6:g} M each)" if world > 1 else "") + ", "
                        + ("uniform random reads" if args.random_reads else f"exact substrings + {args.sub_rate:.0%} substitutions") + f" ({args.cfg_name})",
            "ref_bases": args.ref_bases, "reads_per_step": total, "reads_per_gpu": reads_rank, "read_len": READ_LEN,
            "sub_rate": None if args.random_reads else args.sub_rate,
            "lut_K": LUT_K, "rmi_K": RMI_K, "rmi_experts": list(args.experts), "min_len": 1,
            "parallelism": f"reads sharded x{world}, index replicated; records gathered to rank 0 inside the timed region" if world > 1
                           else "one GPU",
            "l2_policy": f"inputs larger than L2: packed read batch {reads_rank * 48 / 1e6:.0f} MB, rank buckets {bucket_mb:.0f} MB, seed table + outputs "
                         f"> 1 GB vs 126 MB L2 (at --config c3 the 67 MB of buckets are L2-resident by design; see DESIGN.md)"}


def host_reads(ref_codes, n, seed, sub_rate=SUB_RATE, random_reads=False):
    if random_reads:
        return np.random.Generator(np.random.PCG64(seed)).integers(0, 4, (n, READ_LEN), dtype=np.uint8)
    return make_reads_host(ref_codes, n, READ_LEN, seed=seed, sub_rate=sub_rate)


def device_reads(ref_dev, n, L, seed, out, sub_rate=SUB_RATE, chunk=2_000_000):
    """Fill out[(n, L) uint8, device] with synthetic reads: exact substrings + i.i.d. substitutions (torch RNG on the
    device; workload generation only)."""
    import torch
    gen = torch.Generator(device=ref_dev.device)
    gen.manual_seed(seed)
    ar = torch.arange(L, device=ref_dev.device, dtype=torch.int64)[None, :]
    for a in range(0, n, chunk):
        b = min(n, a + chunk)
        starts = torch.randint(0, ref_dev.numel() - L + 1, (b - a, 1), generator=gen, device=ref_dev.device, dtype=torch.int64)
        r = ref_dev[(starts + ar).view(-1)].view(b - a, L)
        mut = torch.rand(r.shape, generator=gen, device=ref_dev.device) < sub_rate
        add = torch.randint(1, 4, r.shape, generator=gen, device=ref_dev.device, dtype=torch.uint8)
        out[a:b] = torch.where(mut, (r + add) & 3, r)
    return out


def algorithmic_bytes(recs_i32, n_rec, n_reads, K=0, probe_bytes=0):
    """SURVEY 8d: bytes(read) = 128 * sum_records(len + [start > 0]) + ceil(L/4) + 16 * #records; for LUT / RMI every record
    with len >= K trades K of its steps for `probe_bytes` (LUT: one 32-byte sector; RMI: P probes x 64 B)."""
    import torch
    steps = n_long = 0
    for a in range(0, n_rec, 50_000_000):
        w = recs_i32[a:a + 50_000_000, 1]
        qs = (w & 0xFFFF).to(torch.int64)
        qe = ((w >> 16) & 0xFFFF).to(torch.int64)
        steps += int(((qe - qs) + (qs > 0).to(torch.int64)).sum().item())
        if K:
            n_long += int(((qe - qs) >= K).sum().item())
    total = 128 * (steps - K * n_long) + probe_bytes * n_long + n_reads * ((READ_LEN + 3) // 4) + 16 * n_rec
    return total, steps, n_long


def dump_outputs(out_dir, engine, n_reads, n_mems, n_rec):
    """What Engine.run hands its caller for the batch the engine just ran (records, CSR offsets, per-read status, counts),
    for DUMP_READS reads drawn with DUMP_SEED, as float64 arrays in out_dir:
      read_ids (S,)      the sampled reads, ascending
      status   (S,)      READ_OK / READ_REF_RAISES / READ_TOO_SHORT of each sampled read
      offsets  (S + 1,)  CSR offsets of the sampled reads' rows in `records`
      records  (R, 5)    read_id, qstart, qend, sa_lo, sa_hi
      totals   (2,)      maximal matches and records of the whole batch"""
    import torch
    from genie_smem_b200.engine import RECORD_DTYPE
    dev = engine.device
    ids = np.sort(np.random.default_rng(DUMP_SEED).choice(n_reads, min(n_reads, DUMP_READS), replace=False))
    ids_t = torch.from_numpy(ids).to(dev)
    lo = engine.rec_off[ids_t].cpu().numpy()
    hi = engine.rec_off[ids_t + 1].cpu().numpy()
    rows = torch.from_numpy(np.concatenate([np.arange(a, b) for a, b in zip(lo, hi)] + [np.empty(0, np.int64)])).to(dev)
    recs = engine.records[: n_rec * 16].view(torch.int32).view(-1, 4)[rows].cpu().numpy().view(RECORD_DTYPE).reshape(-1)
    arrays = {"read_ids": ids, "status": engine.read_status[ids_t].cpu().numpy(), "offsets": np.concatenate([[0], np.cumsum(hi - lo)]),
              "records": np.stack([recs[f] for f in RECORD_DTYPE.names], axis=1), "totals": np.asarray([n_mems, n_rec])}
    arrays = {k: np.asarray(v, np.float64) for k, v in arrays.items()}
    nbytes = sum(a.nbytes for a in arrays.values())
    assert nbytes <= DUMP_MAX_BYTES, f"output dump of {nbytes} bytes"
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    log(f"outputs of the last timed step: {len(ids)} reads, {len(recs)} records, {nbytes / 1e6:.1f} MB in {out_dir}")


def main():
    args = parse_args()
    _claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        if rank != 0:
            return
        reference_arm(args, workload_dict(args, world, args.total_reads // world if args.scaling == "strong" else args.total_reads))
        return

    import torch
    import torch.distributed as dist
    import genie_smem_b200 as g
    from genie_smem_b200 import sharding

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs runs on one GPU")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        cpus = sharding.bind_to_gpu_numa(local_rank)                # pinned host buffers land on the GPU's NUMA node
        log(f"[rank {rank}] bound to {len(cpus) if cpus else 'no'} CPUs next to GPU {local_rank}")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # stdout carries exactly one JSON line
        dist.init_process_group("nccl", device_id=dev)
    if args.scaling == "strong":
        lo_r, hi_r = sharding.shard_range(args.total_reads, rank, world)
        n_reads = hi_r - lo_r
        n_max = max(sharding.shard_range(args.total_reads, r, world)[1] - sharding.shard_range(args.total_reads, r, world)[0] for r in range(world))
        job_reads = args.total_reads
    else:
        lo_r, n_reads, n_max = rank * args.total_reads, args.total_reads, args.total_reads
        job_reads = args.total_reads * world
    workload = workload_dict(args, world, n_reads)

    # ---- setup: reference, index (built on the GPU), reads, LUT, RMI
    t_setup = time.time()
    ref = make_reference(args.ref_bases, args.seed)
    ref_dev = torch.from_numpy(ref).to(dev)
    t0 = time.time()
    index = g.DeviceIndex.build_on_device(ref_dev, dev)
    log(f"[rank {rank}] reference generated in {t0-t_setup:.1f}s; index built on the GPU in {index.build_stats['build_ms']:.0f} ms "
        f"(workspace {index.build_stats['workspace_bytes']/1e9:.1f} GB, {index.build_stats['doubling_rounds']} doubling rounds)")
    if args.seed_k != 0:
        index.build_seed_table(None if args.seed_k < 0 else args.seed_k)
    n_host = min(HOST_READS, n_reads)
    reads_head = host_reads(ref, n_host, args.seed + 1 + rank, args.sub_rate, args.random_reads)   # numpy: the CPU arms regenerate exactly these
    codes_dev = torch.empty((n_reads, READ_LEN), dtype=torch.uint8, device=dev)
    codes_dev[:n_host] = torch.from_numpy(reads_head).to(dev)
    if n_reads > n_host:
        if args.random_reads:
            gen = torch.Generator(device=dev)
            gen.manual_seed(args.seed + 1 + rank)
            codes_dev[n_host:] = torch.randint(0, 4, (n_reads - n_host, READ_LEN), generator=gen, device=dev, dtype=torch.uint8)
        else:
            device_reads(ref_dev, n_reads - n_host, READ_LEN, args.seed + 1 + rank, codes_dev[n_host:], sub_rate=args.sub_rate)
    batch = g.ReadBatch.from_device_bases(codes_dev, READ_LEN, read_id_base=lo_r)
    extras = not args.skip_extras
    ascii_host = None
    if extras:                      # raw read bytes in pinned host memory (1 byte/base): the ASCII leg of the end-to-end path
        ascii_lut = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device=dev)
        ascii_host = torch.empty((n_reads, READ_LEN), dtype=torch.uint8, pin_memory=True)
        for a in range(0, n_reads, 5_000_000):
            b = min(n_reads, a + 5_000_000)
            ascii_host[a:b].copy_(ascii_lut[codes_dev[a:b].long()])
    del codes_dev, ref_dev
    torch.cuda.empty_cache()
    caps = dict(mems_per_read=96, recs_per_read=64) if args.random_reads else dict(mems_per_read=24, recs_per_read=8)
    engine = g.Engine(index, n_reads, READ_LEN, **caps)
    lut = g.lut_build(index, LUT_K)
    rmi = None
    if not args.skip_rmi:
        t0 = time.time()
        rmi = train_rmi(index, RMI_K, args.experts, dev, probe_table=False, bounds_table=True)
        log(f"[rank {rank}] RMI training in {time.time()-t0:.1f}s (max |prediction error| on the training sample: {rmi.max_err:.0f} rows)")
    torch.cuda.synchronize()
    log(f"[rank {rank}] setup {time.time()-t_setup:.1f}s, index {index.bytes()/1e6:.0f} MB on device")

    gat = None
    if world > 1:                   # the gather destination: one buffer in rank 0's HBM, mapped by every rank
        gat = sharding.RecordGatherer(capacity=(int(caps["recs_per_read"] * n_max * 0.75) + 4096) * world, dst=0, device=dev)
        log(f"[rank {rank}] gather destination mapped ({gat.capacity * 16 / 1e9:.1f} GB on rank 0, NCCL {gat.comm.nccl_version})")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / steps

    def step(method, **kw):
        """one device-resident step: sweep + select + ordered write; at N > 1 the write IS the gather to rank 0"""
        if gat is None:
            engine.launch(method, batch, **kw)
            return
        gat.reset()
        engine.launch(method, batch, gatherer=gat, **kw)
        gat.fence()

    def snapshot(n):
        """host copies of the records / offsets / status of the first n reads of the batch just run (for `parity`)"""
        offs = engine.rec_off[: n + 1].cpu().numpy()
        if gat is not None:         # records went to rank 0's buffer: write them locally too for the check
            engine.collect_local(batch)
        recs = engine.records[: int(offs[n]) * 16].cpu().numpy().view(g.RECORD_DTYPE)
        return recs, offs, engine.read_status[:n].cpu().numpy()

    n_par = min(PARITY_READS if world == 1 else 2048, n_host)
    snaps = {}

    # ---- headline: BWA-SMEM, device-resident inputs
    sampler = ClockSampler(local_rank)
    sampler.start()
    t_region0 = time.time()
    launches0 = engine.kernel_launches
    ms_bwa = timed(lambda: step(g.METHOD_BWA, min_len=1), args.steps, args.warmup)
    gpu_launches = (engine.kernel_launches - launches0) * args.steps // (args.steps + args.warmup)
    t_region1 = time.time()
    clocks = sampler.stop(t_region0, t_region1)
    n_mems, n_rec = engine.check_overflow()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, engine, n_reads, n_mems, n_rec)
    gathered = None
    if gat is not None:
        parts, totals = gat.finish()
        tot = torch.tensor([n_rec], device=dev, dtype=torch.int64)
        dist.all_reduce(tot)
        if rank == 0:
            assert int(totals.sum()) == int(tot.item()) == sum(p.numel() for p in parts) // 16, "gathered record count != sum of the ranks' counts"
            for r in range(world):              # every rank's region holds that rank's global read ids, in order
                if int(totals[r]):
                    lo_s, hi_s = (sharding.shard_range(args.total_reads, r, world) if args.scaling == "strong"
                                  else (r * args.total_reads, (r + 1) * args.total_reads))
                    s = parts[r].view(torch.int32).view(-1, 4)[:, 0]
                    assert int(s[0]) == lo_s and int(s[-1]) == hi_s - 1 and bool((s[1:] >= s[:-1]).all()), f"region of rank {r} is not its shard"
            gathered = {"records": int(tot.item()), "bytes": int(tot.item()) * 16, "per_rank": [int(x) for x in totals]}
    snaps["bwa"] = snapshot(n_par)

    # ---- per-kernel split of the step + algorithmic bytes (roofline of the dominant kernel, k_sweep1)
    ms_sweep = timed(lambda: engine.sweep(batch), args.steps, 1)
    engine.sweep(batch)
    ms_sel_bwa = timed(lambda: engine.select(g.METHOD_BWA, batch, min_len=1), args.steps, 1)
    recs = engine.records[: n_rec * 16].view(torch.int32).view(-1, 4)
    alg_bytes, steps_alg, _ = algorithmic_bytes(recs, n_rec, n_reads)
    peak, peak_src = measured_peak()
    achieved = alg_bytes / (ms_sweep * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tname = {1_000_000_000: "r02_1gbp_sweep_dram_bytes.json", 100_000_000: "r02_100mbp_sweep_dram_bytes.json"}.get(args.ref_bases)
    if tname and os.path.exists(os.path.join(ROOT, "profiles", tname)):        # ncu --set full capture of k_sweep1 on this reference size
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", tname)))
            traffic = tj["dram_bytes_per_read"] * n_reads
            traffic_src = f"profiles/{tname}: {tj['dram_bytes_per_read']:.0f} DRAM bytes/read (ncu dram__bytes_read+write of k_sweep1) x reads per launch"
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "kernel": "k_sweep1", "achieved": round(achieved, 2), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "algorithmic_bytes_per_read": round(alg_bytes / n_reads, 1), "fm_steps_per_read_min": round(steps_alg / n_reads, 2),
                "records_per_read": round(n_rec / n_reads, 3), "ms_sweep": round(ms_sweep, 3), "ms_select_scan_write": round(ms_sel_bwa, 3),
                "reads_per_launch": n_reads,
                "note": "achieved = algorithmic bytes (SURVEY 8d: 128 B per necessary FM step + read + records) of one launch / k_sweep1's "
                        "average launch time (CUDA events on the launching stream).  The kernel replaces the FM steps of unique matches by "
                        "text comparisons, so it moves fewer bytes than the algorithmic count charges (see `traffic`); the access pattern "
                        "is dependent random 16..64-byte fetches, bound by the request rate of the memory system (profiles/r02_notes.md)"}
    methods = {"bwa": {"reads_per_s": job_reads / (ms_bwa * 1e-3), "ms_per_step": ms_bwa}}
    roofline_methods = {"bwa": {"achieved": round(alg_bytes / (ms_bwa * 1e-3) / 1e9, 2), "frac": round(alg_bytes / (ms_bwa * 1e-3) / 1e9 / peak, 4),
                                "algorithmic_bytes_per_read": round(alg_bytes / n_reads, 1), "ms_sweep": round(ms_sweep, 3),
                                "ms_select": round(ms_sel_bwa, 3), "dominant_kernel": "k_sweep1"}}

    # ---- the other two methods (device-resident; same step definition)
    def method_leg(name, method, steps, kw, K, probe_bytes, extra):
        ms = timed(lambda: step(method, **kw), steps, 1)
        _, nr = engine.check_overflow()
        if gat is not None:
            gat.finish()
        snaps[name] = snapshot(n_par)
        engine.sweep(batch)
        ms_sel = timed(lambda: engine.select(method, batch, **kw), max(2, steps), 1)
        rr = engine.records[: nr * 16].view(torch.int32).view(-1, 4)
        ab, st_, nl = algorithmic_bytes(rr, nr, n_reads, K=K, probe_bytes=probe_bytes)
        methods[name] = dict({"reads_per_s": job_reads / (ms * 1e-3), "ms_per_step": ms, "K": K}, **extra)
        roofline_methods[name] = {"achieved": round(ab / (ms * 1e-3) / 1e9, 2), "frac": round(ab / (ms * 1e-3) / 1e9 / peak, 4),
                                  "algorithmic_bytes_per_read": round(ab / n_reads, 1), "records_with_len_ge_K_per_read": round(nl / n_reads, 3),
                                  "ms_sweep": round(ms_sweep, 3), "ms_select": round(ms_sel, 3),
                                  "dominant_kernel": "k_sweep1" if ms_sweep >= ms_sel else f"k_select_seeded<{name.upper()}>"}
        return ms

    g.set_lut_frame_machine(False)
    method_leg("lut", g.METHOD_LUT, max(2, args.steps // 2), {"K": LUT_K, "lut": lut}, LUT_K, 32,
               {"selection": "the sweep's picks: get_smems_lut emits exactly get_SMEMS's records with min_len 1 for reads of >= K bases "
                             "(DESIGN.md section 3); K flags reads that are too short"})
    if extras and world == 1:
        # the reference's frame machine itself (k_select_seeded<LUT>): same records, the cross-check of the identity above
        g.set_lut_frame_machine(True)
        try:
            ms_m = timed(lambda: step(g.METHOD_LUT, K=LUT_K, lut=lut), 2, 1)
            engine.check_overflow()
            snaps["lut_frame_machine"] = snapshot(n_par)
            engine.sweep(batch)
            methods["lut"]["frame_machine_reads_per_s"] = job_reads / (ms_m * 1e-3)
            methods["lut"]["frame_machine_select_ms"] = round(timed(lambda: engine.select(g.METHOD_LUT, batch, K=LUT_K, lut=lut), 2, 1), 3)
        finally:
            g.set_lut_frame_machine(False)
    if rmi is not None:
        P = 2 * int(np.ceil(np.log2(2 * rmi.max_err + 2)))
        method_leg("rmi", g.METHOD_RMI, max(2, args.steps // 2), {"rmi": rmi}, RMI_K, 64 * P,
                   {"experts": list(args.experts), "max_abs_prediction_error_rows": rmi.max_err, "probes_P": P,
                    "lookup": ("predict + true bounds from the dense k-mer bounds table (one fetch)" if rmi.bounds is not None else
                               "predict + seed-table bounds (one fetch + K - seed_K backward steps)") +
                              " + arithmetic replay of the error-bounded search (no probes); literal search on hazards"})
        st = engine.read_status[:n_reads]
        methods["rmi"]["reads_where_reference_raises"] = int((st == g.READ_REF_RAISES).sum().item())
        methods["rmi"]["prefilter"] = {
            "hazard_codes": rmi.n_hazards, "codes": 4 ** RMI_K, "active": rmi.hazard_slots is not None,
            "what": "reads without a hazard window (a k-mer code whose last-mile search is not certified exact) take the BWA-SMEM "
                    "records with min_len 1 (k_rmi_prefilter + k_select<BWA>); only the others run the frame machine"}
        if extras and world == 1 and rmi.hazard_slots is not None:
            # the reference's frame machine on every read (k_select_seeded<RMI> alone): same records, the cross-check
            g.set_rmi_prefilter(False)
            try:
                ms_m = timed(lambda: step(g.METHOD_RMI, rmi=rmi), 2, 1)
                engine.check_overflow()
                snaps["rmi_frame_machine"] = snapshot(n_par)
                engine.sweep(batch)
                methods["rmi"]["frame_machine_reads_per_s"] = job_reads / (ms_m * 1e-3)
                methods["rmi"]["frame_machine_select_ms"] = round(timed(lambda: engine.select(g.METHOD_RMI, batch, rmi=rmi), 2, 1), 3)
            finally:
                g.set_rmi_prefilter(True)
        if extras and world == 1:
            if rmi.bounds is not None:
                # the same lookups with the true bounds taken from the sweep's seed table + K - seed_K backward steps
                rmi.drop_bounds_table()
                torch.cuda.empty_cache()
                engine.sweep(batch)
                methods["rmi"]["seed_table_lookup_select_ms"] = round(timed(lambda: engine.select(g.METHOD_RMI, batch, rmi=rmi), 1, 1), 3)
                engine.check_overflow()
                snaps["rmi_seed_table"] = snapshot(n_par)
            # the probe-based error-bounded search (round-1 path: 16-byte {SA, 32-mer} probe records): same records, more fetches
            rmi.build_probe_table(index)
            seed_keep = (index.seed_table, index.seed_K)
            engine.sweep(batch)
            index.seed_table, index.seed_K = None, 0
            index._bind()
            ms_probe = timed(lambda: engine.select(g.METHOD_RMI, batch, rmi=rmi), 1, 1)
            index.seed_table, index.seed_K = seed_keep
            index._bind()
            _, nr2 = engine.check_overflow()
            methods["rmi"]["probe_search_select_ms"] = round(ms_probe, 3)
            snaps["rmi_probe"] = snapshot(n_par)
            rmi.probe = None
            rmi.c.probe = None
            torch.cuda.empty_cache()

    # ---- locate: SA intervals -> text positions with the sampled suffix array configs[3] names (1/32)
    locate = None
    if extras and world == 1:
        engine.launch(g.METHOD_BWA, batch, min_len=1)
        rows = engine.records[: n_rec * 16].view(torch.int32).view(-1, 4)[:, 2].contiguous()
        index.build_sampled_sa(32, drop_full=False)
        pos = torch.empty_like(rows)
        import ctypes as C
        from genie_smem_b200 import _capi as capi

        def loc():
            capi.check(capi.lib.gsm_locate_sampled_batch(C.byref(index.c), C.c_void_p(index.ssa.data_ptr()), 32, n_rec, C.c_void_p(rows.data_ptr()),
                                                          C.c_void_p(pos.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        ms_loc = timed(loc, 2, 1)
        chk = slice(0, min(n_rec, 2_000_000))
        ok = bool((index.sa[rows[chk].long()] == pos[chk]).all().item())
        assert ok, "sampled-SA positions differ from the full suffix array"
        lf_steps = 31.0          # row-sampled: geometric with p = 1/32
        locate = {"rows_per_s": n_rec / (ms_loc * 1e-3), "reads_per_s": n_reads / (ms_loc * 1e-3), "ms": round(ms_loc, 3), "rows": n_rec,
                  "sample": 32, "expected_lf_steps_per_row": lf_steps,
                  "achieved_GBs": round(n_rec * (64 * lf_steps + 12) / (ms_loc * 1e-3) / 1e9, 1),
                  "frac": round(n_rec * (64 * lf_steps + 12) / (ms_loc * 1e-3) / 1e9 / peak, 4),
                  "equals_full_sa_on": chk.stop,
                  "hbm_footprint_MB": {"buckets_fwd_rev": round(2 * index.fwd.numel() * 4 / 1e6), "sampled_sa": round(index.ssa.numel() * 4 / 1e6),
                                       "full_sa": round(index.sa.numel() * 4 / 1e6), "text": round(index.text.numel() * 4 / 1e6),
                                       "seed_table": round(index.seed_table.numel() * 4 / 1e6) if index.seed_table is not None else 0,
                                       "lut": round(lut.numel() * 4 / 1e6), "rmi_params": round(rmi.params.numel() * 8 / 1e6) if rmi is not None else 0,
                                       "rmi_bounds_table": round((8 << (2 * RMI_K)) / 1e6) if rmi is not None else 0,
                                       "rmi_probe_table_optional": round(index.n_rows * 16 / 1e6)},
                  "note": "one thread per row, LF-walk to the next sampled row (k_locate_sampled); BWA/LUT-SMEM + locate need buckets + sampled SA "
                          "only; the full SA (and text) are kept for RMI-SMEM's literal fallback"}
        del rows, pos

    # ---- NCCL point-to-point gather of the same records (baseline transport of the collective)
    record_gather = None
    if world > 1:
        engine.launch(g.METHOD_BWA, batch, min_len=1)
        cnts = torch.zeros(world, dtype=torch.int64, device=dev)
        mine = torch.tensor([n_rec], dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(cnts, mine)
        cnts_h = cnts.cpu().numpy().astype(np.uint64)
        dst_buf = gat.buffer if rank == 0 else None          # (contiguous from the buffer's start: the regions are rewritten by the next step)
        ms_g = timed(lambda: gat.comm.gather_records(engine.records, n_rec, cnts_h, dst_buf, 0), 3, 1)
        tb = int(cnts_h.sum()) * 16
        record_gather = {"transport": "gsm_gather_records: one ncclGroup of exact-size ncclSend/ncclRecv into a preallocated device buffer on rank 0",
                         "ms": round(ms_g, 3), "bytes": tb, "GBs": round(tb / (ms_g * 1e-3) / 1e9, 1),
                         "fused_alternative": "in `value`/`e2e` the gather is the ordered-write kernel's stores into rank 0's HBM (peer mapping)"}

    # ---- end to end through the public API: host reads in, records out
    del engine
    torch.cuda.empty_cache()
    pipe = g.PipelinedEngine(index, n_max, READ_LEN, n_chunks=args.e2e_chunks, **caps)

    def e2e_time(step_fn, steps=None):
        steps = steps or args.steps
        for _ in range(2):
            step_fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            res = step_fn()
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        return job_reads * steps / dt, res

    batch.to_host(pin=True)

    def run_packed(gatherer):
        if gatherer is not None:
            gatherer.reset()
        r = pipe.run(g.METHOD_BWA, batch, min_len=1, reuse_host_buffers=True, gatherer=gatherer)
        if gatherer is not None:
            gatherer.fence()
        return r

    v_packed, res = e2e_time(lambda: run_packed(gat))
    e2e = {"value": v_packed, "unit": "reads/s", "h2d_bytes_per_step": batch.h2d_bytes(), "d2h_bytes_per_step": pipe.last_d2h_bytes,
           "method": "bwa", "input": "2-bit packed reads in pinned host memory (48 B per 151-bp read)",
           "api": f"PipelinedEngine.run ({args.e2e_chunks} chunks, 3 streams: reads H2D | sweep, select, ordered write | records D2H, all overlapped)"}
    if gat is not None:
        parts, totals = gat.finish()
        e2e["api"] = (f"PipelinedEngine.run(gatherer=RecordGatherer) ({args.e2e_chunks} chunks: reads H2D | sweep, select, ordered write into this "
                      "rank's region of rank 0's buffer over NVLink | offsets + status D2H; one 8-byte-per-rank all-gather as the fence); "
                      "records are delivered gathered on rank 0's device")
        e2e["gathered_records"] = int(totals.sum())
        e2e["nvlink_bytes_into_rank0_per_step"] = (int(totals.sum()) - int(totals[0])) * 16
        v_shard, res2 = e2e_time(lambda: run_packed(None))
        e2e["sharded_host_output"] = {"value": v_shard, "d2h_bytes_per_step": pipe.last_d2h_bytes,
                                      "api": "PipelinedEngine.run: every rank copies its own records to its pinned host memory, no gather"}
    else:
        assert len(res.records) == n_rec, "end-to-end path and device-resident path disagree on the number of records"
        e2e["records_last_step"] = int(len(res.records))
    if extras and ascii_host is not None:
        v_ascii, res3 = e2e_time(lambda: pipe.run_ascii(g.METHOD_BWA, ascii_host, READ_LEN, min_len=1, reuse_host_buffers=True), max(2, args.steps // 2))
        e2e["ascii_input"] = {"value": v_ascii, "h2d_bytes_per_step": pipe.last_h2d_bytes,
                              "api": "PipelinedEngine.run_ascii (raw ASCII read bytes, 1 byte/base H2D, 2-bit packing on the GPU; per-rank host output)"}
        assert len(res3.records) == n_rec
    if extras and world == 1 and ascii_host is not None:
        e2e["from_fastq"] = fastq_leg(g, pipe, ascii_host.numpy(), n_rec_expected=None)

    # ---- parity + CPU baseline on the host cores (rank 0; the timed baseline at N = 1 only)
    cpu_baseline, parity = None, None
    if rank == 0:
        from oracle.c_oracle import COracle
        text = _B[ref].tobytes()
        o = COracle(text, index.suffix_array_host())
        budget = args.cpu_seconds if world == 1 else 0.0
        parity = {"reads": n_par, "against": "oracle/smem_oracle.c (reference get_SMEMS / get_smems_lut / get_smems_rmi restated literally, "
                                             "pinned to tests/golden) on the first reads of this batch"}
        v, n_s, thr, out, counts = cpu_arm(o, reads_head, 0, 0, budget, n_min=n_par)
        parity["bwa"], _ = compare_with_oracle(reads_head, snaps["bwa"], out, counts, n_par)
        if world == 1 and budget > 0:
            cpu_baseline = {"value": round(v, 1), "unit": "reads/s", "cores": thr, "kind": "port",
                            "sample": f"first {n_s} reads of the same batch, BWA-SMEM, oracle/smem_oracle.c (reference algorithm, "
                                      f"O(L^2) restarts included) on {thr} pthreads"}
        v2, _, _, out, counts = cpu_arm(o, reads_head, 1, 0, budget / 2, K=LUT_K, n_min=n_par)
        parity["lut"], _ = compare_with_oracle(reads_head, snaps["lut"], out, counts, n_par)
        if "lut_frame_machine" in snaps:
            parity["lut_frame_machine"], _ = compare_with_oracle(reads_head, snaps["lut_frame_machine"], out, counts, n_par)
        if cpu_baseline:
            cpu_baseline["lut_reads_per_s"] = round(v2, 1)
        if rmi is not None:
            v3, _, _, out, counts = cpu_arm(o, reads_head, 2, 0, budget / 2, rmi=rmi_dict(rmi), n_min=n_par)
            parity["rmi"], parity["ref_raises"] = compare_with_oracle(reads_head, snaps["rmi"], out, counts, n_par)
            if "rmi_probe" in snaps:
                parity["rmi_probe_search"], _ = compare_with_oracle(reads_head, snaps["rmi_probe"], out, counts, n_par)
            if "rmi_frame_machine" in snaps:
                parity["rmi_frame_machine"], _ = compare_with_oracle(reads_head, snaps["rmi_frame_machine"], out, counts, n_par)
            if "rmi_seed_table" in snaps:
                parity["rmi_seed_table_lookup"], _ = compare_with_oracle(reads_head, snaps["rmi_seed_table"], out, counts, n_par)
            if cpu_baseline:
                cpu_baseline["rmi_reads_per_s"] = round(v3, 1)
        if cpu_baseline:
            cpu_baseline["python_port"] = python_port_baseline()
        del o

    if rank == 0:
        out = {"metric": "SMEM reads/sec (BWA-SMEM; LUT/RMI under methods)", "value": job_reads / (ms_bwa * 1e-3), "unit": "reads/s",
               "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_bwa, "higher_is_better": True,
               "scaling": args.scaling, "vs_baseline": None, "dtype": "u32", "data": "synthetic", "config": workload,
               "roofline": roofline, "roofline_methods": roofline_methods, "cpu_baseline": cpu_baseline, "e2e": e2e, "parity": parity,
               "gpu_launches": int(gpu_launches), "clocks": clocks, "methods": methods, "records_total": n_rec if gathered is None else gathered["records"],
               "maximal_matches_per_read": round(n_mems / n_reads, 3), "gathered": gathered, "record_gather": record_gather, "locate": locate,
               "index_build": index.build_stats}
        out["sweep_seed_table_K"] = int(index.c.seed_K)
        out["limiter"] = name_limiter(ms_bwa, ms_sweep, ms_sel_bwa, e2e, job_reads, world)
        if world > 1:
            out["value_includes"] = "sweep + select + scan + ordered write of every rank, the write being the gather into rank 0's HBM (NVLink), + completion fence"
            out["gather_transport"] = ("peer mapping (CUDA IPC): each rank's ordered-write kernel stores into rank 0's buffer" if gat.fused else
                                       f"NCCL send/recv per batch (peer mapping unavailable: {gat.fallback_reason})")
        emit_result(out)
    bad = rank == 0 and parity is not None and any(parity.get(k, 0) for k in ("bwa", "lut", "lut_frame_machine", "rmi", "rmi_frame_machine", "rmi_probe_search", "rmi_seed_table_lookup"))
    if world > 1:
        dist.destroy_process_group()
    if bad:
        log(f"PARITY FAILURE: {parity}")
        sys.exit(3)


def name_limiter(ms_step, ms_sweep, ms_select, e2e, job_reads, world):
    """What bounds the step at this N, from the numbers measured above (never raises: the record matters more)."""
    try:
        other = max(ms_step - ms_sweep - ms_select, 0.0)
        rest = ("NVLink ingest of the other ranks' records into rank 0 + completion fence + kernel tails" if world > 1
                else "launch gaps between the kernels")
        parts = {"k_sweep1 (request-rate bound random 16..64-byte fetches, see roofline)": ms_sweep,
                 "selection + scan + ordered write": ms_select, rest: other}
        top = max(parts, key=parts.get)
        out = {"device": {"limiter": top, "share_of_step": round(parts[top] / ms_step, 3), "ms_step": round(ms_step, 3),
                          "ms_sweep": round(ms_sweep, 3), "ms_select_scan_write_local": round(ms_select, 3), "ms_rest": round(other, 3)}}
        e2e_ms = job_reads / e2e["value"] * 1e3
        gb = (e2e.get("h2d_bytes_per_step", 0) + e2e.get("d2h_bytes_per_step", 0)) / 1e9
        if e2e_ms <= 1.1 * ms_step:
            why = "the device kernels (copies and chunk launches hidden behind them)"
        else:
            why = (f"the host side: {e2e_ms - ms_step:.1f} ms per step beyond the kernels -- first-chunk H2D / last-chunk D2H that cannot overlap, "
                   f"per-chunk launches and the Python loop around them ({gb:.2f} GB cross PCIe per rank and step)")
        out["e2e"] = {"limiter": why, "ms_step": round(e2e_ms, 3), "over_device_step": round(e2e_ms / ms_step, 3)}
        return out
    except Exception as e:          # noqa: BLE001
        return {"unavailable": str(e)[:200]}


def fastq_leg(g, pipe, reads_head, n_rec_expected):
    """File bytes in, records out (reads_head: (n, L) ASCII read bytes).  A 4-line FASTQ of the batch's first reads is written to a temporary file and read back
    (page cache) into pinned memory; timed: (a) PipelinedEngine.run_fastq -- the host only looks for a record boundary near
    each chunk cut, the records are cut and 2-bit packed by GPU kernels, chunk by chunk behind the H2D copies -- and (b)
    the host path of round 1, ingest.read_fastq (multi-threaded scan + gather on the host cores) -> run_ascii."""
    import tempfile
    import torch
    from genie_smem_b200 import ingest
    n = min(len(reads_head), pipe.max_reads, 5_000_000)
    L = reads_head.shape[1]
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "reads.fq")
        rec = np.empty((n, 2 * L + 16), np.uint8)
        rec[:, :10] = np.frombuffer(b"@r0000000\n", np.uint8)
        idx = np.arange(n)
        for k in range(7):
            rec[:, 8 - k] = 48 + (idx // 10 ** k) % 10
        rec[:, 10:10 + L] = reads_head[:n]
        rec[:, 10 + L] = 10
        rec[:, 11 + L] = ord("+")
        rec[:, 12 + L] = 10
        rec[:, 13 + L:13 + 2 * L] = ord("I")
        rec[:, 13 + 2 * L] = 10
        rec[:, :14 + 2 * L].tofile(path)
        nbytes = os.path.getsize(path)
        fq = torch.from_numpy(np.fromfile(path, np.uint8)).pin_memory()
        for _ in range(2):
            r = pipe.run_fastq(g.METHOD_BWA, fq, min_len=1, reuse_host_buffers=True)
        torch.cuda.synchronize()
        steps = 3
        t0 = time.perf_counter()
        for _ in range(steps):
            r = pipe.run_fastq(g.METHOD_BWA, fq, min_len=1, reuse_host_buffers=True)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / steps
        n_rec = int(len(r.records))
        assert len(r.offsets) == n + 1
        # the host-scanner path, for comparison (first 200 k reads are enough to time it)
        m = min(n, 200_000)
        small = os.path.join(d, "small.fq")
        rec[:m, :14 + 2 * L].tofile(small)
        t0 = time.perf_counter()
        bases, off, _ = ingest.read_fastq(small)
        t_ingest = time.perf_counter() - t0
        r2 = pipe.run_ascii(g.METHOD_BWA, torch.from_numpy(bases).view(m, L), L, min_len=1, reuse_host_buffers=True)
        t_host = time.perf_counter() - t0
        assert np.array_equal(r2.offsets, r.offsets[: m + 1])
    return {"value": n / dt, "unit": "reads/s", "reads": n, "file_bytes": nbytes, "h2d_bytes_per_step": nbytes, "records": n_rec,
            "api": "PipelinedEngine.run_fastq: FASTQ file bytes (pinned) H2D in chunks | gsm_fastq_count_device + gsm_fastq_records_device + "
                   "gsm_pack_reads_scattered_device on the copy-in stream | sweep, select | records D2H",
            "host_scanner_path": {"value": m / t_host, "reads": m, "scan_gather_reads_per_s": m / t_ingest,
                                  "api": "ingest.read_fastq (gsm_fastq_scan / gsm_fastq_gather on the host cores) -> PipelinedEngine.run_ascii"}}


def python_port_baseline(budget_s=1.5):
    """BASELINE.md section 3 asks for the reference's own Python on the box's cores: one process and
    multiprocessing.Pool(os.cpu_count()), for get_SMEMS / get_smems_lut / get_smems_rmi.  /root/reference does not travel to the
    GPU box, so the literal Python restatement (oracle/ref_port.py, pinned to the same goldens) is timed instead on configs[0]
    (big_data, 100 kb; 101-bp exact substrings) -- in its own process (oracle/py_baseline.py), so that the pool forks from a
    process that never touched CUDA."""
    try:
        r = subprocess.run([sys.executable, "-m", "oracle.py_baseline", "--seconds", str(budget_s)], cwd=ROOT, capture_output=True,
                           text=True, timeout=120, env=dict(os.environ, PYTHONDONTWRITEBYTECODE="1"))
        if r.returncode != 0:
            return {"unavailable": (r.stderr or "oracle.py_baseline failed").strip().splitlines()[-1][:200]}
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception as e:          # fixtures absent, timeout: report, do not fail the bench
        return {"unavailable": str(e)[:200]}


def train_rmi(index, K, experts, dev, max_keys=8_000_000, probe_table=True, bounds_table=False):
    """RMI over the k-mer -> row keys of this index (reference RMI_LUT.py:36-50).  Training set = a strided sample of the
    (suffix array row, k-mer) pairs read from the suffix array + packed text on the device; model quality only changes the
    last-mile length, never the result.  The fit is the vectorised host trainer.  probe_table: also build the 16-byte
    {SA value, 32-mer} probe records the probe-based search uses (not needed by the seed-table lookup path).  bounds_table:
    also the dense {first row >= k-mer, occurrences} table (4^K x 8 B) when K <= 16 and the device has room for it."""
    import torch
    import genie_smem_b200 as g
    n_rows = index.n_rows
    stride = max(1, n_rows // max_keys)
    rows_t = torch.arange(0, n_rows, stride, device=dev, dtype=torch.int64)
    start = index.sa[rows_t].to(torch.int64) & 0xFFFFFFFF
    start = start - 1                                               # 0-based text index of the suffix
    ok = start + K <= index.n_bases
    rows_t, start = rows_t[ok], start[ok]
    text = index.text.to(torch.int64) & 0xFFFFFFFF
    key = torch.zeros_like(start)
    for t in range(K):                                              # MSB-first k-mer code (LUT.convert_seq_to_num)
        p = start + t
        key = key * 4 + ((text[p >> 4] >> (30 - 2 * (p & 15))) & 3)
    del text
    key_h, rows_h = key.cpu().numpy(), rows_t.cpu().numpy()
    m = g.RMI(list(experts)).fit(key_h, rows_h)
    out = g.RmiParams(K, m.level_sizes, m.coef, m.intercept, dev)
    out.max_err = float(np.abs(m.predict(key_h) - rows_h).max())
    if probe_table:
        out.build_probe_table(index)
    out.build_none_rows(index)
    if bounds_table and K <= 16 and torch.cuda.mem_get_info(index.device)[0] > (8 << (2 * K)) + (24 << 30):
        out.build_bounds_table(index)
    return out


def reference_arm(args, workload):
    """--impl reference: the reference's CPU path (oracle port in C, all host threads) on bounded samples of the same
    workload.  The suffix array both arms search is an INPUT of the path: it is built by whichever builder is available
    (the GPU builder when a device is visible, else host SA-IS) before the timed region; the timed search runs on the
    host cores only, through oracle/smem_oracle.c, with none of the engine's kernels."""
    import genie_smem_b200 as g
    ref = make_reference(args.ref_bases, args.seed)
    text = _B[ref].tobytes()
    sa1, built_by = None, None
    try:
        import torch
        if torch.cuda.is_available():
            idx = g.DeviceIndex.build_on_device(ref, "cuda:0", reverse=False)
            sa1 = idx.suffix_array_host()
            built_by = "gsm_index_build_device (this repo's GPU builder, before the timed region; bit-equal to host SA-IS in tests)"
            del idx
            torch.cuda.empty_cache()
    except Exception as e:          # no usable device: fall through to the host builder
        log(f"reference arm: GPU index build unavailable ({e}); using host SA-IS")
    if sa1 is None:
        sa1, _ = g.HostIndex.build(text, reverse=False).export()
        built_by = "gsm_index_build (this repo's host SA-IS, before the timed region)"
    reads_codes = host_reads(ref, min(args.total_reads, HOST_READS), args.seed + 1, args.sub_rate, args.random_reads)
    from oracle.c_oracle import COracle
    o = COracle(text, sa1)
    thr = o.max_threads
    L = READ_LEN
    # size one step to ~8 s
    n0 = 32 * thr
    joined = _B[reads_codes[:n0].reshape(-1)].tobytes()
    t0 = time.perf_counter()
    o.smems(0, None, min_len=1, threads=thr, joined=joined, lens=np.full(n0, L, np.uint32))
    rate = n0 / (time.perf_counter() - t0)
    n = int(min(len(reads_codes), max(n0, rate * 8.0)))
    joined = _B[reads_codes[:n].reshape(-1)].tobytes()
    lens = np.full(n, L, np.uint32)
    for _ in range(min(args.warmup, 1)):
        o.smems(0, None, min_len=1, threads=thr, joined=joined, lens=lens)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        o.smems(0, None, min_len=1, threads=thr, joined=joined, lens=lens)
    dt = (time.perf_counter() - t0) / args.steps
    v = n / dt
    sample = f"{n} reads per step (first reads of the batch), BWA-SMEM, oracle/smem_oracle.c on {thr} pthreads"
    out = {"impl": "reference", "metric": "SMEM reads/sec (BWA-SMEM; LUT/RMI under methods)", "value": v, "unit": "reads/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": args.scaling,
           "vs_baseline": None, "dtype": "u32", "data": "synthetic", "config": workload,
           "cpu_baseline": {"value": v, "unit": "reads/s", "cores": thr, "kind": "port", "sample": sample},
           "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
           "reference_class": "cpu", "index_built_by": built_by}
    emit_result(out)


if __name__ == "__main__":
    main()
