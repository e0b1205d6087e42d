#!/usr/bin/env python3
"""A/B harness: the bench's index and reads at a reduced read count, per-kernel times (CUDA events) and a checksum of
every method's records, as one JSON line.  Run it once per build and compare the lines.

Usage: python tools/sweep_ab.py [--reads N] [--ref-bases B] [--steps K] [--skip-rmi] [--tag name]"""
import argparse
import hashlib
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=10_000_000)
    ap.add_argument("--ref-bases", type=int, default=1_000_000_000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--seed-k", type=int, default=-1)
    ap.add_argument("--skip-rmi", action="store_true")
    ap.add_argument("--random-reads", action="store_true")
    ap.add_argument("--tag", default="")
    a = ap.parse_args()
    import torch
    import genie_smem_b200 as g
    t0 = time.time()
    seed = 1000 if a.ref_bases >= 500_000_000 else 100
    ref = bench.make_reference(a.ref_bases, seed)
    ref_dev = torch.from_numpy(ref).cuda()
    index = g.DeviceIndex.build_on_device(ref_dev, "cuda")
    if a.seed_k != 0:
        index.build_seed_table(None if a.seed_k < 0 else a.seed_k)
    codes = torch.empty((a.reads, bench.READ_LEN), dtype=torch.uint8, device="cuda")
    if a.random_reads:
        gen = torch.Generator(device="cuda")
        gen.manual_seed(seed + 1)
        codes[:] = torch.randint(0, 4, codes.shape, generator=gen, device="cuda", dtype=torch.uint8)
    else:
        bench.device_reads(ref_dev, a.reads, bench.READ_LEN, seed + 1, codes)
    batch = g.ReadBatch.from_device_bases(codes, bench.READ_LEN)
    del codes, ref_dev
    caps = dict(mems_per_read=96, recs_per_read=64) if a.random_reads else dict(mems_per_read=24, recs_per_read=8)
    eng = g.Engine(index, a.reads, bench.READ_LEN, **caps)
    lut = g.lut_build(index, bench.LUT_K)
    experts = bench.CONFIGS["c3" if a.ref_bases < 500_000_000 else "c4"]["experts"]
    rmi = None if a.skip_rmi else bench.train_rmi(index, bench.RMI_K, experts, "cuda", probe_table=False)
    torch.cuda.synchronize()
    setup = time.time() - t0

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

    out = {"tag": a.tag, "reads": a.reads, "ref_bases": a.ref_bases,
           "seed_K": int(index.seed_K), "setup_s": round(setup, 1)}
    out["ms_sweep"] = round(timed(lambda: eng.sweep(batch), a.steps), 3)
    legs = [("bwa", g.METHOD_BWA, {"min_len": 1}), ("lut", g.METHOD_LUT, {"K": bench.LUT_K, "lut": lut}),
            ("lut_machine", g.METHOD_LUT, {"K": bench.LUT_K, "lut": lut})]
    if rmi is not None:
        legs.append(("rmi", g.METHOD_RMI, {"rmi": rmi}))
        legs.append(("rmi_bounds", g.METHOD_RMI, {"rmi": rmi}))
    persist = os.environ.get("AB_PERSIST")               # A/B: pin the LUT / the RMI parameters in the persisting L2
    for name, method, kw in legs:
        if persist:
            import ctypes as C
            from genie_smem_b200 import _capi as capi
            t = lut if name == "lut" else (rmi.params if name.startswith("rmi") else None)
            st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
            if t is None:
                capi.check(capi.lib.gsm_l2_persist(None, 0, st))
            else:
                capi.check(capi.lib.gsm_l2_persist(C.c_void_p(t.data_ptr()), t.numel() * t.element_size(), st))
        g.set_lut_frame_machine(name == "lut_machine")       # "lut": the sweep's picks; "lut_machine": the reference's frame machine
        if name == "rmi_bounds":                      # same lookups from the dense bounds table (gsm_rmi_bounds_build)
            out["ms_bounds_build"] = round(timed(lambda: rmi.build_bounds_table(index), 1), 1)
        out[f"ms_select_{name}"] = round(timed(lambda: eng.select(method, batch, **kw), a.steps), 3)
        n_mems, n_rec = eng.check_overflow()
        recs = eng.records[: n_rec * 16].cpu().numpy()
        out[f"records_{name}"] = n_rec
        out[f"sha_{name}"] = hashlib.sha256(recs.tobytes()).hexdigest()[:16]
        out["n_mems"] = n_mems
    out["ms_per_10M_reads_sweep"] = round(out["ms_sweep"] * 1e7 / a.reads, 2)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
