"""Hit expansion on the GPU (gsm_hits_count / gsm_hits_locate through locate_hits and Engine.locate_hits): every hit, in order,
against numpy applied to the host SA-IS suffix array, on a multi-sequence reference with empty and one-base sequences and a
300-base segment planted 700 times (intervals above max_occ 500)."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

L = 151
SEG = 300
COPIES = 700
LENGTHS = [0, 1, 50, 10_000, 200_000, 0, 400_000]


def make_reference():
    rng = np.random.default_rng(2024)
    seqs = [rng.integers(0, 4, n).astype(np.uint8) for n in LENGTHS]
    seg = rng.integers(0, 4, SEG).astype(np.uint8)
    # plant the segment at spaced, non-overlapping places in the three long sequences
    slots = [(3, p) for p in range(100, 10_000 - SEG, 2_000)]
    slots += [(4, p) for p in range(50, 200_000 - SEG, 600)]
    slots += [(6, p) for p in range(10, 400_000 - SEG, 900)]
    for i, p in slots[:COPIES]:
        seqs[i][p:p + SEG] = seg
    assert len(slots) >= COPIES
    text = np.concatenate(seqs)
    start = np.concatenate(([0], np.cumsum(LENGTHS))).astype(np.uint32)
    return text, start, slots[:COPIES]


def make_reads(text, start, slots, n_random=2000):
    rng = np.random.default_rng(7)
    n = len(text)
    starts = list(rng.integers(0, n - L, n_random))
    for s in start[1:-1]:                                           # across every boundary (empty sequences share one)
        starts += [max(0, min(n - L, int(s) - d)) for d in (1, 2, 75, 150)]
    for i, p in slots[::3]:                                         # from the repeat
        starts.append(int(start[i]) + p - int(rng.integers(0, 100)))
    reads = text[np.asarray(starts)[:, None] + np.arange(L)[None, :]].copy()
    mut = rng.random(reads.shape) < 0.01
    reads[mut] = (reads[mut] + 1) & 3
    reads = np.concatenate((reads, rng.integers(0, 4, (200, L), dtype=np.uint8)))
    return ["".join("ACGT"[c] for c in r) for r in reads]


def expected(recs, sa, start, max_occ, min_len):
    """The documented semantics in numpy: -> (offsets int64[n+1], hits n_hits x 4 uint32)."""
    lo = recs["sa_lo"].astype(np.int64)
    hi = recs["sa_hi"].astype(np.int64)
    cnt = np.where(hi >= lo, hi - lo + 1, 0)
    ln = np.maximum(recs["qend"].astype(np.int64) - recs["qstart"].astype(np.int64), 0)
    samp = (cnt > max_occ) if max_occ else np.zeros(len(recs), bool)
    n = np.where(ln < min_len, 0, np.where(samp, max_occ, cnt))
    step = np.where(samp, cnt // max(max_occ, 1), 1)
    off = np.concatenate(([0], np.cumsum(n))).astype(np.int64)
    rec = np.repeat(np.arange(len(recs)), n)
    k = np.arange(off[-1]) - off[rec]
    p = sa[lo[rec] + k * step[rec]].astype(np.int64) - 1
    st = start.astype(np.int64)
    c = np.searchsorted(st, p, side="right") - 1
    o = p - st[c]
    flags = (o + ln[rec] > st[c + 1] - st[c]).astype(np.int64) | (samp[rec].astype(np.int64) << 1)
    return off, np.stack([rec, c, o, flags], 1).astype(np.uint32)


def as_u32(res):
    h = res.hits
    return np.stack([h["record"], h["contig"], h["offset"], h["flags"]], 1).astype(np.uint32).reshape(-1, 4)


@pytest.fixture(scope="module")
def world():
    import genie_smem_b200 as g
    text, start, slots = make_reference()
    ascii_ = np.frombuffer(b"ACGT", np.uint8)[text].tobytes()
    host = g.HostIndex.build(ascii_)
    sa, _ = host.export()
    reads = make_reads(text, start, slots)
    contigs = g.Contigs(["s%d" % i for i in range(len(LENGTHS))], start)
    return dict(text=text, ascii=ascii_, host=host, sa=sa, start=start, reads=reads, contigs=contigs)


def run_records(g, index, reads):
    eng = g.Engine(index, len(reads), L, mems_per_read=64, recs_per_read=32)
    res = eng.run(g.METHOD_BWA, g.ReadBatch.from_strings(reads), min_len=1)
    return eng, res


def check(res, recs, sa, start, max_occ, min_len):
    off, want = expected(recs, sa, start, max_occ, min_len)
    assert np.array_equal(res.offsets, off), (max_occ, min_len)
    got = as_u32(res)
    assert got.shape == want.shape, (max_occ, min_len)
    bad = np.flatnonzero((got != want).any(1))
    assert len(bad) == 0, f"max_occ={max_occ} min_len={min_len}: {len(bad)} hits differ, first {got[bad[0]]} != {want[bad[0]]}"


@pytest.mark.parametrize("builder", ["host", "gpu"])
def test_hits_equal_numpy_on_host_sa(world, builder):
    import genie_smem_b200 as g
    index = g.DeviceIndex(world["host"]) if builder == "host" else g.DeviceIndex.build_on_device(world["ascii"])
    assert index.contigs is None
    index.set_contigs(world["contigs"])
    assert index.contigs == world["contigs"]
    eng, res = run_records(g, index, world["reads"])
    recs = res.records
    cnt = recs["sa_hi"].astype(np.int64) - recs["sa_lo"] + 1
    assert (cnt > 500).any() and (cnt >= 700).any(), "the planted repeat must give intervals above max_occ"
    for max_occ in (0, 1, 3, 500):
        for min_len in (0, 19):
            hr = g.locate_hits(index, recs, max_occ=max_occ, min_len=min_len)
            check(hr, recs, world["sa"], world["start"], max_occ, min_len)
    hr = g.locate_hits(index, recs)
    flags = np.unique(hr.hits["flags"])
    assert g.HIT_SPANS in flags and g.HIT_SAMPLED in flags
    # Engine.locate_hits works on the engine's device records: the same hits
    he = eng.locate_hits()
    assert np.array_equal(he.offsets, hr.offsets) and np.array_equal(he.hits, hr.hits)
    for i in (0, 5, len(world["reads"]) - 1):
        assert np.array_equal(hr.for_read(res, i), hr.hits[hr.offsets[res.offsets[i]]:hr.offsets[res.offsets[i + 1]]])
        for k in range(res.offsets[i], res.offsets[i + 1]):
            assert (hr.for_record(k)["record"] == k).all()


def test_hits_from_the_sampled_suffix_array(world):
    import genie_smem_b200 as g
    index = g.DeviceIndex(world["host"]).set_contigs(world["contigs"])
    _, res = run_records(g, index, world["reads"])
    recs = res.records
    full = {(m, n): g.locate_hits(index, recs, max_occ=m, min_len=n) for m in (0, 500) for n in (0, 19)}
    for S in (4, 32):
        idx = g.DeviceIndex(world["host"]).set_contigs(world["contigs"]).build_sampled_sa(S, drop_full=True)
        assert idx.sa is None
        for (m, n), want in full.items():
            hr = g.locate_hits(idx, recs, max_occ=m, min_len=n)
            check(hr, recs, world["sa"], world["start"], m, n)
            assert np.array_equal(hr.hits, want.hits)
        idx.ssa = None
        with pytest.raises(ValueError):
            g.locate_hits(idx, recs)


def test_empty_batches_and_records_without_hits(world):
    import genie_smem_b200 as g
    index = g.DeviceIndex(world["host"]).set_contigs(world["contigs"])
    hr = g.locate_hits(index, np.zeros(0, g.RECORD_DTYPE))
    assert len(hr) == 0 and hr.offsets.tolist() == [0]
    _, res = run_records(g, index, world["reads"][:50])
    hr = g.locate_hits(index, res.records, min_len=1000)
    assert len(hr) == 0 and hr.offsets.tolist() == [0] * (len(res.records) + 1)
    # runs of records without hits between records with hits (records longer than 60 bases keep theirs)
    check(g.locate_hits(index, res.records, min_len=60), res.records, world["sa"], world["start"], 500, 60)


def test_hit_cap_slices_and_overflow(world):
    import torch
    import genie_smem_b200 as g
    from genie_smem_b200 import _capi as capi
    index = g.DeviceIndex(world["host"]).set_contigs(world["contigs"])
    _, res = run_records(g, index, world["reads"])
    recs = res.records
    want = g.locate_hits(index, recs, max_occ=0)
    assert np.diff(want.offsets).max() > 512, "one record must span more than a tile"
    for cap in (1, 700, 1000, 4099):
        got = g.locate_hits(index, recs, max_occ=0, hit_cap=cap)
        assert np.array_equal(got.offsets, want.offsets) and np.array_equal(got.hits, want.hits), cap
    # the raw entry point never writes at or past out_cap, and says so
    dev = index.device
    r = torch.from_numpy(recs.view(np.uint8).copy()).to(dev)
    n = len(recs)
    counts = torch.empty(n, dtype=torch.int32, device=dev)
    off = torch.empty(n + 1, dtype=torch.int64, device=dev)
    tb = C.c_uint64()
    capi.check(capi.lib.gsm_hits_workspace_info(n, C.byref(tb)))
    tmp = torch.empty(int(tb.value), dtype=torch.uint8, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    capi.check(capi.lib.gsm_hits_count(r.data_ptr(), n, 500, 0, counts.data_ptr(), off.data_ptr(), tmp.data_ptr(), int(tb.value), stream))
    total = int(off[-1].item())
    ref = g.locate_hits(index, recs)
    assert total == len(ref) and np.array_equal(off.cpu().numpy(), ref.offsets)
    assert np.array_equal(counts.cpu().numpy(), np.diff(ref.offsets))
    cap = total - 37
    out = torch.full(((total + 64) * 4,), -1, dtype=torch.int32, device=dev)
    status = torch.zeros(1, dtype=torch.int64, device=dev)
    capi.check(capi.lib.gsm_hits_locate(C.byref(index.c), None, 0, C.byref(index._contigs_c), r.data_ptr(), off.data_ptr(), 0, n, 500, 0,
                                        out.data_ptr(), cap, status.data_ptr(), stream))
    o = out.cpu().numpy().view(np.uint32).reshape(-1, 4)
    assert int(status.item()) & 1
    assert np.array_equal(o[:cap], as_u32(ref)[:cap])
    assert (o[cap:] == 0xFFFFFFFF).all()


def test_one_sequence_without_a_table(world):
    import genie_smem_b200 as g
    index = g.DeviceIndex(world["host"])
    _, res = run_records(g, index, world["reads"][:300])
    start = np.asarray([0, len(world["text"])], np.uint32)
    for m in (0, 500):
        check(g.locate_hits(index, res.records, max_occ=m), res.records, world["sa"], start, m, 0)
    with pytest.raises(ValueError):
        index.set_contigs(g.Contigs(["a", "b"], [0, 5, 9]))


def test_index_file_keeps_the_sequence_table(world, tmp_path):
    import genie_smem_b200 as g
    index = g.DeviceIndex(world["host"]).set_contigs(world["contigs"])
    _, res = run_records(g, index, world["reads"][:400])
    want = g.locate_hits(index, res.records)
    p_with, p_without = str(tmp_path / "with.gsm"), str(tmp_path / "without.gsm")
    g.IndexFile.save(p_with, index, contigs=world["contigs"])
    g.IndexFile.save(p_without, index)
    head = g.IndexFile.header(p_with)
    assert head["contigs"] == world["contigs"].names
    assert "contig_start" in [d["name"] for d in head["sections"]]
    head0 = g.IndexFile.header(p_without)
    assert "contigs" not in head0 and "contig_start" not in [d["name"] for d in head0["sections"]]
    loaded, lut, lut_K, rmi = g.IndexFile.load(p_with, verify=True)
    assert loaded.contigs == world["contigs"]
    got = g.locate_hits(loaded, res.records)
    assert np.array_equal(got.hits, want.hits) and np.array_equal(got.offsets, want.offsets)
    loaded0, _, _, _ = g.IndexFile.load(p_without)
    assert loaded0.contigs is None
    got0 = g.locate_hits(loaded0, res.records)
    assert (got0.hits["contig"] == 0).all()
    with pytest.raises(ValueError):
        g.IndexFile.save(str(tmp_path / "bad.gsm"), index, contigs=g.Contigs.single(5))


def test_many_tiles_per_block(world):
    """Millions of hits: every block walks a run of tiles, taking each tile's first record from the previous tile's staging
    (also across runs of records without hits, min_len 40)."""
    import genie_smem_b200 as g
    index = g.DeviceIndex(world["host"]).set_contigs(world["contigs"])
    _, res = run_records(g, index, world["reads"])
    recs = np.tile(res.records, 150)
    for m, n in ((500, 0), (0, 0), (3, 40)):
        hr = g.locate_hits(index, recs, max_occ=m, min_len=n)
        assert m != 500 or len(hr) > 3_000_000
        check(hr, recs, world["sa"], world["start"], m, n)
    idx = g.DeviceIndex(world["host"]).set_contigs(world["contigs"]).build_sampled_sa(32, drop_full=True)
    check(g.locate_hits(idx, recs, max_occ=500, min_len=40), recs, world["sa"], world["start"], 500, 40)


def test_large_sequence_tables(world):
    """Start tables of 1,000 and 10,000 sequences (many empty): searched in shared memory or through L2 depending on size and
    path; the same hits either way."""
    import genie_smem_b200 as g
    rng = np.random.default_rng(5)
    n_bases = len(world["text"])
    index = g.DeviceIndex(world["host"])
    _, res = run_records(g, index, world["reads"])
    recs = res.records
    sampled = g.DeviceIndex(world["host"]).build_sampled_sa(32, drop_full=True)
    for n_seq in (1000, 10_000):
        cuts = np.sort(rng.integers(0, n_bases + 1, n_seq - 1))
        cuts[: n_seq // 10] = cuts[n_seq // 10]                     # a run of empty sequences
        start = np.concatenate(([0], np.sort(cuts), [n_bases])).astype(np.uint32)
        ct = g.Contigs([str(i) for i in range(n_seq)], start)
        for idx in (index, sampled):
            idx.set_contigs(ct)
            for m, n in ((500, 0), (0, 19)):
                check(g.locate_hits(idx, recs, max_occ=m, min_len=n), recs, world["sa"], start, m, n)
