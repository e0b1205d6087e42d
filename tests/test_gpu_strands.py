"""Both strands on the GPU: the strand-doubled batch (gsm_reads_both_strands_device) against the host packer of the
interleaved strings, Engine / PipelinedEngine with strands=2 against strands=1 and against the C oracle on the reverse
complements, and reads drawn from the reverse strand placed at their true origin."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

L = 151
LENGTHS = [0, 1, 15, 16, 17, 63, 64, 65, 151, 1024, 1025, 65535]
_COMP = str.maketrans("ACGT", "TGCA")


def rc(s):
    return s[::-1].translate(_COMP)


def interleave(reads):
    return [s for r in reads for s in (r, rc(r))]


@pytest.fixture(scope="module")
def gs():
    import genie_smem_b200 as g
    return g


@pytest.fixture(scope="module")
def world(gs):
    """3 Mbp synthetic reference, device index with seed table, 1,500 reads of 151 bp (1 % substitution reads from both
    strands, uniform-random reads) and a 150-base palindrome (151 bases cannot equal their reverse complement)."""
    rng = np.random.default_rng(77)
    ref = rng.integers(0, 4, 3_000_000, dtype=np.uint8)
    text = np.frombuffer(b"ACGT", np.uint8)[ref].tobytes()
    idx = gs.DeviceIndex.build_on_device(ref)
    idx.build_seed_table()
    sa = idx.suffix_array_host()
    tstr = text.decode()
    reads = []
    for k in range(1200):
        p = int(rng.integers(0, len(tstr) - L))
        q = list(tstr[p:p + L])
        for j in np.nonzero(rng.random(L) < 0.01)[0]:
            q[j] = "ACGT"[("ACGT".index(q[j]) + 1) % 4]
        q = "".join(q)
        reads.append(rc(q) if k % 2 else q)
    reads += ["".join("ACGT"[c] for c in rng.integers(0, 4, L)) for _ in range(300)]
    half = tstr[1000:1075]
    return dict(ref=ref, text=text, idx=idx, sa=sa, reads=reads, pal=half + rc(half))


def _dicts(reads, res, strand):
    out = []
    for i, q in enumerate(reads):
        d = {}
        for r in res.for_read(i, strand):
            d[q[int(r["qstart"]):int(r["qend"])]] = (int(r["sa_lo"]), int(r["sa_hi"]))
        out.append([[k, v[0], v[1]] for k, v in d.items()])
    return out


def _check_oracle(gs, res, reads, exp, what):
    """Slot 2i+1 of res against the oracle's records of the reverse-complement strings `reads`, status included."""
    got = _dicts(reads, res, 1)
    st = res.status[1::2]
    for k, e in enumerate(exp):
        if e == "raises":
            assert st[k] == gs.READ_REF_RAISES, (what, k)
        elif e == "short":
            assert st[k] == gs.READ_TOO_SHORT, (what, k)
        else:
            assert st[k] == gs.READ_OK, (what, k)
            assert got[k] == e, (what, k, reads[k])


def _same_but_read_id(a, b):
    for f in ("qstart", "qend", "sa_lo", "sa_hi"):
        if not np.array_equal(a[f], b[f]):
            return False
    return True


# ---------------------------------------------------------------------------------------------- the doubled batch
def _host_pack(gs, reads):
    b = gs.ReadBatch.from_strings(reads)
    return b.packed_host, b.chunk_off_host, b.len_host


def test_device_doubling_equals_host_pack(gs):
    rng = np.random.default_rng(1)
    reads = ["".join("ACGT"[c] for c in rng.integers(0, 4, n)) for n in LENGTHS]
    half = "".join("ACGT"[c] for c in rng.integers(0, 4, 33))
    reads.append(half + rc(half))
    want = _host_pack(gs, interleave(reads))
    batch = gs.ReadBatch.from_strings(reads, read_id_base=5)
    d = batch.both_strands()
    assert d.n == 2 * len(reads) and d.read_id_base == 10 and d.packed.is_cuda
    got = (d.packed.cpu().numpy(), d.chunk_off.cpu().numpy().view(np.uint32), d.len.cpu().numpy().view(np.uint32))
    for g_, w in zip(got, want):
        assert np.array_equal(g_, w)
    assert np.array_equal(d.chunk_off_host, want[1]) and np.array_equal(d.len_host, want[2])


@pytest.mark.parametrize("lo,hi", [(3, 9), (11, 12), (0, 12), (6, 6)])
def test_device_doubling_of_a_view(gs, lo, hi):
    import torch
    from genie_smem_b200 import _capi as capi
    rng = np.random.default_rng(2)
    reads = ["".join("ACGT"[c] for c in rng.integers(0, 4, n)) for n in LENGTHS]
    batch = gs.ReadBatch.from_strings(reads).to(torch.device("cuda"))
    assert lo == 0 or int(batch.chunk_off_host[lo]) != 0
    want = _host_pack(gs, interleave(reads[lo:hi]))
    r = capi.DevReads()
    r.n_reads = hi - lo
    r.packed = batch.packed.data_ptr()
    r.chunk_off = batch.chunk_off.data_ptr() + 4 * lo
    r.len = batch.len.data_ptr() + 4 * lo
    r.max_len, r.read_id_base = batch.max_len, 0
    nch = int(batch.chunk_off_host[hi]) - int(batch.chunk_off_host[lo])
    packed = torch.full((2 * nch * 16 + 16,), 0xAB, dtype=torch.uint8, device="cuda")
    coff = torch.full((2 * (hi - lo) + 1,), -1, dtype=torch.int32, device="cuda")
    lens = torch.full((max(2 * (hi - lo), 1),), -1, dtype=torch.int32, device="cuda")
    capi.check(capi.lib.gsm_reads_both_strands_device(C.byref(r), packed.data_ptr(), coff.data_ptr(), lens.data_ptr(),
                                                      C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    assert np.array_equal(packed.cpu().numpy(), want[0])
    assert np.array_equal(coff.cpu().numpy().view(np.uint32), want[1])
    assert np.array_equal(lens.cpu().numpy().view(np.uint32)[: 2 * (hi - lo)], want[2])


# ---------------------------------------------------------------------------------------------- records
def test_engine_strands2_all_methods(gs, world):
    import bench
    from oracle.c_oracle import COracle
    idx, reads = world["idx"], world["reads"]
    rcs = [rc(q) for q in reads]
    base = 1000
    batch = gs.ReadBatch.from_strings(reads, read_id_base=base)
    one = gs.Engine(idx, len(reads), L, mems_per_read=128, recs_per_read=96)
    two = gs.Engine(idx, len(reads), L, mems_per_read=128, recs_per_read=96, strands=2)
    o = COracle(world["text"], world["sa"])
    lut = gs.lut_build(idx, 10)
    rmi = bench.train_rmi(idx, 11, (64, 4096), idx.device)
    cases = [("bwa 1", gs.METHOD_BWA, {"min_len": 1}, o.smem_dicts(0, rcs, min_len=1)),
             ("bwa 20", gs.METHOD_BWA, {"min_len": 20}, o.smem_dicts(0, rcs, min_len=20)),
             ("lut", gs.METHOD_LUT, {"K": 10, "lut": lut}, o.smem_dicts(1, rcs, K=10)),
             ("rmi", gs.METHOD_RMI, {"rmi": rmi}, o.smem_dicts(2, rcs, rmi=bench.rmi_dict(rmi)))]
    for what, method, kw, exp in cases:
        a = one.run(method, batch, **kw)
        b = two.run(method, batch, **kw)
        assert b.strands == 2 and a.strands == 1 and len(b.offsets) == 2 * len(reads) + 1
        assert np.array_equal(b.lengths, np.full(len(reads), L, np.uint32))
        # read ids: 2 * (read_id_base + i) + strand
        slot = np.repeat(np.arange(2 * len(reads)), np.diff(b.offsets))
        assert np.array_equal(b.records["read_id"], (2 * base + slot).astype(np.uint32)), what
        # slot 2i = the strands=1 records of read i, in every field but read_id; status too
        assert np.array_equal(b.status[0::2], a.status), what
        for i in range(len(reads)):
            assert _same_but_read_id(b.for_read(i, 0), a.for_read(i)), (what, i)
        # slot 2i+1 = the method on the reverse complement
        _check_oracle(gs, b, rcs, exp, what)
        # for_read(i) without a strand = both slots
        i = 3
        assert len(b.for_read(i)) == len(b.for_read(i, 0)) + len(b.for_read(i, 1))


def test_pipelined_paths_equal_engine(gs, world):
    import torch
    idx = world["idx"]
    rng = np.random.default_rng(4)
    tstr = world["text"].decode()
    ragged = []
    for k in range(3001):
        n = int(rng.integers(20, 161))
        p = int(rng.integers(0, len(tstr) - n))
        q = tstr[p:p + n]
        ragged.append(rc(q) if k % 3 == 0 else q)
    ragged.append(world["pal"])
    fixed = world["reads"][:1499]
    eng = gs.Engine(idx, len(ragged), 160, mems_per_read=64, recs_per_read=64, strands=2)
    pipe = gs.PipelinedEngine(idx, len(ragged) + 10, 160, n_chunks=3, mems_per_read=64, recs_per_read=64, strands=2)

    def same(x, y):
        assert np.array_equal(x.offsets, y.offsets) and np.array_equal(x.records, y.records)
        assert np.array_equal(x.status, y.status) and np.array_equal(x.lengths, y.lengths)
        assert x.strands == y.strands == 2

    want = eng.run(gs.METHOD_BWA, gs.ReadBatch.from_strings(ragged, read_id_base=7), min_len=1)
    same(pipe.run(gs.METHOD_BWA, gs.ReadBatch.from_strings(ragged, read_id_base=7, pin=True), min_len=1), want)
    # the palindrome: identical records on both strands
    i = len(ragged) - 1
    assert _same_but_read_id(want.for_read(i, 0), want.for_read(i, 1))
    # FASTQ bytes, variable lengths
    fq = "".join(f"@r{k}\n{q}\n+\n{'I' * len(q)}\n" for k, q in enumerate(ragged)).encode()
    fq_t = torch.frombuffer(bytearray(fq), dtype=torch.uint8).pin_memory()
    want0 = eng.run(gs.METHOD_BWA, gs.ReadBatch.from_strings(ragged), min_len=1)
    same(pipe.run_fastq(gs.METHOD_BWA, fq_t, min_len=1), want0)
    # fixed-length ASCII
    eng_f = gs.Engine(idx, len(fixed), L, mems_per_read=64, recs_per_read=64, strands=2)
    want_f = eng_f.run(gs.METHOD_BWA, gs.ReadBatch.from_strings(fixed, read_id_base=3), min_len=1)
    asc = torch.from_numpy(np.frombuffer("".join(fixed).encode(), np.uint8).reshape(len(fixed), -1).copy()).pin_memory()
    same(pipe.run_ascii(gs.METHOD_BWA, asc, L, min_len=1, read_id_base=3), want_f)


# ---------------------------------------------------------------------------------------------- the user-visible result
def test_reverse_strand_reads_are_placed(gs):
    """Reads cut from the reverse strand of a multi-sequence reference, 1 % substitutions: with strands=2 each read's longest
    record is on strand 1 and its hit lies at the read's true sequence and offset; with strands=1 no read gets that."""
    from tests.test_gpu_hits import LENGTHS as SEQ_LENGTHS, make_reference
    text, start, _ = make_reference()
    index = gs.DeviceIndex(gs.HostIndex.build(np.frombuffer(b"ACGT", np.uint8)[text].tobytes()))
    index.set_contigs(gs.Contigs(["s%d" % i for i in range(len(SEQ_LENGTHS))], start))
    rng = np.random.default_rng(12)
    long_seqs = [i for i, n in enumerate(SEQ_LENGTHS) if n >= 10_000]
    reads, truth = [], []
    for _ in range(600):
        c = int(rng.choice(long_seqs))
        off = int(rng.integers(0, SEQ_LENGTHS[c] - L))
        w = text[int(start[c]) + off:int(start[c]) + off + L]
        q = (3 - w[::-1]).astype(np.uint8)                        # the reverse strand of the window
        mut = rng.random(L) < 0.01
        q[mut] = (q[mut] + 1) & 3
        reads.append("".join("ACGT"[x] for x in q))
        truth.append((c, off))
    truth = np.asarray(truth, np.int64)
    batch = gs.ReadBatch.from_strings(reads)

    def placed(res):
        """Per read: (longest record's strand, whether one of its hits is at the true origin)."""
        co = res.read_coords()
        hits = gs.locate_hits(index, res.records, max_occ=0)          # every occurrence: the planted repeat has 700
        ln = co["qend"].astype(np.int64) - co["qbeg"]
        strand, ok = np.zeros(len(reads), np.int64), np.zeros(len(reads), bool)
        for i in range(len(reads)):
            a, b = res.offsets[res.strands * i], res.offsets[res.strands * (i + 1)]
            k = a + int(np.argmax(ln[a:b]))
            strand[i] = co["strand"][k]
            h = hits.for_record(k)
            # a strand-1 match read[qbeg:qend] lies on the reverse strand; its forward-strand image starts at
            # origin + (L - qend) of the forward window = origin + qbeg' in RC coordinates
            want_off = truth[i, 1] + (L - int(co["qend"][k])) if co["strand"][k] else truth[i, 1] + int(co["qbeg"][k])
            ok[i] = bool(((h["contig"] == truth[i, 0]) & (h["offset"] == want_off)).any())
        return strand, ok

    two = gs.Engine(index, len(reads), L, mems_per_read=64, recs_per_read=32, strands=2).run(gs.METHOD_BWA, batch, min_len=1)
    s2, ok2 = placed(two)
    assert (s2 == 1).mean() > 0.99 and ok2.mean() > 0.99
    # hits of strand-1 records through HitResult.for_read
    hits = gs.locate_hits(index, two.records)
    assert len(hits.for_read(two, 0)) == len(hits.for_read(two, 0, 0)) + len(hits.for_read(two, 0, 1))
    one = gs.Engine(index, len(reads), L, mems_per_read=64, recs_per_read=32).run(gs.METHOD_BWA, batch, min_len=1)
    _, ok1 = placed(one)
    assert ok1.mean() < 0.05


def test_refusals(gs, world):
    idx = world["idx"]
    with pytest.raises(ValueError):
        gs.Engine(idx, 10, L, strands=3)
    pipe = gs.PipelinedEngine(idx, 100, L, n_chunks=2, strands=2)
    batch = gs.ReadBatch.from_strings(world["reads"][:50], pin=True)
    with pytest.raises(ValueError):
        pipe.run(gs.METHOD_BWA, batch, gatherer=object())
    with pytest.raises(ValueError):
        gs.Engine(idx, 100, L, strands=2).select(gs.METHOD_BWA, batch.both_strands(), gatherer=object())
    big = gs.ReadBatch.from_strings(world["reads"][:50], read_id_base=(1 << 31) - 25)
    with pytest.raises(ValueError):
        big.both_strands()
    with pytest.raises(ValueError):
        gs.Engine(idx, 100, L, strands=2).run(gs.METHOD_BWA, big)
    ok = gs.ReadBatch.from_strings(world["reads"][:50], read_id_base=(1 << 31) - 51)
    assert ok.both_strands().read_id_base == (1 << 32) - 102
