"""Seed chaining on the GPU (gsm_chain_seeds / gsm_chains_collect through Engine.chain_seeds and chain_seeds): every chain,
offset and hit id against the literal restatement of tests/test_chains_host.py applied to the returned hits, on a
multi-sequence reference with empty and one-base sequences, a 300-base segment planted 700 times (slots with hundreds of
chains: the slow path) and a tandem repeat; placement of simulated reads drawn from both strands by best()."""
import ctypes as C

import numpy as np
import pytest

from tests.test_chains_host import oracle_chains

pytestmark = pytest.mark.gpu

L = 151
SEG = 300
COPIES = 700
LENGTHS = [0, 1, 50, 10_000, 200_000, 0, 400_000]
TANDEM = (6, 350_000, 1_400)          # sequence, offset, length of a period-7 tandem repeat
FAST_CAP = 8                          # chains per slot on the fast path (csrc/chains.cu)


def make_reference():
    rng = np.random.default_rng(2024)
    seqs = [rng.integers(0, 4, n).astype(np.uint8) for n in LENGTHS]
    seg = rng.integers(0, 4, SEG).astype(np.uint8)
    slots = [(3, p) for p in range(100, 10_000 - SEG, 2_000)]
    slots += [(4, p) for p in range(50, 200_000 - SEG, 600)]
    slots += [(6, p) for p in range(10, 400_000 - SEG, 900)]
    slots = slots[:COPIES]
    for i, p in slots:
        seqs[i][p:p + SEG] = seg
    c, p, n = TANDEM
    assert all(not (i == c and q + SEG > p and q < p + n) for i, q in slots)
    seqs[c][p:p + n] = np.tile(rng.integers(0, 4, 7).astype(np.uint8), n // 7 + 1)[:n]
    start = np.concatenate(([0], np.cumsum(LENGTHS))).astype(np.uint32)
    return np.concatenate(seqs), start, slots


def revcomp(codes):
    return (3 - codes[::-1]).astype(np.uint8)


def make_reads(text, start, slots):
    """-> (reads as strings, truth per read: (contig, offset, strand) or None when the read is not a clean placement)."""
    rng = np.random.default_rng(7)
    repeats = [(i, p, SEG) for i, p in slots] + [TANDEM]
    reads, truth = [], []
    long_seqs = [i for i, n in enumerate(LENGTHS) if n >= L]
    weights = np.asarray([LENGTHS[i] for i in long_seqs], np.float64)
    for _ in range(2000):                                           # simulated, both strands, 1 % substitutions
        c = long_seqs[int(rng.choice(len(long_seqs), p=weights / weights.sum()))]
        o = int(rng.integers(0, LENGTHS[c] - L + 1))
        strand = int(rng.integers(0, 2))
        r = text[int(start[c]) + o:int(start[c]) + o + L].copy()
        mut = rng.random(L) < 0.01
        r[mut] = (r[mut] + 1) & 3
        clean = not any(i == c and p < o + L and o < p + n for i, p, n in repeats)
        reads.append(revcomp(r) if strand else r)
        truth.append((c, o, strand) if clean else None)
    n = len(text)
    for s in start[1:-1]:                                           # across every boundary
        for d in (1, 2, 75, 150):
            p = max(0, min(n - L, int(s) - d))
            reads.append(text[p:p + L].copy())
            truth.append(None)
    for i, p in slots[::12]:                                        # from the planted repeat
        q = int(start[i]) + p - int(rng.integers(0, 100))
        reads.append(text[q:q + L].copy())
        truth.append(None)
    c, p, m = TANDEM
    for k in range(20):                                             # from the tandem repeat, both strands
        q = int(start[c]) + p + int(rng.integers(0, m - L))
        r = text[q:q + L].copy()
        reads.append(revcomp(r) if k & 1 else r)
        truth.append(None)
    for _ in range(200):
        reads.append(rng.integers(0, 4, L).astype(np.uint8))
        truth.append(None)
    return ["".join("ACGT"[x] for x in r) for r in reads], truth


@pytest.fixture(scope="module")
def world():
    import genie_smem_b200 as g
    text, start, slots = make_reference()
    ascii_ = np.frombuffer(b"ACGT", np.uint8)[text].tobytes()
    host = g.HostIndex.build(ascii_)
    reads, truth = make_reads(text, start, slots)
    contigs = g.Contigs(["s%d" % i for i in range(len(LENGTHS))], start)
    index = g.DeviceIndex(host).set_contigs(contigs)
    sampled = g.DeviceIndex(host).set_contigs(contigs).build_sampled_sa(16, drop_full=True)
    return dict(host=host, index=index, sampled=sampled, lut=g.lut_build(index, 8), reads=reads, truth=truth, start=start)


def run(g, world, strands, method, index=None):
    index = index if index is not None else world["index"]
    eng = g.Engine(index, len(world["reads"]), L, mems_per_read=64, recs_per_read=32, strands=strands)
    kw = dict(K=8, lut=world["lut"]) if method == g.METHOD_LUT else dict(min_len=1)
    res = eng.run(method, g.ReadBatch.from_strings(world["reads"]), **kw)
    return eng, res


def u32(a, k):
    return np.ascontiguousarray(a).view(np.uint32).reshape(-1, k)


def check_against_oracle(g, index, res, cr, max_occ, min_len, w, max_gap):
    want_hits = g.locate_hits(index, res.records, max_occ=max_occ, min_len=min_len)
    assert np.array_equal(cr.hits.offsets, want_hits.offsets) and np.array_equal(cr.hits.hits, want_hits.hits)
    assert np.array_equal(cr.rec_offsets, res.offsets)
    chains, off, ids = oracle_chains(u32(res.records, 4), res.offsets, u32(cr.hits.hits, 4), cr.hits.offsets, w, max_gap)
    assert np.array_equal(cr.offsets, off)
    got = u32(cr.chains, 8)
    assert got.shape == chains.shape
    bad = np.flatnonzero((got != chains).any(1))
    assert len(bad) == 0, f"{len(bad)} chains differ, first {got[bad[0]]} != {chains[bad[0]]}"
    bad = np.flatnonzero(cr.hit_chain != ids)
    assert len(bad) == 0, f"{len(bad)} hit ids differ, first {cr.hit_chain[bad[0]]:#x} != {ids[bad[0]]:#x}"


CONFIGS = [
    # strands, method, max_occ, min_len, w, max_gap, sampled SA
    (2, "BWA", 500, 19, 100, 10000, False),
    (1, "BWA", 500, 19, 100, 10000, False),
    (2, "LUT", 3, 0, 0, 1, False),
    (2, "BWA", 0, 19, 100, 10000, True),
    (1, "LUT", 500, 0, 100, 1, True),
    (2, "BWA", 3, 19, 0, 10000, False),
    (1, "BWA", 0, 0, 0, 10000, False),
    (2, "LUT", 500, 19, 100, 10000, True),
]


@pytest.mark.parametrize("strands,method,max_occ,min_len,w,max_gap,sampled", CONFIGS)
def test_chains_equal_the_oracle(world, strands, method, max_occ, min_len, w, max_gap, sampled):
    import genie_smem_b200 as g
    index = world["sampled"] if sampled else world["index"]
    eng, res = run(g, world, strands, getattr(g, "METHOD_" + method), index)
    cr = eng.chain_seeds(max_occ=max_occ, min_len=min_len, w=w, max_gap=max_gap)
    assert cr.strands == strands and len(cr.offsets) == len(res.offsets)
    check_against_oracle(g, index, res, cr, max_occ, min_len, w, max_gap)
    per_slot = np.diff(cr.offsets)
    if max_occ in (0, 500):
        assert per_slot.max() > FAST_CAP, "some slot must take the slow path"
    if max_occ == 0:
        assert per_slot.max() >= 500
    assert (cr.hit_chain == g.CHAIN_NONE).sum() == ((cr.hits.hits["flags"] & g.HIT_SPANS) != 0).sum()


def test_entry_points_agree(world):
    import torch
    import genie_smem_b200 as g
    index = world["index"]
    eng, res = run(g, world, 2, g.METHOD_BWA)
    a = eng.chain_seeds()
    b = g.chain_seeds(index, res)
    for f in ("chains", "offsets", "hit_chain", "rec_offsets", "lengths"):
        assert np.array_equal(getattr(a, f), getattr(b, f)), f
    assert np.array_equal(a.hits.hits, b.hits.hits) and np.array_equal(a.hits.offsets, b.hits.offsets)
    asc = torch.from_numpy(np.frombuffer("".join(world["reads"]).encode(), np.uint8).reshape(len(world["reads"]), L).copy()).pin_memory()
    pipe = g.PipelinedEngine(index, len(world["reads"]), L, n_chunks=3, mems_per_read=64, recs_per_read=32, strands=2)
    pr = pipe.run_ascii(g.METHOD_BWA, asc, L, min_len=1)
    c = g.chain_seeds(index, pr)
    for f in ("chains", "offsets", "hit_chain", "rec_offsets", "lengths"):
        assert np.array_equal(getattr(a, f), getattr(c, f)), f
    # the accessors
    for i in (0, 7, len(world["reads"]) - 1):
        both = a.for_read(i)
        assert np.array_equal(both, a.chains[a.offsets[2 * i]:a.offsets[2 * i + 2]])
        assert len(a.for_read(i, 0)) + len(a.for_read(i, 1)) == len(both)
    for k in range(0, len(a), max(1, len(a) // 50)):
        m = a.seeds(k)
        assert len(m) == a.chains["n_seeds"][k] and (a.hits.hits["contig"][m] == a.chains["contig"][k]).all()
        assert a.hits.hits["offset"][m[0]] == a.chains["rbeg"][k]
    rc = a.read_coords()
    L_ = np.asarray(a.lengths)[rc["read"]]
    assert (rc["qend"] <= L_).all() and (rc["qbeg"] < rc["qend"]).all()
    one = eng.chain_seeds(max_occ=500, min_len=19)
    assert np.array_equal(one.chains, a.chains)
    with pytest.raises(ValueError):
        g.chain_seeds(world["sampled"], res, w=-1)


def test_best_places_simulated_reads(world):
    import genie_smem_b200 as g
    eng, res = run(g, world, 2, g.METHOD_BWA)
    cr = eng.chain_seeds()
    best = cr.best()
    assert len(best) == len(world["reads"])
    # the definition: heaviest chain over the read's slots, ties to the lower slot, then the earlier chain
    for i in range(0, len(world["reads"]), 37):
        ch = cr.chains[cr.offsets[2 * i]:cr.offsets[2 * i + 2]]
        assert best[i] == (-1 if len(ch) == 0 else cr.offsets[2 * i] + int(np.argmax(ch["weight"])))
    n_ok = n = 0
    for i, t in enumerate(world["truth"]):
        if t is None:
            continue
        n += 1
        k = best[i]
        if k < 0:
            continue
        c = cr.chains[k]
        q = int(c["q"]) & 0xFFFF
        n_ok += int(c["slot"]) & 1 == t[2] and int(c["contig"]) == t[0] and int(c["rbeg"]) - q == t[1]
    assert n > 700
    assert n_ok >= 0.99 * n, f"{n_ok} of {n} reads placed"


def test_refusals_and_out_cap(world):
    import torch
    import genie_smem_b200 as g
    from genie_smem_b200 import _capi as capi
    from genie_smem_b200 import engine as E
    index = world["index"]
    eng, res = run(g, world, 2, g.METHOD_BWA)
    want = eng.chain_seeds()
    dev = index.device
    n_rec = len(res.records)
    recs = eng.records
    off, offsets, hits, total = E._device_hits(index, recs, n_rec, 500, 19)
    n_slots = len(res.offsets) - 1
    rec_off = eng.rec_off
    ids = torch.empty(total, dtype=torch.int32, device=dev)
    cnt = torch.empty(n_slots, dtype=torch.int32, device=dev)
    coff = torch.empty(n_slots + 1, dtype=torch.int64, device=dev)
    need = C.c_uint64()
    capi.check(capi.lib.gsm_chains_workspace_info(n_slots, total, C.byref(need)))
    ws = torch.empty(int(need.value), dtype=torch.uint8, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    P = lambda t: C.c_void_p(t.data_ptr())                          # noqa: E731
    args = [P(recs), P(rec_off), n_slots, P(hits), P(off), total, 100, 10000, P(ids), P(cnt), P(coff), P(ws), int(need.value), stream]
    for k in (0, 1, 3, 4, 8, 9, 10, 11):                            # every pointer the call needs
        bad = list(args)
        bad[k] = None
        assert capi.lib.gsm_chain_seeds(*bad) == capi.E_INVALID, k
    short = list(args)
    short[12] = int(need.value) - 1
    assert capi.lib.gsm_chain_seeds(*short) == capi.E_CAPACITY
    capi.check(capi.lib.gsm_chain_seeds(*args))
    n_ch = int(coff[-1].item())
    assert n_ch == len(want.chains)
    cap = n_ch - 29
    out = torch.full(((n_ch + 16) * 8,), -1, dtype=torch.int32, device=dev)
    status = torch.zeros(1, dtype=torch.int64, device=dev)
    assert capi.lib.gsm_chains_collect(P(rec_off), n_slots, P(off), total, P(coff), P(ws), int(need.value) - 1, P(out), cap, P(status),
                                       stream) == capi.E_CAPACITY
    assert capi.lib.gsm_chains_collect(P(rec_off), n_slots, P(off), total, P(coff), P(ws), int(need.value), P(out), cap, None, stream) == capi.E_INVALID
    capi.check(capi.lib.gsm_chains_collect(P(rec_off), n_slots, P(off), total, P(coff), P(ws), int(need.value), P(out), cap, P(status), stream))
    o = out.cpu().numpy().view(np.uint32).reshape(-1, 8)
    assert int(status.item()) & 1
    assert np.array_equal(o[:cap], u32(want.chains, 8)[:cap])
    assert (o[cap:] == 0xFFFFFFFF).all()
    assert np.array_equal(ids.cpu().numpy().view(np.uint32), want.hit_chain)


def test_empty_batches(world):
    import genie_smem_b200 as g
    index = world["index"]
    empty = g.SmemResult(np.zeros(0, g.RECORD_DTYPE), np.zeros(4, np.int64), np.zeros(3, np.uint8), 0)
    cr = g.chain_seeds(index, empty)
    assert len(cr) == 0 and cr.offsets.tolist() == [0, 0, 0, 0] and cr.best().tolist() == [-1, -1, -1]
    eng, res = run(g, world, 1, g.METHOD_BWA)
    cr = eng.chain_seeds(min_len=1000)                              # records without hits
    assert len(cr) == 0 and len(cr.hits) == 0 and (cr.offsets == 0).all()
