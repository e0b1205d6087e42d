"""Seed chaining without a GPU: a literal Python restatement of BWA-MEM's mem_chain / test_and_merge / mem_chain_weight
(the semantics of gsm_chain_seeds, include/genie_smem.h), pinned to hand-worked slots, and the per-seed rule of
csrc/chain_logic.cuh compiled with g++ against it on random seed lists built to reach every branch."""
import bisect
import ctypes as C
import os
import subprocess
from collections import Counter

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "genie_smem_b200", "csrc")

NONE, CONTAINED = 0xFFFFFFFF, 0x80000000
SPANS = 1


def bwa_test_and_merge(ch, qbeg, ln, rbeg, contig, w, max_gap, ev):
    """BWA's test_and_merge (no strand test): 1 contained, 2 appended, 0 failed.  ev counts the branches taken."""
    if contig != ch["contig"]:
        ev["other_contig"] += 1
        return 0
    first, last = ch["seeds"][0], ch["seeds"][-1]
    qend, rend = last[0] + last[1], last[2] + last[1]
    if qbeg >= first[0] and qbeg + ln <= qend and rbeg >= first[2] and rbeg + ln <= rend:
        ev["contained"] += 1
        return 1
    x, y = qbeg - last[0], rbeg - last[2]
    ok = y >= 0 and x - y <= w and y - x <= w and x - last[1] < max_gap and y - last[1] < max_gap
    if y < 0:
        ev["y<0"] += 1
    elif abs(x - y) == w:
        ev["|x-y|==w ok" if ok else "|x-y|==w"] += 1
    elif abs(x - y) == w + 1:
        ev["|x-y|==w+1"] += 1
    if y >= 0 and abs(x - y) <= w:
        for d in (x - last[1], y - last[1]):
            if d == max_gap - 1:
                ev["gap==max_gap-1"] += 1
            elif d == max_gap:
                ev["gap==max_gap"] += 1
    if ok:
        ch["seeds"].append((qbeg, ln, rbeg))
        ev["appended"] += 1
        return 2
    ev["failed"] += 1
    return 0


def chain_weight(seeds):
    """mem_chain_weight, literally."""
    def cover(key):
        w, end = 0, 0
        for s in seeds:
            b, e = key(s), key(s) + s[1]
            if b >= end:
                w += s[1]
            elif e > end:
                w += e - end
            end = max(end, e)
        return w
    w = min(cover(lambda s: s[0]), cover(lambda s: s[2]))
    return w if w < 1 << 30 else (1 << 30) - 1


def chain_slot(seeds, w, max_gap, ev):
    """mem_chain over one slot's seeds [(qbeg, len, rbeg, contig, flags)] -> (chains in output order, ids)."""
    table = []          # (contig, pos, creation index), kept sorted: ties on (contig, pos) stay in creation order
    chains = []         # creation order
    ids = []
    for qbeg, ln, rbeg, contig, flags in seeds:
        if flags & SPANS:
            ids.append(NONE)
            continue
        up = bisect.bisect_right(table, (contig, rbeg, 1 << 62))
        res = 0
        if up:
            c, p, _ = table[up - 1]
            lo = bisect.bisect_left(table, (c, p, -1))          # the first created chain of the lower key
            if lo != up - 1:
                ev["tie"] += 1
            cid = table[lo][2]
            res = bwa_test_and_merge(chains[cid], qbeg, ln, rbeg, contig, w, max_gap, ev)
            if res:
                ids.append(cid | (CONTAINED if res == 1 else 0))
        else:
            ev["no_lower"] += 1
        if not res:
            cid = len(chains)
            chains.append({"contig": contig, "seeds": [(qbeg, ln, rbeg)]})
            bisect.insort(table, (contig, rbeg, cid))
            ids.append(cid)
    rank = {t[2]: k for k, t in enumerate(table)}
    ids = [i if i == NONE else (i & CONTAINED) | rank[i & ~CONTAINED] for i in ids]
    return [chains[t[2]] for t in table], ids


def oracle_chains(recs, rec_off, hits, hit_off, w=100, max_gap=10000, ev=None):
    """The whole batch: recs (n x 4 u32: read, qstart | qend << 16, lo, hi), rec_off per slot, hits (n x 4 u32: record,
    contig, offset, flags), hit_off per record -> (chains n x 8 u32, chain_off int64, hit_chain u32)."""
    ev = Counter() if ev is None else ev
    out, off, hit_chain = [], [0], np.full(len(hits), NONE, np.uint32)
    for s in range(len(rec_off) - 1):
        seeds, where = [], []
        for r in range(int(rec_off[s]), int(rec_off[s + 1])):
            y = int(recs[r][1])
            qs, qe = y & 0xFFFF, y >> 16
            for h in range(int(hit_off[r]), int(hit_off[r + 1])):
                seeds.append((qs, max(qe - qs, 0), int(hits[h][2]), int(hits[h][1]), int(hits[h][3])))
                where.append(h)
        chains, ids = chain_slot(seeds, w, max_gap, ev)
        hit_chain[where] = np.asarray(ids, np.uint32)
        for ch in chains:
            sd = ch["seeds"]
            q = min(x[0] for x in sd) | (max(x[0] + x[1] for x in sd) << 16)
            out.append((s, ch["contig"], sd[0][2], max(x[2] + x[1] for x in sd), q, chain_weight(sd), len(sd), 0))
        off.append(off[-1] + len(chains))
    return np.asarray(out, np.uint32).reshape(-1, 8), np.asarray(off, np.int64), hit_chain


def one_record_per_seed(slots):
    """slots: list of seed lists [(qbeg, len, rbeg, contig, flags)] -> (recs, rec_off, hits, hit_off), one record and hit per seed."""
    recs, hits, rec_off = [], [], [0]
    for s, seeds in enumerate(slots):
        for qbeg, ln, rbeg, contig, flags in seeds:
            hits.append((len(recs), contig, rbeg, flags))
            recs.append((s, qbeg | ((qbeg + ln) << 16), 0, 0))
        rec_off.append(len(recs))
    return (np.asarray(recs, np.uint32).reshape(-1, 4), np.asarray(rec_off, np.uint64), np.asarray(hits, np.uint32).reshape(-1, 4),
            np.arange(len(hits) + 1, dtype=np.uint64))


def Q(a, b):
    return a | b << 16


HAND = [
    # A: contained, appended, a chain before the first one, a fail on the diagonal test (w = 100)
    ([(0, 30, 1000, 0, 0), (10, 15, 1010, 0, 0), (40, 20, 1045, 0, 0), (5, 20, 500, 0, 0), (70, 25, 1300, 0, 0)],
     [(500, 520, Q(5, 25), 20, 1), (1000, 1065, Q(0, 60), 50, 2), (1300, 1325, Q(70, 95), 25, 1)],
     [1, CONTAINED | 1, 1, 0, 2]),
    # B: two chains share pos 100 on sequence 1; the seed at 105 is tested against the one created first (it fails there,
    # though it would extend the second); a spanning hit; a chain on an earlier sequence
    ([(0, 20, 100, 1, 0), (50, 20, 300, 1, 0), (150, 20, 100, 1, 0), (160, 10, 105, 1, 0), (3, 40, 7, 2, SPANS), (0, 20, 50, 0, 0)],
     [(50, 70, Q(0, 20), 20, 1), (100, 120, Q(0, 20), 20, 1), (100, 120, Q(150, 170), 20, 1), (105, 115, Q(160, 170), 10, 1),
      (300, 320, Q(50, 70), 20, 1)],
     [1, 4, 2, 3, NONE, 0]),
    # C: overlapping members, one of them before the first seed on the query (weight = min(40, 55))
    ([(20, 30, 1000, 0, 0), (30, 30, 1012, 0, 0), (10, 25, 1030, 0, 0)],
     [(1000, 1055, Q(10, 60), 40, 3)],
     [0, 0, 0]),
    # D: no hits at all
    ([], [], []),
]


def test_oracle_on_hand_worked_slots():
    slots = [h[0] for h in HAND]
    recs, rec_off, hits, hit_off = one_record_per_seed(slots)
    chains, off, ids = oracle_chains(recs, rec_off, hits, hit_off)
    contig = [[0, 0, 0], [0, 1, 1, 1, 1], [0], []]         # sequence of each chain, slot by slot
    want = [[s, contig[s][k], *c, 0] for s, (_, cs, _) in enumerate(HAND) for k, c in enumerate(cs)]
    assert chains.tolist() == want
    assert off.tolist() == [0, 3, 8, 9, 9]
    assert ids.tolist() == [i for h in HAND for i in h[2]]


SHIM = r"""
#include "chain_logic.cuh"
#include <vector>
using namespace gsm;
// Host table over vectors, the shape of the kernels' tables (a view: copies share the vectors)
struct VecTable {
    std::vector<uint32_t>* order;
    std::vector<ChainState>* st;
    uint32_t n;
    uint64_t key(uint32_t i) const { const ChainState& c = (*st)[(*order)[i]]; return chain_key(c.contig, c.pos); }
    uint32_t id(uint32_t i) const { return (*order)[i]; }
    ChainState load(uint32_t id) const { return (*st)[id]; }
    void store(uint32_t id, const ChainState& c) const { (*st)[id] = c; }
    void insert(uint32_t i, const ChainState& c) { order->insert(order->begin() + i, n); st->push_back(c); ++n; }
};
// gsm_chain_seeds + gsm_chains_collect on the host from the kernels' per-seed rule: a slot that needs more than cap chains
// starts over without a cap, as the kernels' slow path does.
extern "C" uint64_t shim_chains(const uint32_t* recs, const uint64_t* rec_off, uint64_t n_slots, const uint32_t* hits, const uint64_t* hit_off,
                                uint32_t w, uint32_t max_gap, uint32_t cap, uint32_t* hit_chain, uint64_t* chain_off, uint32_t* out, uint64_t out_cap,
                                uint64_t* n_slow) {
    uint64_t total = 0;
    chain_off[0] = 0;
    for (uint64_t s = 0; s < n_slots; ++s) {
        std::vector<uint32_t> order;
        std::vector<ChainState> st;
        VecTable t{&order, &st, 0u};
        for (int pass = 0; pass < 2; ++pass) {
            bool full = false;
            for (uint64_t r = rec_off[s]; r < rec_off[s + 1] && !full; ++r) {
                const uint32_t y = recs[4 * r + 1], qs = y & 0xFFFFu, qe = y >> 16;
                for (uint64_t h = hit_off[r]; h < hit_off[r + 1]; ++h) {
                    uint32_t id = CHAIN_NONE;
                    if (!(hits[4 * h + 3] & 1u)) {
                        ChainSeed sd{qs, qe > qs ? qe - qs : 0u, hits[4 * h + 2], hits[4 * h + 1]};
                        id = chain_step(t, sd, w, max_gap, pass ? 0xFFFFFFFFu : cap);
                        if (id == CHAIN_FULL) { full = true; break; }
                    }
                    hit_chain[h] = id;
                }
            }
            if (!full) break;
            ++*n_slow;
            order.clear(); st.clear(); t.n = 0;
        }
        std::vector<uint32_t> rank(t.n);
        for (uint32_t k = 0; k < t.n; ++k) {
            rank[t.id(k)] = k;
            if (total + k < out_cap) chain_output(t.load(t.id(k)), (uint32_t)s, out + 8 * (total + k));
        }
        if (rec_off[s] < rec_off[s + 1])
            for (uint64_t h = hit_off[rec_off[s]]; h < hit_off[rec_off[s + 1]]; ++h)
                if (hit_chain[h] != CHAIN_NONE) hit_chain[h] = (hit_chain[h] & CHAIN_CONTAINED) | rank[hit_chain[h] & ~CHAIN_CONTAINED];
        total += t.n;
        chain_off[s + 1] = total;
    }
    return total;
}
"""


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    d = tmp_path_factory.mktemp("chains_shim")
    src, lib = d / "shim.cpp", d / "libshim.so"
    src.write_text(SHIM)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", CSRC, str(src), "-o", str(lib)])
    so = C.CDLL(str(lib))
    P = C.c_void_p
    so.shim_chains.argtypes = [P, P, C.c_uint64, P, P, C.c_uint32, C.c_uint32, C.c_uint32, P, P, P, C.c_uint64, P]
    so.shim_chains.restype = C.c_uint64
    return so


def run_shim(shim, recs, rec_off, hits, hit_off, w, max_gap, cap=8):
    recs, hits = np.ascontiguousarray(recs, np.uint32), np.ascontiguousarray(hits, np.uint32)
    rec_off, hit_off = np.ascontiguousarray(rec_off, np.uint64), np.ascontiguousarray(hit_off, np.uint64)
    n_slots = len(rec_off) - 1
    ids = np.full(max(len(hits), 1), 0x12345678, np.uint32)
    off = np.zeros(n_slots + 1, np.uint64)
    out = np.zeros((max(len(hits), 1), 8), np.uint32)
    slow = np.zeros(1, np.uint64)
    n = shim.shim_chains(recs.ctypes.data, rec_off.ctypes.data, n_slots, hits.ctypes.data, hit_off.ctypes.data, w, max_gap, cap,
                         ids.ctypes.data, off.ctypes.data, out.ctypes.data, len(out), slow.ctypes.data)
    return out[:n], off.astype(np.int64), ids[:len(hits)], int(slow[0])


def random_batch(rng, n_slots, w, max_gap):
    """Slots of several records, each with a few hits: a few diagonals per slot on up to three sequences, offsets nudged by
    exactly w, w + 1, max_gap - 1 and max_gap, repeated positions, spanning hits, slots without hits."""
    recs, hits, rec_off, hit_off = [], [], [0], [0]
    for s in range(n_slots):
        n_rec = 0 if rng.random() < 0.1 else int(rng.integers(1, 12))
        diags = [(int(rng.integers(0, 3)), int(rng.integers(0, 400))) for _ in range(int(rng.integers(1, 4)))]
        for _ in range(n_rec):
            qs = int(rng.integers(0, 140))
            ln = int(rng.integers(1, 40))
            recs.append((s, qs | ((qs + ln) << 16), 0, 0))
            for _ in range(int(rng.integers(0, 5))):
                contig, d = diags[int(rng.integers(0, len(diags)))]
                r = d + qs
                u = rng.random()
                if u < 0.15:
                    r += int(rng.choice([w, w + 1, -w, -w - 1, max_gap - 1, max_gap, max_gap + ln - 1, max_gap + ln]))
                elif u < 0.3:
                    r = d                                   # the same position again: ties on pos
                elif u < 0.4:
                    r += int(rng.integers(-60, 60))
                flags = SPANS if rng.random() < 0.05 else 0
                hits.append((len(recs) - 1, contig, max(r, 0), flags))
            hit_off.append(len(hits))
        rec_off.append(len(recs))
    return (np.asarray(recs, np.uint32).reshape(-1, 4), np.asarray(rec_off, np.uint64), np.asarray(hits, np.uint32).reshape(-1, 4),
            np.asarray(hit_off, np.uint64))


@pytest.mark.parametrize("w,max_gap", [(100, 10000), (0, 1), (5, 30), (20, 200)])
def test_chain_logic_equals_the_oracle(shim, w, max_gap):
    ev = Counter()
    slow = 0
    for seed in range(12):
        rng = np.random.default_rng(1000 * w + seed)
        recs, rec_off, hits, hit_off = random_batch(rng, 60, w, max_gap)
        want = oracle_chains(recs, rec_off, hits, hit_off, w, max_gap, ev)
        for cap in (8, 1 << 30):
            got = run_shim(shim, recs, rec_off, hits, hit_off, w, max_gap, cap)
            assert np.array_equal(got[0], want[0]), (seed, cap)
            assert np.array_equal(got[1], want[1]), (seed, cap)
            assert np.array_equal(got[2], want[2]), (seed, cap)
            slow += got[3] if cap == 8 else 0
    assert slow > 0, "some slot must need more than 8 chains"
    needed = ["contained", "appended", "failed", "other_contig", "no_lower", "tie", "y<0", "|x-y|==w+1"]
    if w >= 5 and max_gap <= 100:
        # a gap of max_gap on both axes only fits on a read when max_gap is short
        needed += ["gap==max_gap-1", "gap==max_gap"]
    missing = [k for k in needed if ev[k] == 0]
    assert not missing, (missing, dict(ev))
    assert ev["|x-y|==w ok"] + ev["|x-y|==w"] > 0, dict(ev)


def test_chain_logic_pinned_slots(shim):
    slots = [h[0] for h in HAND]
    recs, rec_off, hits, hit_off = one_record_per_seed(slots)
    want = oracle_chains(recs, rec_off, hits, hit_off)
    for cap in (1, 2, 8):
        got = run_shim(shim, recs, rec_off, hits, hit_off, 100, 10000, cap)
        assert all(np.array_equal(a, b) for a, b in zip(got[:3], want)), cap


def test_many_chains_in_one_slot(shim):
    """A 500-copy repeat: one record with 700 hits on distinct far-apart positions gives 700 chains in its slot."""
    rng = np.random.default_rng(5)
    pos = rng.permutation(700) * 20_000
    hits = np.stack([np.zeros(700), pos % 3, pos, np.zeros(700)], 1).astype(np.uint32)
    recs = np.asarray([(0, Q(10, 60), 0, 699), (0, Q(70, 100), 0, 0)], np.uint32)
    hits = np.concatenate((hits, [(1, 1, 60, 0)])).astype(np.uint32)
    rec_off, hit_off = np.asarray([0, 2], np.uint64), np.asarray([0, 700, 701], np.uint64)
    want = oracle_chains(recs, rec_off, hits, hit_off)
    got = run_shim(shim, recs, rec_off, hits, hit_off, 100, 10000)
    assert got[3] == 1 and len(want[0]) == 701
    assert all(np.array_equal(a, b) for a, b in zip(got[:3], want))


def test_chain_types_match_the_header(tmp_path):
    """gsm_chain compiles as C99 with 32 bytes and the field offsets CHAIN_DTYPE and the bindings assume; the id macros agree."""
    from genie_smem_b200 import _capi as capi
    from genie_smem_b200.engine import CHAIN_DTYPE
    src = tmp_path / "chains_abi.c"
    src.write_text('#include "genie_smem.h"\n#include <stdio.h>\n#include <stddef.h>\n'
                   'int main(void) { uint64_t b = 0; int st = gsm_chains_workspace_info(1000, 5000, &b);\n'
                   '  printf("%zu %zu %zu %zu %zu %zu %zu %zu %u %u %d %llu\\n", sizeof(gsm_chain), offsetof(gsm_chain, contig),\n'
                   '    offsetof(gsm_chain, rbeg), offsetof(gsm_chain, rend), offsetof(gsm_chain, q), offsetof(gsm_chain, weight),\n'
                   '    offsetof(gsm_chain, n_seeds), offsetof(gsm_chain, reserved), GSM_CHAIN_NONE, GSM_CHAIN_CONTAINED, st,\n'
                   '    (unsigned long long)b); return 0; }\n')
    exe = tmp_path / "chains_abi"
    lib_dir = os.path.dirname(capi.LIB_PATH)
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                           "-L", lib_dir, "-lgenie_smem", f"-Wl,-rpath,{lib_dir}"])
    out = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    assert out[0] == 32 == C.sizeof(capi.Chain) == CHAIN_DTYPE.itemsize
    names = ("contig", "rbeg", "rend", "q", "weight", "n_seeds", "reserved")
    assert out[1:8] == [getattr(capi.Chain, f).offset for f in names] == [CHAIN_DTYPE.fields[f][1] for f in names] == [4, 8, 12, 16, 20, 24, 28]
    assert out[8:10] == [capi.CHAIN_NONE, capi.CHAIN_CONTAINED] == [NONE, CONTAINED]
    assert out[10] == 0 and out[11] >= 84 * 5000


def test_chain_entry_points_refuse_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from genie_smem_b200 import _capi as capi
    off = np.zeros(2, np.uint64)
    assert capi.lib.gsm_chain_seeds(None, None, 0, None, None, 0, 100, 10000, None, None, off.ctypes.data, None, 0, None) == capi.E_NODEVICE
    assert capi.lib.gsm_chain_seeds(None, None, 1, None, None, 0, 100, 10000, None, None, off.ctypes.data, None, 0, None) == capi.E_INVALID
    assert capi.lib.gsm_chains_collect(None, 0, None, 0, None, None, 0, None, 0, None, None) == capi.E_INVALID
