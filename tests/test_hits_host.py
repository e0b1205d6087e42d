"""Hit expansion without a GPU: the reference reader (multi-record FASTA -> text + sequence table), the per-hit arithmetic
of csrc/hits_logic.cuh compiled with g++ against a numpy model of the documented semantics, and the C ABI of the hit
types."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "genie_smem_b200", "csrc")

SHIM = r"""
#include "hits_logic.cuh"
using namespace gsm;
// Host restatement of gsm_hits_count + gsm_hits_locate (full suffix array) from the kernels' own per-hit functions.
extern "C" uint64_t shim_hits(const uint32_t* rec, uint64_t n, uint32_t max_occ, uint32_t min_len, const uint32_t* sa,
                              const uint32_t* start, uint32_t n_entries, uint32_t* counts, uint32_t* out, uint64_t cap) {
    auto ld = [start](uint32_t i) { return start[i]; };
    uint64_t w = 0;
    for (uint64_t r = 0; r < n; ++r) {
        const uint32_t* q = rec + 4 * r;
        const uint32_t cnt = hit_rows(q[2], q[3]), len = hit_len(q[1]);
        const uint32_t nh = hit_count(cnt, len, max_occ, min_len), step = hit_step(cnt, max_occ);
        counts[r] = nh;
        for (uint32_t k = 0; k < nh; ++k, ++w) {
            const U4 h = make_hit(ld, n_entries, (uint32_t)r, sa[hit_row(q[2], k, step)] - 1u, len, hit_sampled(cnt, max_occ));
            if (w < cap) { out[4 * w] = h.x; out[4 * w + 1] = h.y; out[4 * w + 2] = h.z; out[4 * w + 3] = h.w; }
        }
    }
    return w;
}
extern "C" uint32_t shim_contig(const uint32_t* start, uint32_t n_entries, uint32_t p) {
    return contig_of([start](uint32_t i) { return start[i]; }, n_entries, p);
}
"""


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    d = tmp_path_factory.mktemp("hits_shim")
    src, lib = d / "shim.cpp", d / "libshim.so"
    src.write_text(SHIM)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", CSRC, str(src), "-o", str(lib)])
    so = C.CDLL(str(lib))
    P = C.c_void_p
    so.shim_hits.argtypes = [P, C.c_uint64, C.c_uint32, C.c_uint32, P, P, C.c_uint32, P, P, C.c_uint64]
    so.shim_hits.restype = C.c_uint64
    so.shim_contig.argtypes = [P, C.c_uint32, C.c_uint32]
    so.shim_contig.restype = C.c_uint32
    return so


def model_hits(recs, max_occ, min_len, sa, start):
    """The semantics, literally: records (n x 4 uint32: read, qstart | qend << 16, lo, hi) -> (counts, hits n x 4)."""
    counts, hits = [], []
    for r, (_, q, lo, hi) in enumerate(recs.tolist()):
        cnt = hi - lo + 1 if hi >= lo else 0
        ln = max((q >> 16) - (q & 0xFFFF), 0)
        n = 0 if ln < min_len else (min(cnt, max_occ) if max_occ else cnt)
        step = cnt // max_occ if (max_occ and cnt > max_occ) else 1
        counts.append(n)
        for k in range(n):
            p = int(sa[lo + k * step]) - 1
            c = int(np.searchsorted(start, p, side="right")) - 1
            off = p - int(start[c])
            flags = (1 if off + ln > int(start[c + 1]) - int(start[c]) else 0) | (2 if (max_occ and cnt > max_occ) else 0)
            hits.append((r, c, off, flags))
    return np.asarray(counts, np.uint32), np.asarray(hits, np.uint32).reshape(-1, 4)


def run_shim(shim, recs, max_occ, min_len, sa, start):
    recs = np.ascontiguousarray(recs, np.uint32)
    sa = np.ascontiguousarray(sa, np.uint32)
    start = np.ascontiguousarray(start, np.uint32)
    counts = np.zeros(max(len(recs), 1), np.uint32)
    cap = int(sum(min(int(h) - int(lo) + 1, max_occ or 1 << 40) for _, _, lo, h in recs.tolist() if h >= lo)) + 1
    out = np.zeros((cap, 4), np.uint32)
    n = shim.shim_hits(recs.ctypes.data, len(recs), max_occ, min_len, sa.ctypes.data, start.ctypes.data, len(start), counts.ctypes.data,
                       out.ctypes.data, cap)
    assert n < cap
    return counts[:len(recs)], out[:n]


def random_case(rng, n_seq, n_recs, n_rows_min=50):
    """A sequence table with empty sequences, a suffix array of random positions that hits every boundary, records."""
    lengths = rng.integers(0, 40, n_seq)
    lengths[rng.random(n_seq) < 0.3] = 0
    lengths[rng.integers(0, n_seq)] += 1
    start = np.concatenate(([0], np.cumsum(lengths))).astype(np.int64)
    n_bases = int(start[-1])
    n_rows = max(n_rows_min, 2 * n_bases)
    sa = rng.integers(1, n_bases + 1, n_rows).astype(np.uint32)
    # positions on boundaries: the first and last base of every non-empty sequence
    nz = np.flatnonzero(lengths > 0)
    edge = np.concatenate((start[nz] + 1, start[nz + 1]))
    sa[rng.choice(n_rows, min(len(edge), n_rows), replace=False)] = edge[:n_rows]
    lo = rng.integers(0, n_rows, n_recs)
    cnt = np.minimum(rng.geometric(0.05, n_recs), n_rows - lo)
    qs = rng.integers(0, 100, n_recs)
    qe = qs + rng.integers(1, 60, n_recs)
    recs = np.stack([np.arange(n_recs), qs | (qe << 16), lo, lo + cnt - 1], 1).astype(np.uint32)
    return recs, sa, start


@pytest.mark.parametrize("seed", range(6))
def test_hits_logic_equals_the_model(shim, seed):
    rng = np.random.default_rng(seed)
    recs, sa, start = random_case(rng, int(rng.integers(1, 40)), 300)
    cnts = recs[:, 3].astype(np.int64) - recs[:, 2] + 1
    c0 = int(cnts[0])
    for max_occ in (0, 1, 2, 3, 7, 500, c0, max(c0 - 1, 1)):
        for min_len in (0, 1, 19, 40):
            want_c, want_h = model_hits(recs, max_occ, min_len, sa, start)
            got_c, got_h = run_shim(shim, recs, max_occ, min_len, sa, start)
            assert np.array_equal(got_c, want_c), (max_occ, min_len)
            assert np.array_equal(got_h, want_h), (max_occ, min_len)
    # every flag combination occurs across the cases
    _, h = model_hits(recs, 3, 0, sa, start)
    assert set(np.unique(h[:, 3]).tolist()) == {0, 1, 2, 3}


def test_hits_logic_edge_records(shim):
    rng = np.random.default_rng(9)
    _, sa, start = random_case(rng, 12, 1, n_rows_min=600)
    n_rows = len(sa)
    # cnt == max_occ, cnt == max_occ + 1, a whole-index interval, one row, an inverted interval, qend < qstart, len 0
    rows = [(0, 20 << 16, 0, 499), (1, 0 | (30 << 16), 0, n_rows - 1), (2, 5 | (6 << 16), 17, 17), (3, 5 | (9 << 16), 9, 8),
            (4, 9 | (5 << 16), 3, 40), (5, 7 | (7 << 16), 3, 40), (6, 1 << 16, 100, 100 + 11)]
    recs = np.asarray(rows, np.uint32)
    for max_occ in (0, 1, 11, 12, 13, 499, 500, 501, n_rows, n_rows - 1):
        for min_len in (0, 1, 4):
            want = model_hits(recs, max_occ, min_len, sa, start)
            got = run_shim(shim, recs, max_occ, min_len, sa, start)
            assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), (max_occ, min_len)


def test_contig_search_on_large_tables(shim):
    """Start tables beyond the 8,192 entries the kernel keeps in shared memory, with runs of empty sequences."""
    rng = np.random.default_rng(3)
    for n_seq in (1, 2, 8191, 8192, 8193, 20000):
        lengths = rng.integers(0, 5, n_seq)
        lengths[-1] += 1
        start = np.concatenate(([0], np.cumsum(lengths))).astype(np.uint32)
        n_bases = int(start[-1])
        ps = np.unique(np.concatenate((rng.integers(0, n_bases, 3000), start[:-1][lengths > 0], start[1:][lengths > 0] - 1)))
        want = np.searchsorted(start, ps, side="right") - 1
        got = np.asarray([shim.shim_contig(start.ctypes.data, len(start), int(p)) for p in ps])
        assert np.array_equal(got, want), n_seq
        assert (lengths[got] > 0).all()              # never an empty sequence


def test_read_reference_multi_record(tmp_path):
    import genie_smem_b200 as g
    p = tmp_path / "ref.fa"
    p.write_bytes(b">chr1 first\r\nACGT\r\nAC\r\n>empty\r\n>one\r\nG\r\n>chr3\r\nTTTT\r\nA\r\n")
    text, ct = g.read_reference(str(p))
    assert text.dtype == np.uint8 and text.tobytes() == b"ACGTACGTTTTA"
    assert ct.names == ["chr1 first", "empty", "one", "chr3"]
    assert ct.start.dtype == np.uint32 and ct.start.tolist() == [0, 6, 6, 7, 12]
    assert ct.lengths.tolist() == [6, 0, 1, 5]
    assert ct.n_bases == len(text) and len(ct) == 4
    single = g.Contigs.single(12)
    assert single.names == [""] and single.start.tolist() == [0, 12]
    # headerless file: one sequence named ""
    q = tmp_path / "plain.fa"
    q.write_bytes(b"ACG\nT\n")
    text, ct = g.read_reference(str(q))
    assert text.tobytes() == b"ACGT" and ct == g.Contigs.single(4)


@pytest.mark.parametrize("body", [b">a\nACGT\n>b\nACNT\n", b">a\nACgT\n", b">a\r\nAC\r\n>b\r\nRY\r\n"])
def test_read_reference_rejects_non_acgt(tmp_path, body):
    import genie_smem_b200 as g
    p = tmp_path / "bad.fa"
    p.write_bytes(body)
    with pytest.raises(g.BaseError):
        g.read_reference(str(p))


def test_contigs_validation():
    import genie_smem_b200 as g
    with pytest.raises(ValueError):
        g.Contigs(["a"], [0, 5, 9])
    with pytest.raises(ValueError):
        g.Contigs(["a", "b"], [1, 5, 9])
    with pytest.raises(ValueError):
        g.Contigs(["a", "b"], [0, 5, 4])
    c = g.Contigs.from_lengths(["a", "b", "c"], [3, 0, 2])
    assert c.start.tolist() == [0, 3, 3, 5]


def test_hit_types_match_the_header(tmp_path):
    """gsm_hit / gsm_dev_contigs compile as C99 with the sizes and field offsets the bindings assume; the flag macros and
    the scratch-size query agree with Python."""
    from genie_smem_b200 import _capi as capi
    from genie_smem_b200.engine import HIT_DTYPE
    src = tmp_path / "hits_abi.c"
    src.write_text('#include "genie_smem.h"\n#include <stdio.h>\n#include <stddef.h>\n'
                   'int main(void) { uint64_t b = 0; int st = gsm_hits_workspace_info(100000, &b);\n'
                   '  printf("%zu %zu %zu %zu %zu %zu %u %u %d %llu\\n", sizeof(gsm_hit), offsetof(gsm_hit, contig), offsetof(gsm_hit, offset),\n'
                   '    offsetof(gsm_hit, flags), sizeof(gsm_dev_contigs), offsetof(gsm_dev_contigs, start), GSM_HIT_SPANS, GSM_HIT_SAMPLED,\n'
                   '    st, (unsigned long long)b); return 0; }\n')
    exe = tmp_path / "hits_abi"
    lib_dir = os.path.dirname(capi.LIB_PATH)
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                           "-L", lib_dir, "-lgenie_smem", f"-Wl,-rpath,{lib_dir}"])
    out = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    assert out[:6] == [16, 4, 8, 12, C.sizeof(capi.DevContigs), capi.DevContigs.start.offset]
    assert out[0] == C.sizeof(capi.Hit) == HIT_DTYPE.itemsize
    assert [capi.Hit.contig.offset, capi.Hit.offset.offset, capi.Hit.flags.offset] == out[1:4]
    assert [HIT_DTYPE.fields[f][1] for f in ("record", "contig", "offset", "flags")] == [0, 4, 8, 12]
    assert out[6:8] == [capi.HIT_SPANS, capi.HIT_SAMPLED]
    assert out[8] == 0 and out[9] >= 8 * (100000 // 2048 + 2)


def test_hit_entry_points_refuse_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from genie_smem_b200 import _capi as capi
    off = np.zeros(2, np.uint64)
    assert capi.lib.gsm_hits_count(None, 0, 500, 0, None, off.ctypes.data, None, 0, None) == capi.E_NODEVICE
    assert capi.lib.gsm_hits_locate(None, None, 0, None, None, None, 0, 0, 500, 0, None, 0, None, None) == capi.E_INVALID
