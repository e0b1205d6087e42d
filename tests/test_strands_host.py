"""Strand-doubled batches without a GPU: the per-word arithmetic of csrc/strand_logic.cuh compiled with g++ and run the way
k_both_strands runs it, against gsm_pack_reads of the interleaved strings [r0, rc(r0), r1, rc(r1), ...]; the entry point's
argument checks."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "genie_smem_b200", "csrc")

LENGTHS = [0, 1, 15, 16, 17, 63, 64, 65, 151, 1024, 1025, 65535]

SHIM = r"""
#include "strand_logic.cuh"
using namespace gsm;
// Host restatement of k_both_strands over reads [0, n) of a (possibly offset) view: same functions, same word loop.
extern "C" void shim_both_strands(const uint32_t* src, const uint32_t* chunk_off, const uint32_t* len, uint64_t n, uint32_t* dst,
                                  uint32_t* chunk_off_out, uint32_t* len_out) {
    const uint32_t c0 = chunk_off[0];
    const uint32_t end = 2u * (chunk_off[n] - c0);
    chunk_off_out[2 * n] = end;
    for (int k = 0; k < 4; ++k) dst[4ull * end + k] = 0u;
    for (uint64_t r = 0; r < n; ++r) {
        const uint32_t a = chunk_off[r] - c0, nch = chunk_off[r + 1] - c0 - a;
        const uint32_t L0 = len[r], L = L0 < nch * 64u ? L0 : nch * 64u;
        chunk_off_out[2 * r] = 2u * a;
        chunk_off_out[2 * r + 1] = 2u * a + nch;
        len_out[2 * r] = len_out[2 * r + 1] = L0;
        const uint32_t* s = src + (uint64_t)(a + c0) * 4u;
        uint32_t* fwd = dst + (uint64_t)a * 8u;
        uint32_t* rc = fwd + (uint64_t)nch * 4u;
        for (uint32_t w = 0; w < nch * 4u; ++w) {
            const uint32_t m = strand_word_mask(L, w);
            fwd[w] = m ? s[w] & m : 0u;
            StrandSrc q;
            uint32_t v = 0u;
            if (strand_rc_src(L, w, &q)) {
                const uint32_t hi = q.q >= 0 ? s[q.q] : 0u;
                const uint32_t lo = q.sh ? s[q.q + 1] : 0u;
                v = strand_rc_word(hi, lo, q.sh, L, w);
            }
            rc[w] = v;
        }
    }
}
extern "C" uint32_t shim_reverse_fields(uint32_t x) { return strand_reverse_fields(x); }
"""


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    d = tmp_path_factory.mktemp("strand_shim")
    src, lib = d / "shim.cpp", d / "libshim.so"
    src.write_text(SHIM)
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", CSRC, str(src), "-o", str(lib)])
    so = C.CDLL(str(lib))
    P = C.c_void_p
    so.shim_both_strands.argtypes = [P, P, P, C.c_uint64, P, P, P]
    so.shim_both_strands.restype = None
    so.shim_reverse_fields.argtypes = [C.c_uint32]
    so.shim_reverse_fields.restype = C.c_uint32
    return so


def rc(s):
    return s[::-1].translate(str.maketrans("ACGT", "TGCA"))


def host_pack(reads):
    """gsm_pack_reads of `reads` -> (packed uint32 words incl. the zero pad chunk, chunk_off, lens)."""
    from genie_smem_b200 import _capi as capi
    lens = np.asarray([len(r) for r in reads], np.uint32)
    joined = "".join(reads).encode()
    off = np.zeros(len(reads) + 1, np.uint32)
    capi.check(capi.lib.gsm_pack_reads(joined, lens.ctypes.data, len(reads), off.ctypes.data, None))
    packed = np.zeros(int(off[-1]) * 4 + 4, np.uint32)
    capi.check(capi.lib.gsm_pack_reads(joined, lens.ctypes.data, len(reads), off.ctypes.data, packed.ctypes.data))
    return packed, off, lens


def doubled(shim, packed, off, lens, lo, hi):
    """The shim on the view of reads [lo, hi) of a packed batch; output buffers poisoned first."""
    n = hi - lo
    c = off[lo:hi + 1]
    words = 2 * int(c[-1] - c[0]) * 4 + 4
    out = np.full(words, 0xDEADBEEF, np.uint32)
    coff = np.full(2 * n + 1, 0xDEADBEEF, np.uint32)
    lout = np.full(max(2 * n, 1), 0xDEADBEEF, np.uint32)
    c = np.ascontiguousarray(c)
    ln = np.ascontiguousarray(lens[lo:hi]) if n else np.zeros(1, np.uint32)
    shim.shim_both_strands(packed.ctypes.data, c.ctypes.data, ln.ctypes.data, n, out.ctypes.data, coff.ctypes.data, lout.ctypes.data)
    return out, coff, lout[:2 * n]


def interleave(reads):
    return [s for r in reads for s in (r, rc(r))]


def random_reads(rng, lengths):
    return ["".join("ACGT"[c] for c in rng.integers(0, 4, int(n))) for n in lengths]


def test_reverse_fields(shim):
    rng = np.random.default_rng(0)
    for x in rng.integers(0, 1 << 32, 200, dtype=np.uint64).tolist() + [0, 0xFFFFFFFF, 0x1B000000]:
        fields = [(x >> (30 - 2 * t)) & 3 for t in range(16)]
        want = sum(f << (30 - 2 * t) for t, f in enumerate(reversed(fields)))
        assert shim.shim_reverse_fields(int(x)) == want


def test_doubled_batch_equals_host_pack_of_interleaved_strings(shim):
    rng = np.random.default_rng(1)
    reads = random_reads(rng, LENGTHS)
    half = "".join("ACGT"[c] for c in rng.integers(0, 4, 40))
    reads.append(half + rc(half))                                  # a palindrome: equal to its own reverse complement
    assert reads[-1] == rc(reads[-1])
    packed, off, lens = host_pack(reads)
    want_p, want_o, want_l = host_pack(interleave(reads))
    got_p, got_o, got_l = doubled(shim, packed, off, lens, 0, len(reads))
    assert np.array_equal(got_o, want_o)
    assert np.array_equal(got_l, want_l)
    assert np.array_equal(got_p, want_p)                            # including the zero pad bits and the zero pad chunk
    # slot 2i+1 of the palindrome is byte-identical to slot 2i
    i = len(reads) - 1
    a, b, e = (int(x) for x in got_o[2 * i:2 * i + 3])
    assert np.array_equal(got_p[4 * a:4 * b], got_p[4 * b:4 * e])


@pytest.mark.parametrize("lo,hi", [(3, 9), (1, 2), (5, 5), (0, 13), (11, 13)])
def test_views_with_a_nonzero_first_offset(shim, lo, hi):
    rng = np.random.default_rng(2)
    reads = random_reads(rng, LENGTHS + [151])
    packed, off, lens = host_pack(reads)
    want_p, want_o, want_l = host_pack(interleave(reads[lo:hi]))
    got_p, got_o, got_l = doubled(shim, packed, off, lens, lo, hi)
    assert np.array_equal(got_o, want_o) and np.array_equal(got_l, want_l) and np.array_equal(got_p, want_p)


def test_many_random_lengths(shim):
    rng = np.random.default_rng(3)
    reads = random_reads(rng, rng.integers(0, 300, 400))
    packed, off, lens = host_pack(reads)
    want = host_pack(interleave(reads))
    got = doubled(shim, packed, off, lens, 0, len(reads))
    for g, w in zip(got, want):
        assert np.array_equal(g, w)


def test_entry_point_refuses_without_gpu_and_checks_arguments():
    import torch
    from genie_smem_b200 import _capi as capi
    buf = np.zeros(64, np.uint32)
    r = capi.DevReads()
    r.n_reads, r.packed, r.chunk_off, r.len, r.max_len, r.read_id_base = 1, buf.ctypes.data, buf.ctypes.data, buf.ctypes.data, 151, 0
    p = buf.ctypes.data
    f = capi.lib.gsm_reads_both_strands_device
    assert f(None, p, p, p, None) == capi.E_INVALID
    assert f(C.byref(r), None, p, p, None) == capi.E_INVALID
    assert f(C.byref(r), p, None, p, None) == capi.E_INVALID
    assert f(C.byref(r), p, p, None, None) == capi.E_INVALID
    r0 = capi.DevReads()
    r0.n_reads, r0.packed, r0.chunk_off, r0.len = 1, None, p, p
    assert f(C.byref(r0), p, p, p, None) == capi.E_INVALID
    big = capi.DevReads()
    big.n_reads, big.packed, big.chunk_off, big.len, big.max_len = 1 << 26, p, p, p, 65535      # 2 * 2^26 * 1024 chunks
    assert f(C.byref(big), p, p, p, None) == capi.E_CAPACITY
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    assert f(C.byref(r), p, p, p, None) == capi.E_NODEVICE


def test_result_views_of_a_strand_doubled_batch():
    """SmemResult / HitResult of a strand-doubled batch, built by hand: slot ranges per read and strand, and read_coords()
    in the original read's orientation."""
    import genie_smem_b200 as g
    # read_id_base 5.  read 0 (L = 10): slot 0 has records [0, 4), [3, 10); slot 1 has [2, 7).  read 1 (L = 6): [0, 6) and [1, 6)
    rows = [(2 * 5 + 0, 0, 4), (2 * 5 + 0, 3, 10), (2 * 5 + 1, 2, 7), (2 * 6 + 0, 0, 6), (2 * 6 + 1, 1, 6)]
    recs = np.zeros(len(rows), g.RECORD_DTYPE)
    for k, (rid, a, b) in enumerate(rows):
        recs[k] = (rid, a, b, k, k)
    offs = np.asarray([0, 2, 3, 4, 5], np.int64)
    res = g.SmemResult(recs, offs, np.zeros(4, np.uint8), 0, strands=2, lengths=np.asarray([10, 6], np.uint32))
    assert res.for_read(0)["sa_lo"].tolist() == [0, 1, 2]
    assert res.for_read(0, 0)["sa_lo"].tolist() == [0, 1] and res.for_read(0, 1)["sa_lo"].tolist() == [2]
    assert res.for_read(1, 1)["sa_lo"].tolist() == [4]
    co = res.read_coords()
    assert co["read"].tolist() == [5, 5, 5, 6, 6] and co["strand"].tolist() == [0, 0, 1, 0, 1]
    assert co["qbeg"].tolist() == [0, 3, 3, 0, 0] and co["qend"].tolist() == [4, 10, 8, 6, 5]
    hits = g.HitResult(np.zeros(7, g.HIT_DTYPE), np.asarray([0, 1, 3, 4, 6, 7], np.int64))
    assert len(hits.for_read(res, 0)) == 4 and len(hits.for_read(res, 0, 1)) == 1 and len(hits.for_read(res, 1, 0)) == 2
    with pytest.raises(ValueError):
        res.for_read(0, 2)
    one = g.SmemResult(recs[:2], np.asarray([0, 2], np.int64), np.zeros(1, np.uint8), 0)
    assert one.strands == 1 and len(one.for_read(0)) == 2 and len(one.for_read(0, 0)) == 2
    assert one.read_coords()["qbeg"].tolist() == [0, 3]
    with pytest.raises(ValueError):
        one.for_read(0, 1)
