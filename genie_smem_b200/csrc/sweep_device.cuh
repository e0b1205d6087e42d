// Device side of the sweep kernel.
//   k_sweep1: ONE LANE PER READ, 32 reads in flight per warp.  Every iteration each lane runs its per-read control
//   (sweep_logic.cuh: registers and shared memory only) and then the whole warp executes ONE uniform memory section -- a
//   predicated seed-table fetch, a predicated suffix-array / text fetch, and the two 256-bit loads of one rank bucket with
//   the bit-plane masks built once and popcounted below both offsets (lane_step) -- so all 32 chains' fetches are in flight
//   together.  Finished reads hand their matches to the pool cooperatively (flush_finished): one atomic per warp,
//   coalesced copies, lists of up to 64 matches ordered and stored field by field, the BWA-SMEM picks of lists of up to 32
//   made on the way.
//   One lane per read measured fastest: 187 M reads/s against 103 M for two lanes per read (one bucket half each) and
//   78 M for four lanes with 128-bit loads on the same bench (profiles/r01_notes.md, r02_notes.md).
#pragma once
#include <cuda_runtime.h>

#include "sweep_logic.cuh"

namespace gsm {

// mem_cnt[read]: number of maximal matches in the low 30 bits, and how the sweep left the list
constexpr uint32_t MEMS_ORDERED = 0x80000000u;   // ascending and field by field (n start|end words, n lo, n count, n sweep ordinals)
constexpr uint32_t MEMS_PICKED = 0x40000000u;    // ... and the first sweep ordinal replaced by the BWA-SMEM picks (bit = position)
constexpr uint32_t MEMS_COUNT = 0x3FFFFFFFu;

struct SweepArgs {
    const uint4* fwd;
    const uint4* rev;
    IndexMeta meta;
    const uint4* reads;
    const uint32_t* chunk_off;
    const uint32_t* len;
    uint32_t n_reads;
    uint32_t max_len;
    const uint4* seed_tab;   // optional 4^seed_K x {fwd lo, count, rev lo, 0} (gsm_seed_table_build), else NULL
    uint32_t seed_K;
    uint4* mem_pool;
    unsigned long long mem_cap;
    uint32_t* mem_off;
    uint32_t* mem_cnt;
    uint4* scratch;          // per lane: [0, max_len) match staging, [max_len, 2 max_len) candidate spill
    unsigned long long* counters;
    const uint32_t* sa;      // unique-match shortcut (k_sweep1<.., true>): suffix array (1-based values) ...
    const uint32_t* text;    // ... and the 2-bit packed text (MSB-first, readable 2 words past its end)
    uint32_t n_bases;
};

// Shared memory: [per lane: SWEEP1_CAP candidates of 16 B {end, lo, cnt, -}, then (short reads) the read's packed
// words][16 B pad] (sweep1_lane_u4).  Indexed through one extern array so that the compiler emits LDS/STS.
extern __shared__ uint4 g_sweep_smem[];

// one 32-byte half of a bucket: a single 256-bit read-only load
__device__ __forceinline__ Half ldg_half(const uint4* halves_base, size_t half_index) {
    Half h;
    asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(h.c0), "=r"(h.c1), "=r"(h.l0), "=r"(h.l1), "=r"(h.l2), "=r"(h.h0), "=r"(h.h1), "=r"(h.h2)
                 : "l"(halves_base + half_index * 2));
    return h;
}

// One FM extension step by a lane pair (k_backsearch, k_add_one), all pairs of the warp together: each lane of a pair
// loads one half of the bucket and the halves' counts are summed with shuffles.  Every lane passes its pair's operands;
// `active` pairs get their result, inactive ones issue no loads.  g = lane within pair.
__device__ __forceinline__ StepOut pair_step(const uint4* __restrict__ bk, uint32_t P0, uint32_t P1, uint32_t ch, uint32_t Cc,
                                             uint32_t primary, uint32_t g, bool active) {
    constexpr uint32_t FULLM = 0xFFFFFFFFu;
    uint32_t b0, r0, b1, r1;
    split192(P0, b0, r0);
    split192(P1, b1, r1);
    Half v0 = Half{0, 0, 0, 0, 0, 0, 0, 0}, v1;
    if (active) v0 = ldg_half(bk, (size_t)b0 * 2 + g);
    v1 = v0;
    if (active && b1 != b0) v1 = ldg_half(bk, (size_t)b1 * 2 + g);
    const SymK k = sym_consts(ch);
    uint32_t packed = half_counts(v0, r0, k, g) | (half_counts(v1, r1, k, g) << 16);
    uint32_t he0, hl0, he1, hl1;
    half_header(v0, ch, g, he0, hl0);
    half_header(v1, ch, g, he1, hl1);
    uint32_t A = he0, B = he1, D = hl1 - hl0;
    packed += __shfl_xor_sync(FULLM, packed, 1);
    A += __shfl_xor_sync(FULLM, A, 1);
    B += __shfl_xor_sync(FULLM, B, 1);
    D += __shfl_xor_sync(FULLM, D, 1);
    const uint32_t eq0 = A + (packed & 0xFFu);
    const uint32_t eq1 = B + ((packed >> 16) & 0xFFu);
    const uint32_t ltd = D + ((packed >> 24) & 0xFFu) - ((packed >> 8) & 0xFFu);
    return finish_step(eq0, eq1, ltd, P0, P1, ch, Cc, primary);
}

// one 16-byte seed-table entry (read-only path; volatile so that it is issued before the bucket loads' consumers)
__device__ __forceinline__ uint4 ldg_seed(const uint4* p) {
    uint4 v;
    asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}

// ------------------------------------------------------------------------------------------------ one lane per read
// Every lane fetches whole 64-byte buckets itself (two 256-bit loads) and popcounts all 192 symbols, so a warp-wide
// instruction of the uniform section advances 32 FM chains, no shuffles are needed, and the divergent per-read control is
// amortised over 32 reads.  The kernel is bound by instruction issue (profiles/r01_notes.md).
constexpr int SWEEP1_THREADS = 128;
constexpr int SWEEP1_CAP = 8;                              // candidates kept in shared memory per read
constexpr int SWEEP1_MIN_BLOCKS = 7;                       // register budget: 72 per thread (measured best of 6 / 7 / 8, profiles/r02_notes.md)

// One FM extension step by ONE lane, ONE bucket per pass.  Rows P0 and P1 usually fall into the same 192-row bucket
// (the interval is narrow after the seed): one pass reads that bucket (two 256-bit loads), builds the "equals c" /
// "less than c" masks once and counts below both offsets.  When they straddle two buckets (about one step in eight) the
// first pass banks the counts at P0 and the lane comes back in the next iteration for P1's bucket: one more trip for
// those steps instead of 16 more live registers and a second set of masks in every step.
struct LanePartial {
    uint32_t eq0, lt0;
    bool have;
};

// The lane loads both halves of its bucket itself.  Fetching a bucket as one 64-byte request by a lane pair (shuffles hand
// the other half over) measured slower: 54.7 vs 44.3 ms per 10 M reads at C4, the shuffles sit between the loads and their
// use (profiles/r02_notes.md).
__device__ __forceinline__ bool lane_step(const uint4* __restrict__ fwd, const uint4* __restrict__ rev, bool use_rev, uint32_t P0, uint32_t P1,
                                          uint32_t ch, uint32_t Cc, uint32_t primary, bool active, LanePartial& part, StepOut& out) {
    uint32_t b0, r0, b1, r1;
    split192(P0, b0, r0);
    split192(P1, b1, r1);
    const bool second = part.have;
    const uint32_t b = second ? b1 : b0;
    Half a0 = Half{0, 0, 0, 0, 0, 0, 0, 0}, a1 = a0;
    if (active) {
        const uint4* bk = use_rev ? rev : fwd;
        a0 = ldg_half(bk, (size_t)b * 2);
        a1 = ldg_half(bk, (size_t)b * 2 + 1);
    }
    const SymK k = sym_consts(ch);
    uint32_t E[6], T[6];
    bucket_masks(a0, a1, k, E, T);
    const uint32_t accA = bucket_counts(E, T, second ? r1 : r0);
    const uint32_t accB = bucket_counts(E, T, r1);
    uint32_t e0, l0, e1, l1;
    half_header(a0, ch, 0u, e0, l0);
    half_header(a1, ch, 1u, e1, l1);
    const uint32_t he = e0 + e1, hl = l0 + l1;
    if (!active) return false;
    if (!second && b1 != b0) {                       // P1 lies in the next bucket: bank P0's counts, come back for it
        part.eq0 = he + (accA & 0xFFFFu);
        part.lt0 = hl + (accA >> 16);
        part.have = true;
        return false;
    }
    const uint32_t eq0 = second ? part.eq0 : he + (accA & 0xFFFFu);
    const uint32_t eq1 = he + ((second ? accA : accB) & 0xFFFFu);
    const uint32_t ltd = second ? hl + (accA >> 16) - part.lt0 : (accB >> 16) - (accA >> 16);
    part.have = false;
    out = finish_step(eq0, eq1, ltd, P0, P1, ch, Cc, primary);
    return true;
}

// flush_finished for a list of 33..64 matches (one read in a dozen at 1 % substitutions): same ordered, field-by-field
// hand-over with two entries per lane -- entry x sits in lane x & 31 (x < 32: v0, else v1).  Out of line: its registers
// are not the sweep loop's.
__device__ __noinline__ void hand_over_long(const uint4* sp, uint32_t n, uint4* dst) {
    constexpr uint32_t FULLM = 0xFFFFFFFFu;
    const uint32_t lane = threadIdx.x & 31u;
    uint4 v0 = make_uint4(0u, 0u, 0u, 0u), v1 = v0;
    if (lane < n) v0 = __ldcg(sp + lane);
    if (lane + 32u < n) v1 = __ldcg(sp + lane + 32u);
    const uint32_t prev0 = __shfl_up_sync(FULLM, v0.w, 1);
    const uint32_t last0 = __shfl_sync(FULLM, v0.w, 31);
    uint32_t prev1 = __shfl_up_sync(FULLM, v1.w, 1);
    if (lane == 0u) prev1 = last0;
    const unsigned long long heads =
        (unsigned long long)__ballot_sync(FULLM, lane < n && (lane == 0u || v0.w != prev0)) |
        ((unsigned long long)__ballot_sync(FULLM, lane + 32u < n && v1.w != prev1) << 32);
    uint32_t* seg = reinterpret_cast<uint32_t*>(dst);
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const uint32_t x = lane + 32u * half;
        if (x < n) {
            const uint4 v = half ? v1 : v0;
            const unsigned long long upto = heads & (~0ull >> (63u - x));              // heads at or below this entry
            const uint32_t s0 = 63u - (uint32_t)__clzll((long long)upto);
            const unsigned long long above = x == 63u ? 0ull : heads & (~0ull << (x + 1u));
            const uint32_t s1 = above ? (uint32_t)__ffsll((long long)above) - 1u : n;
            const uint32_t d = s0 + (s1 - 1u - x);
            seg[d] = v.x; seg[n + d] = v.y; seg[2u * n + d] = v.z; seg[3u * n + d] = v.w;
        }
    }
}

template <bool LONG, bool UNIQ>
struct DevSweepCtx1 {
    const SweepArgs& a;
    uint32_t cand0;       // index (uint4) of this lane's candidate slots
    uint32_t words0;      // word offset of this lane's packed read in shared memory (!LONG)
    uint4* stage;         // global: match staging of this lane
    uint4* spill;         // global: candidate spill of this lane
    const uint32_t* gwords;   // LONG: the read's packed words in global memory
    uint32_t fin_rid, fin_n;  // a finished read waiting for the warp's cooperative flush (fin_n == NO_FIN: none)
    static constexpr uint32_t NO_FIN = 0xFFFFFFFFu;

    __device__ __forceinline__ bool fetch(uint32_t& rid, uint32_t& L) {
        const unsigned long long r = atomicAdd(&a.counters[3], 1ull);
        if (r >= a.n_reads) return false;
        rid = (uint32_t)r;
        L = __ldg(a.len + rid);
        const uint32_t off = __ldg(a.chunk_off + rid);
        if (LONG) {
            gwords = reinterpret_cast<const uint32_t*>(a.reads + (size_t)off);
        } else {
            const uint32_t nch = (L + 63u) >> 6;
            for (uint32_t c = 0; c < nch; ++c) g_sweep_smem[(words0 >> 2) + c] = __ldg(a.reads + (size_t)off + c);
        }
        return true;
    }
    __device__ __forceinline__ uint32_t word(uint32_t w) const {
        return LONG ? __ldg(gwords + w) : reinterpret_cast<const uint32_t*>(g_sweep_smem)[words0 + w];
    }
    __device__ __forceinline__ uint32_t base(uint32_t pos) const { return (word(pos >> 4) >> (30u - 2u * (pos & 15u))) & 3u; }
    __device__ __forceinline__ uint32_t seed_k() const { return a.seed_K; }
    // unique-match shortcut, forward direction: once q[x:pos) occurs once, its extent is read off the text (sweep_logic.cuh)
    __device__ __forceinline__ constexpr bool uniq() const { return UNIQ; }
    __device__ __forceinline__ constexpr bool uniq_back() const { return false; }
    __device__ __forceinline__ uint32_t kmer(uint32_t pos) const {
        return __funnelshift_l(word((pos >> 4) + 1u), word(pos >> 4), 2u * (pos & 15u)) >> (32u - 2u * a.seed_K);
    }
    // Number of leading bases (at most 64) on which text[t..) and q[p..) agree: both sides are MSB-first 2-bit words, so
    // after one funnel shift per word to a common phase a mismatch is the first set bit of the XOR.  Callers cap the
    // result by the bases that really exist on both sides (Sweeper::cmp_max).
    __device__ __forceinline__ uint32_t match_forward(uint32_t t, uint32_t p) const {
        const uint32_t tw = t >> 4, ts = 2u * (t & 15u), qw = p >> 4, qs = 2u * (p & 15u);
        const uint32_t tlast = ((a.n_bases + 15u) >> 4) + 1u;           // the text is readable 2 words past its end
        uint32_t T[5], Q[5];
#pragma unroll
        for (uint32_t i = 0; i < 5u; ++i) {
            const uint32_t w = tw + i;
            T[i] = __ldg(a.text + (w < tlast ? w : tlast));
            Q[i] = word(qw + i);
        }
        uint32_t matched = 64u;
#pragma unroll
        for (int i = 3; i >= 0; --i) {
            const uint32_t x = __funnelshift_l(T[i + 1], T[i], ts) ^ __funnelshift_l(Q[i + 1], Q[i], qs);
            if (x != 0u) matched = 16u * (uint32_t)i + ((uint32_t)__clz((int)x) >> 1);
        }
        return matched;
    }
    __device__ __forceinline__ void cand_put(uint32_t i, uint32_t j, uint32_t lo, uint32_t cnt) {
        if (i < (uint32_t)SWEEP1_CAP) g_sweep_smem[cand0 + i] = make_uint4(j, lo, cnt, 0u);
        else __stcg(spill + (i - SWEEP1_CAP), make_uint4(j, lo, cnt, 0u));
    }
    __device__ __forceinline__ void cand_get(uint32_t i, uint32_t& j, uint32_t& lo, uint32_t& cnt) const {
        uint4 v;
        if (i < (uint32_t)SWEEP1_CAP) v = g_sweep_smem[cand0 + i];
        else v = __ldcg(spill + (i - SWEEP1_CAP));
        j = v.x; lo = v.y; cnt = v.z;
    }
    __device__ __forceinline__ void cand_sync() {}
    __device__ __forceinline__ void emit(uint32_t idx, MemEntry e) { __stcg(stage + idx, make_uint4(e.se, e.lo, e.cnt, e.sweep)); }
    // the read's matches stay in this lane's staging slots until the warp flushes them together (flush_finished)
    __device__ __forceinline__ void finish(uint32_t rid, uint32_t n) { fin_rid = rid; fin_n = n; }

    // Warp-cooperative hand-over of the finished reads' matches to the pool: one atomic per warp reserves the space, then
    // all 32 lanes copy each finished read's staged matches (coalesced 16-byte stores) instead of the owning lane copying
    // them one by one behind dependent L2 loads.  Lists of up to 32 matches are put in ascending order on the way -- the
    // sweep emits every sweep's matches longest end first -- stored field by field, and flagged (bit 31 of mem_cnt) so
    // that the selection kernels neither reorder them nor read them as 16-byte entries.  Called by the whole warp.
    static constexpr uint32_t SOA_MAX = 64;          // lists up to this long are handed over ordered and field by field
    __device__ __forceinline__ void flush_finished() {
        constexpr uint32_t FULLM = 0xFFFFFFFFu;
        const uint32_t lane = threadIdx.x & 31u;
        uint32_t todo = __ballot_sync(FULLM, fin_n != NO_FIN);
        if (todo == 0u) return;
        // exclusive prefix of the finished reads' match counts, warp total to the pool counter
        const uint32_t mine = fin_n != NO_FIN ? fin_n : 0u;
        uint32_t incl = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(FULLM, incl, d);
            if (lane >= (uint32_t)d) incl += y;
        }
        const uint32_t total = __shfl_sync(FULLM, incl, 31);
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(&a.counters[0], (unsigned long long)total);
        base = __shfl_sync(FULLM, base, 0);
        const bool fits = base + total <= a.mem_cap;
        if (!fits && lane == 0) atomicOr(&a.counters[2], 1ull);
        const unsigned long long my_off = base + (incl - mine);
        const unsigned long long st = (unsigned long long)(uintptr_t)stage;
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1u;
            const uint32_t n = __shfl_sync(FULLM, fin_n, src);
            const unsigned long long off = __shfl_sync(FULLM, my_off, src);
            const uint4* sp = reinterpret_cast<const uint4*>((uintptr_t)__shfl_sync(FULLM, st, src));
            if (!fits) continue;
            // Short lists are handed over in ascending order and stored field by field (n start|end words, then n lo, n count,
            // n sweep ordinals): the selection kernels look starts and ends up over and over, and this way those lookups
            // share one or two sectors.  A segment = run of equal sweep ordinals (.w), emitted in descending order of the
            // end: each run is reversed on the way.
            if (n <= 32u) {
                uint4 v = make_uint4(0u, 0u, 0u, 0u);
                if (lane < n) v = __ldcg(sp + lane);
                const uint32_t prev = __shfl_up_sync(FULLM, v.w, 1);
                const uint32_t heads = __ballot_sync(FULLM, lane < n && (lane == 0u || v.w != prev));
                uint32_t d = 64u;                                                         // this lane's entry goes to position d of the ordered list
                if (lane < n) {
                    const uint32_t upto = heads & (0xFFFFFFFFu >> (31u - lane));          // heads at or below this lane
                    const uint32_t s0 = 31u - (uint32_t)__clz((int)upto);
                    const uint32_t above = lane == 31u ? 0u : heads & (0xFFFFFFFFu << (lane + 1u));
                    const uint32_t s1 = above ? (uint32_t)__ffs((int)above) - 1u : n;
                    d = s0 + (s1 - 1u - lane);
                }
                // While the list is in registers: the BWA-SMEM selection over it (get_SMEMS, SMEM.py:456-467 = Selector::run_bwa:
                // from position p take the longest match covering p -- ties: the first; nothing covers p: the first match
                // ending beyond it --, jump to its end), the warp working on one read: one reduction and one shuffle per pick.
                // The picks (bit = position in the ordered list) take the place of the first sweep ordinal, which nobody
                // reads once the list is in order: gsm_smem_select(BWA) needs no pass over the list, and the records are
                // written straight from it.
                const uint32_t ox = __shfl_sync(FULLM, v.x, d & 31u);      // entry at position `lane`: lane d holds it (reversing is an involution)
                const uint32_t os = ox & 0xFFFFu, oe = ox >> 16;
                const uint32_t pmax = __shfl_sync(FULLM, oe, (n - 1u) & 31u);
                uint32_t picks = 0u;
                for (uint32_t p = 0u; p < pmax;) {
                    const uint32_t b = bwa_pick_of(__reduce_max_sync(FULLM, lane < n ? bwa_pick_key(os, oe, lane, p) : 0u));
                    picks |= 1u << b;
                    p = __shfl_sync(FULLM, oe, b);
                }
                if (lane < n) {
                    uint32_t* seg = reinterpret_cast<uint32_t*>(a.mem_pool + off);
                    seg[d] = v.x; seg[n + d] = v.y; seg[2u * n + d] = v.z; seg[3u * n + d] = d == 0u ? picks : v.w;
                }
            } else if (n <= SOA_MAX) {
                hand_over_long(sp, n, a.mem_pool + off);
            } else {
                for (uint32_t k = lane; k < n; k += 32u) a.mem_pool[off + k] = __ldcg(sp + k);
            }
        }
        if (fin_n != NO_FIN) {
            a.mem_off[fin_rid] = fits ? (uint32_t)my_off : 0u;
            a.mem_cnt[fin_rid] = fits ? (fin_n | (fin_n <= SOA_MAX ? MEMS_ORDERED : 0u) | (fin_n >= 1u && fin_n <= 32u ? MEMS_PICKED : 0u)) : 0u;
            fin_n = NO_FIN;
        }
    }
};

constexpr uint32_t SWEEP1_SMEM_MAX_LEN = 1024;             // longer reads run k_sweep1<true> (bases from global memory)
constexpr uint64_t SWEEP1_LONG_SCRATCH = 4ull << 30;       // staging budget that sizes the long-read grid

// shared memory per lane: SWEEP1_CAP candidates + (short reads) the packed read and one readable pad chunk for kmer()
__host__ __device__ inline uint32_t sweep1_lane_u4(uint32_t max_len, bool long_reads) {
    return SWEEP1_CAP + (long_reads ? 0u : (max_len + 63u) / 64u + 1u);
}
inline size_t sweep1_smem_bytes(uint32_t max_len, bool long_reads) {
    return (size_t)SWEEP1_THREADS * sweep1_lane_u4(max_len, long_reads) * sizeof(uint4) + 16;
}

// LONG = false: the packed read is staged in shared memory (reads up to SWEEP1_SMEM_MAX_LEN bases).
// LONG = true : the bases are read from the packed batch in global memory (L1 / L2 hits: 4 bases per byte), shared
//               memory only holds the candidate slots, so any length up to 65535 runs; the grid is sized so that the
//               per-lane match / candidate staging (2 x max_len x 16 bytes) fits a fixed budget.
// UNIQ  : the unique-match shortcut, for an index with the suffix array and the packed text on the device.
template <bool LONG, bool UNIQ>
__global__ void __launch_bounds__(SWEEP1_THREADS, SWEEP1_MIN_BLOCKS) k_sweep1(const SweepArgs a) {
    using Ctx = DevSweepCtx1<LONG, UNIQ>;
    const uint32_t lane_u4 = sweep1_lane_u4(a.max_len, LONG);
    const uint32_t p0 = threadIdx.x * lane_u4;
    const size_t gl = (size_t)blockIdx.x * SWEEP1_THREADS + threadIdx.x;
    Ctx ctx{a, p0, (p0 + SWEEP1_CAP) * 4u, a.scratch + gl * 2 * a.max_len, a.scratch + gl * 2 * a.max_len + a.max_len, nullptr, 0u, Ctx::NO_FIN};
    Sweeper<Ctx> sw;
    LanePartial part{0u, 0u, false};
    for (;;) {
        ctx.flush_finished();                 // reads finished by the last iteration's consume: before their lanes reuse the staging slots
        const bool need = sw.next(ctx, a.meta);
        if (__any_sync(0xFFFFFFFFu, ctx.fin_n != Ctx::NO_FIN)) ctx.flush_finished();      // reads finished inside next() (empty reads)
        if (!__any_sync(0xFFFFFFFFu, need)) break;
        // ONE uniform memory section per iteration: every lane issues its pending fetch here -- a seed-table entry, the
        // (at most two) buckets of an FM step, a suffix-array value or the text words of a comparison -- so all 32 chains'
        // loads are in flight together.
        const bool is_seed = need && sw.pending_seed();
        const bool is_word = UNIQ && need && sw.pending_word();
        const bool is_cmp = UNIQ && need && sw.pending_cmp();
        const bool is_step = need && !is_seed && !is_word && !is_cmp;
        uint4 se = make_uint4(0u, 0u, 0u, 0u);
        if (is_seed) se = ldg_seed(a.seed_tab + sw.P0);
        uint32_t wv = 0u, matched = 0u;
        if (UNIQ && is_word) wv = __ldg(a.sa + sw.aux);
        if (UNIQ && is_cmp) {
            matched = ctx.match_forward(sw.cmp_text(), sw.cmp_read());
            const uint32_t mx = sw.cmp_max(a.n_bases);
            matched = matched < mx ? matched : mx;
        }
        const bool rev = sw.on_reverse();
        StepOut r;
        const bool stepped = lane_step(a.fwd, a.rev, rev, sw.P0, sw.P0 + sw.cnt, sw.ch, a.meta.C[sw.ch & 3u],
                                       rev ? a.meta.prim_r : a.meta.prim_f, is_step, part, r);
        if (stepped) sw.consume(ctx, a.meta, r);
        else if (is_seed) sw.consume_seed(ctx, a.meta, SeedEntry{se.x, se.y, se.z, se.w});
        else if (UNIQ && is_word) sw.consume_word(ctx, a.meta, wv);
        else if (UNIQ && is_cmp) sw.consume_cmp(ctx, a.meta, matched);
    }
}

}  // namespace gsm
