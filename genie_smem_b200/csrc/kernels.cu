// sm_100a kernels + C ABI of the SMEM-seeding engine.
//
// Work decomposition (B200: 148 SMs, 126 MB L2, HBM3e).  The path is random access of 16..64 bytes behind dependent
// addresses: no TMA, no tensor cores; what matters is how many independent fetches a warp keeps in flight.
//   * a rank query is one aligned 64-byte bucket = two 32-byte halves, each one 256-bit load (LDG.E.ENL2.256).
//   * k_sweep1 (sweep_device.cuh; the dominant kernel): persistent grid, ONE LANE PER READ (32 reads in flight per warp,
//     dynamic read queue), bidirectional FM extension enumerating every maximal exact match of the read; per iteration
//     every lane runs its control and the warp executes ONE uniform memory section (seed-table entry / bucket / suffix-array
//     value / text words).  Finished reads hand their match lists over cooperatively (flush_finished): ordered, field by
//     field, and with the BWA-SMEM picks already made.
//   * BWA-SMEM selection: k_select_bwa_picked (count + min_len filter where the sweep made the picks), k_select<BWA> (one
//     thread per read, Selector::run_bwa) for the reads it queues, k_select_bwa_finish.  LUT-SMEM takes the same records
//     (get_smems_lut == get_SMEMS with min_len 1 on reads of >= K bases, DESIGN.md section 3) unless the frame machine is
//     asked for.  RMI-SMEM: k_rmi_prefilter sends every read without a hazard window (k_rmi_hazard_scan: the K-mer codes
//     whose last-mile search is not certified exact) through k_select<BWA> as well; only the others run the frame machine.
//   * k_select_seeded<LUT|RMI>: persistent threads, one read per thread, the reference's frame machine one ROUND at a
//     time with the warp in lock step: pass 1 = all table lookups of the round, spread evenly over the warp's lanes, results
//     in shared memory (LUT gather; RMI predict + true bounds from the k-mer bounds table or the seed table + the
//     error-bounded search replayed on row numbers, literal probe search only on a hazard), pass 2 = the integer
//     machine, pass 3 = the winner's interval; explicit backward searches are queued for k_resolve_lazy.
//   * k_scan_* / k_gather_records: counts -> offsets -> records in (read, emission) order, from the record pool or
//     straight from the picked match lists; the destination may be a peer GPU's memory (gsm_peer_*), which makes the
//     ordered write the NVLink gather of the multi-GPU path.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>

#include "../../include/genie_smem.h"
#include "host_common.hpp"
#include "select_logic.cuh"
#include "sweep_device.cuh"


namespace gsm {

#define GSM_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess)                                                                 \
            return fail(GSM_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));       \
    } while (0)

constexpr uint32_t FULL = 0xFFFFFFFFu;
// gsm_option_lut_frame_machine: 0 = LUT-SMEM records are taken from the sweep's picks (see gsm_smem_select), 1 = k_select_seeded<LUT>
static int g_lut_frame_machine = getenv("GSM_LUT_MACHINE") ? atoi(getenv("GSM_LUT_MACHINE")) : 0;
// gsm_option_rmi_prefilter: 1 = RMI-SMEM reads without a hazard window take their records from the BWA-SMEM selection
// (k_rmi_prefilter, see gsm_smem_select), 0 = every read runs the frame machine (k_select_seeded<RMI>)
static int g_rmi_prefilter = getenv("GSM_RMI_PREFILTER") ? atoi(getenv("GSM_RMI_PREFILTER")) : 1;
constexpr uint8_t READ_PENDING = 0xFFu;      // read_status while a pre-filtered RMI batch waits for the frame machine (never survives a select)
constexpr int SELECT_THREADS = 128;
constexpr int SELECT_BLOCKS = 7;             // k_select_seeded: resident blocks per SM the registers are allocated for (72 registers;
                                             // 6 and 8 measured slower for both methods)
constexpr uint32_t SELECT_STAGE = 64;   // staged records per selection thread; reads emitting more are run twice (see DevSelCtx::close)

// ===================================================================================== select
struct SelectArgs {
    const uint4* fwd;
    IndexMeta meta;
    uint64_t n_bases;
    const uint32_t* sa;
    const uint32_t* text;
    const uint4* probe;         // optional {sa, 32-mer code} records (gsm_rmi_probe_build), else NULL
    const uint32_t* reads;      // as words
    const uint32_t* chunk_off;
    const uint32_t* len;
    uint32_t n_reads;
    uint32_t max_len;
    uint32_t read_id_base;
    uint32_t min_len;
    uint32_t K;
    const uint2* lut;
    const uint4* seed_tab;      // optional sweep seed table (gsm_seed_table_build): shortens explicit backward searches
    uint32_t seed_K;
    RmiModel rmi;
    const uint2* rmi_bounds;    // optional {first row >= k-mer, occurrences} per K-mer code (gsm_rmi_bounds_build), else NULL
    uint4* mem_pool;
    const uint32_t* mem_off;
    const uint32_t* mem_cnt;
    uint4* stage;               // per thread: stage_stride records (a read that emits more is run a second time, writing in place)
    uint32_t stage_stride;
    uint4* rec_tmp;
    unsigned long long rec_cap;
    uint32_t* rec_tmp_off;
    uint32_t* rec_cnt;
    uint8_t* read_status;
    unsigned long long* counters;
    uint4* fix;                 // deferred explicit searches {read, record ordinal, start | end << 16, 0} (k_resolve_lazy): the tail of the record pool
    unsigned long long fix_cap;
    const uint32_t* hz_slots;   // RMI pre-filter: hash set of the model's hazard codes (gsm_rmi_hazard_scan / gsm_rmi_hazard_hash), else NULL
    uint32_t hz_mask;           // slots - 1
    uint32_t only_pending;      // k_select_seeded: run only the reads k_rmi_prefilter left at READ_PENDING
};

// 16-byte probe record {s, code64 hi, code64 lo, 0}: one fetch per get_ref_seq (RMI_LUT.py:89-92)
struct TableProbe {
    const uint4* t;
    __device__ __forceinline__ void operator()(uint64_t row, int64_t& s, uint64_t& code64) const {
        const uint4 v = __ldg(t + row);
        s = (int64_t)v.x;
        code64 = ((uint64_t)v.y << 32) | (uint64_t)v.z;
    }
};

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

template <int METHOD>
struct DevSelCtx {
    // LUT seeds are real table rows (32 bits); the RMI search may return negative or wrapped rows
    using iv_t = typename std::conditional<METHOD == GSM_METHOD_RMI, int64_t, uint32_t>::type;
    const SelectArgs& a;
    const uint32_t* words;
    uint4* mems;
    uint4* out;           // where this read's records go: the thread's staging slots, or (second run of a read that
    uint32_t cap;         // overflowed them) its exactly sized segment of the record pool; cap = slots available
    uint32_t L, K, n_mems, min_len, rid, n_rec;
    bool raised;
    bool overflow;        // more records than slots: counted, not stored
    // bit 31 of mem_cnt: the sweep stored this list in ascending order and field by field (n start|end words, n lo, n count, ...)
    bool soa;
    __device__ __forceinline__ uint32_t se(uint32_t k) const { return soa ? reinterpret_cast<const uint32_t*>(mems)[k] : mems[k].x; }

    __device__ __forceinline__ MemEntry mem(uint32_t k) const {
        if (soa) {
            const uint32_t* seg = reinterpret_cast<const uint32_t*>(mems);
            return MemEntry{seg[k], seg[n_mems + k], seg[2u * n_mems + k], seg[3u * n_mems + k]};
        }
        uint4 v = mems[k];
        return MemEntry{v.x, v.y, v.z, v.w};
    }
    __device__ __forceinline__ uint32_t base(uint32_t pos) const { return (__ldg(words + (pos >> 4)) >> (30u - 2u * (pos & 15u))) & 3u; }
    __device__ __forceinline__ bool failed() const { return raised; }
    __device__ __forceinline__ bool seeds_are_true() const { return METHOD == GSM_METHOD_LUT; }

    // True SA interval of q[i:j) by backward search (ExactMatch.exact_match_back_prop, ExactMatch.py:132-151), resumable:
    // interval_begin takes the first K / seed_K steps from a table entry, interval_step prepends q[p-1].
    __device__ __forceinline__ void interval_begin(uint32_t i, uint32_t j, uint32_t& lo, uint32_t& cnt, uint32_t& p) const {
        lo = 0; cnt = a.meta.n_rows; p = j;
        const uint32_t* w = words;
        auto rd = [w](uint64_t x) { return __ldg(w + x); };
        if (a.seed_K != 0u && j - i >= a.seed_K && (METHOD != GSM_METHOD_LUT || a.seed_K >= K)) {
            const uint4 e = __ldg(a.seed_tab + kmer_code(rd, j - a.seed_K, a.seed_K));   // the longest table first
            lo = e.x; cnt = e.y; p = j - a.seed_K;
        } else if (METHOD == GSM_METHOD_LUT && j - i >= K) {      // the table replaces the first K backward steps
            const uint2 e = __ldg(a.lut + kmer_code(rd, j - K, K));
            lo = e.x; cnt = e.y; p = j - K;
        }
    }
    __device__ __forceinline__ void interval_step(uint32_t& lo, uint32_t& cnt, uint32_t& p) const {
        const uint4* fwd = a.fwd;
        auto load = [fwd](uint64_t idx) { return ldg_half(fwd, idx); };
        const uint32_t ch = base(p - 1);
        const StepOut r = step_single(load, lo, lo + cnt, ch, a.meta.C[ch], a.meta.prim_f);
        lo = r.lo_new; cnt = r.cnt_new; --p;
    }
    __device__ void interval(uint32_t i, uint32_t j, uint32_t& lo, uint32_t& cnt) {
        uint32_t p;
        interval_begin(i, j, lo, cnt, p);
        while (p > i && cnt != 0u) interval_step(lo, cnt, p);
    }

    // One probe of the RMI last-mile search (RMI_LUT.get_ref_seq, RMI_LUT.py:89-92): the 16-byte {SA value, 32-mer}
    // record when the probe table exists (one fetch), else the suffix array and then the packed text.
    __device__ __forceinline__ void probe_row(uint64_t row, int64_t& s, uint64_t& code64) const {
        if (a.probe) {
            const uint4 v = __ldg(a.probe + row);
            s = (int64_t)v.x;
            code64 = ((uint64_t)v.y << 32) | (uint64_t)v.z;
        } else {
            const uint32_t* tx = a.text;
            auto txl = [tx](uint64_t i) { return __ldg(tx + i); };
            s = (int64_t)__ldg(a.sa + row);
            code64 = kmer_code(txl, (uint64_t)(s - 1), 32);
        }
    }

    __device__ __forceinline__ uint64_t window_code(uint32_t cpos) const {
        const uint32_t* w = words;
        auto rd = [w](uint64_t i) { return __ldg(w + i); };
        return kmer_code(rd, cpos, K);
    }

    // true bounds (first row >= k-mer, occurrences) of window cpos from the sweep's seed table (needs seed_K <= K)
    __device__ __forceinline__ void window_bounds(uint32_t cpos, uint32_t& A, uint32_t& cnt) const {
        const uint32_t* w = words;
        const uint4* fwd = a.fwd;
        const uint4* tab = a.seed_tab;
        auto rd = [w](uint64_t i) { return __ldg(w + i); };
        auto load = [fwd](uint64_t idx) { return ldg_half(fwd, idx); };
        auto seed = [tab](uint64_t code) { const uint4 v = __ldg(tab + code); return U4{v.x, v.y, v.z, v.w}; };
        kmer_bounds_seeded(rd, load, seed, a.meta, cpos, K, a.seed_K, A, cnt);
    }

    __device__ bool sequential(uint32_t c, int64_t clo, int64_t chi, uint32_t pc, int64_t plo, int64_t phi, bool both_true) {
        const uint4* fwd = a.fwd;
        auto load = [fwd](uint64_t idx) { return ldg_half(fwd, idx); };
        if (METHOD == GSM_METHOD_LUT || both_true) {
            const DevSelCtx* self = this;
            auto bs = [self](uint32_t p) { return self->base(p); };
            return true_sequential(bs, load, a.meta, K, c, pc, plo, phi);
        }
        // RMI: check on the RETURNED intervals (SMEM.py:262-265), which may be wrong: x == LF(y) in O(1)
        const uint32_t* sa = a.sa;
        auto sal = [sa](uint64_t r) { return __ldg(sa + r); };
        return rmi_sequential(load, sal, a.meta, clo, chi, plo, phi);
    }

    __device__ __forceinline__ void emit(uint32_t i, uint32_t j, int64_t lo, int64_t hi) {
        if (n_rec < cap) out[n_rec] = make_uint4(a.read_id_base + rid, i | (j << 16), (uint32_t)lo, (uint32_t)hi);
        else overflow = true;
        n_rec++;
    }

    // Read finished: hand its records to the pool.  Staged records are copied to a freshly reserved segment; a read that
    // overflowed its staging slots reserves its exact count and returns true -- the caller runs it again (the selection
    // is deterministic) with `out` pointing at that segment, and the second close only publishes offset and count.
    __device__ __forceinline__ bool close(uint8_t status, bool& direct) {
        if (raised) { status = GSM_READ_REF_RAISES; n_rec = 0; overflow = false; }
        bool again = false;
        if (direct) {
            a.rec_tmp_off[rid] = (uint32_t)(out - a.rec_tmp); a.rec_cnt[rid] = n_rec;
            direct = false;
        } else {
            const unsigned long long off = atomicAdd(&a.counters[1], (unsigned long long)n_rec);
            if (off + n_rec > a.rec_cap) {
                atomicOr(&a.counters[2], 2ull);
                a.rec_tmp_off[rid] = 0; a.rec_cnt[rid] = 0;
            } else if (overflow) {
                out = a.rec_tmp + off; cap = n_rec; n_rec = 0; overflow = false;
                direct = again = true;
            } else {
                for (uint32_t k = 0; k < n_rec; ++k) a.rec_tmp[off + k] = out[k];
                a.rec_tmp_off[rid] = (uint32_t)off; a.rec_cnt[rid] = n_rec;
            }
        }
        if (!again) a.read_status[rid] = status;
        return again;
    }
};

// the sweep emits each sweep's matches longest-end first: put every segment in ascending order
// (idempotent: a second selection pass over the same sweep finds the segment ascending)
__device__ __forceinline__ void order_segments(uint4* mems, uint32_t n_mems) {
    for (uint32_t s0 = 0; s0 < n_mems;) {
        uint32_t s1 = s0 + 1;
        const uint32_t id = mems[s0].w;
        while (s1 < n_mems && mems[s1].w == id) ++s1;
        const bool descending = (mems[s0].x >> 16) > (mems[s1 - 1].x >> 16);
        for (uint32_t x = s0, y = s1 - 1; descending && x < y; ++x, --y) {
            uint4 t = mems[x]; mems[x] = mems[y]; mems[y] = t;
        }
        s0 = s1;
    }
}

// BWA-SMEM selection, one thread per read: over all reads, or (queue != nullptr) over the reads k_select_bwa_picked left.
template <int METHOD>
__global__ void __launch_bounds__(SELECT_THREADS) k_select(const SelectArgs a, const uint32_t* queue) {
    const size_t gtid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t nthreads = (size_t)gridDim.x * blockDim.x;
    uint4* const stage = a.stage + gtid * a.stage_stride;
    const size_t n_work = queue ? (size_t)a.counters[4] : (size_t)a.n_reads;
    for (size_t w = gtid; w < n_work; w += nthreads) {
        const size_t rid = queue ? queue[w] : w;
        const uint32_t mc = a.mem_cnt[rid];
        DevSelCtx<METHOD> c{a,
                            a.reads + (size_t)__ldg(a.chunk_off + rid) * 4,
                            a.mem_pool + a.mem_off[rid],
                            stage, a.stage_stride,
                            __ldg(a.len + rid), a.K, mc & MEMS_COUNT, a.min_len, (uint32_t)rid, 0u, false, false, (mc & MEMS_ORDERED) != 0u};
        if (!c.soa) order_segments(c.mems, c.n_mems);        // MEMS_ORDERED: the sweep already ordered the list
        bool direct = false;
        if (a.K != 0u && c.L < a.K) { c.close(GSM_READ_TOO_SHORT, direct); continue; }       // LUT-SMEM through this kernel: K = the table's k
        do {
            static_assert(METHOD == GSM_METHOD_BWA, "LUT- and RMI-SMEM run in k_select_seeded");
            Selector<DevSelCtx<METHOD>>::run_bwa(c);
            if (!c.close(GSM_READ_OK, direct)) break;
        } while (true);
    }
}

// BWA-SMEM selection where the sweep has already made the picks (MEMS_PICKED: lists of 1..32 matches, nine reads in ten):
// the read's records ARE the picked entries of its match list, so "selecting" is the min_len filter and a count --
// rec_cnt[read] = records, rec_tmp_off[read] = the picks (k_gather_records writes the records from the list).  Reads
// without picks are queued for k_select<BWA>; counters[6] += records counted here.
__global__ void __launch_bounds__(256) k_select_bwa_picked(const SelectArgs a, uint32_t* queue) {
    const size_t rid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t n_rec = 0;
    bool later = false;
    if (rid < a.n_reads) {
        const uint32_t mc = a.mem_cnt[rid];
        if (a.K != 0u && __ldg(a.len + rid) < a.K) {                  // LUT-SMEM through this kernel: reads shorter than the table's k
            a.rec_cnt[rid] = 0u; a.rec_tmp_off[rid] = 0u; a.read_status[rid] = GSM_READ_TOO_SHORT;
        } else if (mc & MEMS_PICKED) {
            const uint32_t n = mc & MEMS_COUNT;
            const uint32_t* seg = reinterpret_cast<const uint32_t*>(a.mem_pool + a.mem_off[rid]);
            uint32_t picks = seg[3u * n];
            if (a.min_len > 1u)
                for (uint32_t m = picks; m != 0u; m &= m - 1u) {
                    const uint32_t k = (uint32_t)__ffs((int)m) - 1u, w = seg[k];
                    if ((w >> 16) - (w & 0xFFFFu) < a.min_len) picks &= ~(1u << k);
                }
            n_rec = (uint32_t)__popc(picks);
            a.rec_cnt[rid] = n_rec; a.rec_tmp_off[rid] = picks; a.read_status[rid] = GSM_READ_OK;
        } else {
            later = true;
        }
    }
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t lm = __ballot_sync(FULL, later);
    if (lm) {
        unsigned long long slot = 0;
        if (lane == (uint32_t)__ffs((int)lm) - 1u) slot = atomicAdd(&a.counters[4], (unsigned long long)__popc(lm));
        slot = __shfl_sync(FULL, slot, __ffs((int)lm) - 1);
        if (later) queue[slot + __popc(lm & ((1u << lane) - 1u))] = (uint32_t)rid;
    }
    const uint32_t total = __reduce_add_sync(FULL, n_rec);
    if (lane == 0 && total) atomicAdd(&a.counters[6], (unsigned long long)total);
}

// after the two BWA kernels: counters[1] (records of the batch; so far the pool cursor of k_select<BWA>) += counters[6]
__global__ void k_select_bwa_finish(unsigned long long* counters) { counters[1] += counters[6]; }

// RMI-SMEM pre-filter, one thread per read: a read none of whose K-mer windows is a hazard code of the model (select_logic.cuh,
// "hazard codes of a model") emits exactly the BWA-SMEM records with min_len 1, so it is queued for k_select<BWA> (which also
// flags reads shorter than K); a read with a hazard window is left at READ_PENDING for the frame machine (k_select_seeded<RMI>
// with only_pending).  Queue: 4 read numbers per 16-byte slot of the record pool's last eighth, length in counters[4].
__global__ void __launch_bounds__(256) k_rmi_prefilter(const SelectArgs a, uint32_t* queue) {
    const size_t rid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool picks = false;
    if (rid < a.n_reads) {
        const uint32_t* w = a.reads + (size_t)__ldg(a.chunk_off + rid) * 4;
        const uint32_t* slots = a.hz_slots;
        picks = rmi_read_hazard_free([w](uint32_t x) { return __ldg(w + x); }, __ldg(a.len + rid), a.K,
                                     [slots](uint32_t h) { return __ldg(slots + h); }, a.hz_mask);
        if (!picks) a.read_status[rid] = READ_PENDING;
    }
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t pm = __ballot_sync(FULL, picks);
    if (pm) {
        unsigned long long slot = 0;
        if (lane == (uint32_t)__ffs((int)pm) - 1u) slot = atomicAdd(&a.counters[4], (unsigned long long)__popc(pm));
        slot = __shfl_sync(FULL, slot, __ffs((int)pm) - 1);
        if (picks) queue[slot + __popc(pm & ((1u << lane) - 1u))] = (uint32_t)rid;
    }
}

// Every K-mer code whose lookup the arithmetic replay cannot certify (rmi_code_is_hazard) is appended to out[] (at most cap
// codes are stored; *count keeps counting, so the caller sees an overflow).  bounds = gsm_rmi_bounds_build's table.
__global__ void __launch_bounds__(256) k_rmi_hazard_scan(RmiModel m, const uint2* bounds, uint64_t n_codes, uint32_t n_rows, uint32_t* out,
                                                         unsigned long long cap, unsigned long long* count) {
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint32_t lane = threadIdx.x & 31u;
    for (uint64_t code = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; code - lane < n_codes; code += stride) {     // whole warps take a trip
        bool hz = false;
        if (code < n_codes) {
            const uint2 b = __ldg(bounds + code);
            hz = rmi_code_is_hazard(m, code, b.x, b.y, n_rows);
        }
        const uint32_t hm = __ballot_sync(FULL, hz);                   // a poor model has hazards everywhere: one atomic per warp
        if (hm) {
            unsigned long long k = 0;
            if (lane == (uint32_t)__ffs((int)hm) - 1u) k = atomicAdd(count, (unsigned long long)__popc(hm));
            k = __shfl_sync(FULL, k, __ffs((int)hm) - 1) + __popc(hm & ((1u << lane) - 1u));
            if (hz && k < cap) out[k] = (uint32_t)code;
        }
    }
}

// The lookup results of one round (Selector::round_decide's `win`) in shared memory: two planes (lo, hi) of K windows x
// WIN_STRIDE words, window i of a thread at word i * WIN_STRIDE + threadIdx.x -- nothing of it lives in local memory (as
// per-thread arrays the two planes were 512 bytes of stack per thread: with 151,552 resident threads more than the L2
// holds), and ANY lane of the warp can store a thread's result (pass 1 of k_select_seeded spreads the windows of the warp's
// 32 reads evenly over its lanes).  WIN_STRIDE is odd: the windows of one thread lie in different banks, and so do the
// same window of the 32 threads.  RMI rows may be negative (down to -n_rows, Python indexing of a wrong interval;
// n_rows < 2^32): the low 32 bits are stored and the signs kept in two masks (bit = window).
constexpr int WIN_STRIDE = SELECT_THREADS + 1;
constexpr int WIN_MASKS = 5;                               // per thread: hit, true, redo, lo negative, hi negative
enum : int { WM_HIT = 0, WM_TRUE = 1, WM_REDO = 2, WM_NEG_LO = 3, WM_NEG_HI = 4 };
__host__ __device__ constexpr size_t select_smem_bytes(uint32_t K) {
    return (2ull * K * WIN_STRIDE + (size_t)WIN_MASKS * SELECT_THREADS) * sizeof(uint32_t) + (size_t)K * SELECT_THREADS * sizeof(uint16_t);
}
template <int METHOD>
struct SmemWindows {
    using iv_t = typename DevSelCtx<METHOD>::iv_t;
    uint32_t* lo_w;         // this thread's column of the two planes
    uint32_t* hi_w;
    uint32_t neg_lo, neg_hi;
    __device__ __forceinline__ iv_t lo(uint32_t i) const {
        const uint32_t v = lo_w[i * WIN_STRIDE];
        if (METHOD == GSM_METHOD_RMI) return (iv_t)((int64_t)v - ((int64_t)((neg_lo >> i) & 1u) << 32));
        return (iv_t)v;
    }
    __device__ __forceinline__ iv_t hi(uint32_t i) const {
        const uint32_t v = hi_w[i * WIN_STRIDE];
        if (METHOD == GSM_METHOD_RMI) return (iv_t)((int64_t)v - ((int64_t)((neg_hi >> i) & 1u) << 32));
        return (iv_t)v;
    }
    __device__ __forceinline__ void put(uint32_t i, iv_t l, iv_t h) {
        lo_w[i * WIN_STRIDE] = (uint32_t)l;
        hi_w[i * WIN_STRIDE] = (uint32_t)h;
        if (METHOD == GSM_METHOD_RMI) {
            neg_lo = (neg_lo & ~(1u << i)) | ((uint32_t)((int64_t)l < 0) << i);
            neg_hi = (neg_hi & ~(1u << i)) | ((uint32_t)((int64_t)h < 0) << i);
        }
    }
    // store into the column of the thread `d` lanes away (same warp); signs are the caller's business
    __device__ __forceinline__ void put_for(int d, uint32_t i, uint32_t l, uint32_t h) const {
        lo_w[(int)(i * WIN_STRIDE) + d] = l;
        hi_w[(int)(i * WIN_STRIDE) + d] = h;
    }
};

// One phase of the error-bounded search over the windows in `mask` (bit = window), run by the whole warp in lock step:
// a thread that finishes a window banks it and begins its next one (divergent, a few instructions), then everybody
// meets at the single probe + straight-line feed; the warp leaves when no thread has a window left.
template <typename Machine, typename Begin, typename Bank, typename Feed>
__device__ __forceinline__ void phase_loop(uint32_t mask, Machine& mach, Begin begin, Bank bank, Feed feed) {
    int cur = -1;
    bool more = mask != 0u;
    for (;;) {
        while (more && !mach.busy) {
            if (cur >= 0) { bank(cur); cur = -1; }
            if (mask == 0u) { more = false; break; }
            cur = __ffs(mask) - 1;
            mask &= mask - 1u;
            begin(cur);
        }
        const bool need = more && mach.busy;
        if (!__any_sync(FULL, need)) break;
        if (need) feed();
    }
}

// The literal exponential + binary search (RmiSearch: probe for probe the reference's) for the windows in `redo` of every
// thread of the warp, one probe site.  Only hazardous lookups come here (a handful per million), and the search state is
// large: kept out of line so that its registers are not the selection kernel's.
// Arguments and results travel by value (nothing of the caller's state has its address taken).
struct LiteralOut { uint32_t whit, neg_lo, neg_hi, raised; };
template <int METHOD>
__device__ __noinline__ LiteralOut literal_lookups(const SelectArgs& a, const uint32_t* words, SmemWindows<METHOD> win, uint32_t redo,
                                                   uint32_t e, bool first, uint32_t whit) {
    using iv_t = typename DevSelCtx<METHOD>::iv_t;
    DevSelCtx<METHOD> c{a, words, nullptr, nullptr, 0u, 0u, a.K, 0u, 0u, 0u, 0u, false, false, false};
    RmiSearch rs;
    int cur = -1;
    bool more = redo != 0;
    for (;;) {
        while (more && !rs.pending()) {
            if (cur >= 0) {
                if (rs.raised) { c.raised = true; more = false; break; }
                win.put((uint32_t)cur, (iv_t)rs.out_lo, (iv_t)rs.out_hi);
                if (rs.hit()) whit |= 1u << cur;
                cur = -1;
            }
            if (redo == 0) { more = false; break; }
            cur = __ffs(redo) - 1;               // windows in ascending order, like the reference
            redo &= redo - 1;
            const uint32_t cpos = first ? 0u : e - (uint32_t)cur;
            rs.begin(a.rmi, c.window_code(cpos), (int64_t)a.meta.n_rows, (int64_t)a.n_bases);
        }
        const bool need = more && rs.pending();
        if (!__any_sync(FULL, need)) break;
        if (need) {
            int64_t sv;
            uint64_t code64;
            c.probe_row(rs.row(), sv, code64);   // the probe site of the literal search
            rs.feed(sv, code64);
        }
    }
    return LiteralOut{whit, win.neg_lo, win.neg_hi, c.raised ? 1u : 0u};
}

// LUT- and RMI-SMEM selection with the warp kept in lock step.  One thread per read (persistent threads pull reads
// grid-stride: a thread always has a round to run, whatever the record counts of its neighbours' reads), and the round
// structure of the frame machine (select_logic.cuh) is driven warp-wide:
//   pass 1  the table lookups of every window of the round, one converged counted loop:
//             LUT  one 8-byte gather per window (LUT.py:15-35 as a dense table);
//             RMI  predict (RMI.py:52-69) + the k-mer's true bounds from the sweep's seed table (one 16-byte fetch and
//                  K - seed_K FM steps) + rmi_arith_lookup: the error-bounded search replayed on row numbers, no probes.
//                  Without a usable seed table: the probe-based phases RmiGallop / RmiLower / RmiUpper (one probe site
//                  each, warp in lock step).  Windows either path declares hazardous (None rows in the bracket,
//                  prediction outside the table: a handful per million) go through the literal RmiSearch;
//   pass 2  each thread runs the integer frame machine of its round (divergent, no table probes) -> the round's winner;
//   pass 3  the winner's interval if it is not on the match list (rare): explicit backward search, one lock-step loop;
//           then emit, and open the next read when the current one is finished.
// Measured alternatives (profiles/r01_notes.md): the reference's control flow per thread end to end (2.2 active threads
// per instruction on the probes), and teams of 16 lanes per read with one window per lane (converged, but 16x fewer reads
// in flight: latency-bound on the machine's dependent loads, 1.7x slower than this kernel).
// ARITH (RMI only): 1 = the launch has a usable seed table (seed_K <= K) and the None rows, so every lookup is the probe-free
// rmi_arith_lookup and the probe-based phases are compiled out (fewer registers for the path that always runs);
// 2 = as 1, the k-mer's true bounds read from the dense table of gsm_rmi_bounds_build (one fetch, no backward steps).
template <int METHOD, int ARITH>
__global__ void __launch_bounds__(SELECT_THREADS, SELECT_BLOCKS) k_select_seeded(const __grid_constant__ SelectArgs a) {
    using CtxT = DevSelCtx<METHOD>;
    using Sel = Selector<CtxT>;
    const size_t gtid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t nthreads = (size_t)gridDim.x * blockDim.x;
    size_t rid = gtid;
    bool have = false;
    uint4* const stage = a.stage + gtid * a.stage_stride;
    CtxT c{a, nullptr, nullptr, stage, a.stage_stride, 0u, a.K, 0u, a.min_len, 0u, 0u, false, false, false};
    bool direct = false;
    typename Sel::Seeded st;
    using iv_t = typename CtxT::iv_t;
    extern __shared__ uint32_t sel_smem[];                 // select_smem_bytes(K): window planes | masks | the warps' item lists
    SmemWindows<METHOD> win{sel_smem + threadIdx.x, sel_smem + a.K * WIN_STRIDE + threadIdx.x, 0u, 0u};
    uint32_t* const wm = sel_smem + 2u * a.K * WIN_STRIDE + threadIdx.x;                      // mask m of this thread: wm[m * SELECT_THREADS]
    uint16_t* const items = reinterpret_cast<uint16_t*>(sel_smem + 2u * a.K * WIN_STRIDE + WIN_MASKS * SELECT_THREADS)
                            + (threadIdx.x >> 5) * (a.K * 32u);                                // this warp's (lane, window) pairs of a round
    const uint32_t lane = threadIdx.x & 31u;
    // measured per method (tools/sweep_ab.py, profiles/r02_notes.md): two (thread, window) pairs per lane and trip of pass 1,
    // and for the probe-free RMI lookups the thread's next read brought into the L2 while this one runs
    constexpr int IPL = 2;
    constexpr bool PREFETCH = METHOD == GSM_METHOD_RMI && ARITH != 0;
    uint32_t nx_chunk = 0, nx_off = 0;                     // PREFETCH: where the next read's bases and match list are

    auto close_read = [&](uint8_t status) {
        if (c.close(status, direct)) { st = typename Sel::Seeded(); return; }      // overflowed its staging slots: run it again in place
        rid += nthreads;
        have = false;
    };
    // open reads until one needs a round (reads shorter than K are closed at once)
    auto open_reads = [&]() {
        while (!have && rid < a.n_reads) {
            if (a.only_pending && a.read_status[rid] != READ_PENDING) { rid += nthreads; continue; }     // k_rmi_prefilter gave it to k_select<BWA>
            c.words = a.reads + (size_t)__ldg(a.chunk_off + rid) * 4;
            c.mems = a.mem_pool + a.mem_off[rid];
            const uint32_t mc = a.mem_cnt[rid];
            c.L = __ldg(a.len + rid); c.n_mems = mc & MEMS_COUNT; c.rid = (uint32_t)rid; c.n_rec = 0; c.raised = false; c.overflow = false;
            c.out = stage; c.cap = a.stage_stride;
            c.soa = (mc & MEMS_ORDERED) != 0u;
            if (!c.soa) order_segments(c.mems, c.n_mems);                      // bit 31: the sweep already ordered the list
            st = typename Sel::Seeded();
            if (PREFETCH && rid + nthreads < a.n_reads) {
                // the next read's offsets: loaded now, used (prefetch_next) once this read's first round is over, by when
                // they have arrived; its length and match count are pulled into the L2 for its own open_reads
                nx_chunk = __ldg(a.chunk_off + rid + nthreads);
                nx_off = a.mem_off[rid + nthreads];
                prefetch_l2(a.mem_cnt + rid + nthreads);
                prefetch_l2(a.len + rid + nthreads);
            }
            if (c.L < c.K) { close_read(GSM_READ_TOO_SHORT); continue; }
            have = true;
        }
    };
    constexpr bool arith = METHOD == GSM_METHOD_RMI && ARITH != 0;

    for (;;) {
        while (true) {                                   // finished reads are closed, the next ones opened
            open_reads();
            if (!have || Sel::round_needed(c, st)) break;
            close_read(GSM_READ_OK);
        }
        if (!__any_sync(FULL, have)) break;
        const uint32_t nwin = st.first ? 1u : c.K;
        uint32_t whit = 0, wtrue = 0, redo = 0;
        // ---------------- pass 1: lookups, warp in lock step
        // visited windows of this round, as a bit mask (window i covers q[cpos_i : cpos_i + K), cpos_i = first ? 0 : e - i)
        uint32_t vis = 0;
        if (have) {
            for (uint32_t i = 0; i < nwin; ++i) {
                const uint32_t cpos = st.first ? 0u : st.e - i;
                if (st.first || (i < st.plen && cpos + c.K <= c.L)) vis |= 1u << i;
            }
        }
        if (METHOD == GSM_METHOD_LUT || arith) {
            // The threads of a warp visit different numbers of windows (1 in a read's first round, min(K, previous SMEM's
            // length) later): the warp lists its (thread, window) pairs and every lane takes every 32nd pair, whoever's it is
            // -- the read's words and the round's position come over by shuffle, the result goes to the owner's column of the
            // planes, the hit / true / redo bits to the owner's masks (one shared-memory atomic per owner and loop trip).
            uint32_t incl = __popc(vis);
            const uint32_t nv = incl;
            for (uint32_t d = 1; d < 32u; d <<= 1) {
                const uint32_t y = __shfl_up_sync(FULL, incl, d);
                if (lane >= d) incl += y;
            }
            const uint32_t total = __shfl_sync(FULL, incl, 31);
            uint32_t slot = incl - nv;
            for (uint32_t m = vis; m != 0u; m &= m - 1u) items[slot++] = (uint16_t)(lane | ((uint32_t)(__ffs(m) - 1) << 5));
#pragma unroll
            for (int m = 0; m < WIN_MASKS; ++m) wm[m * SELECT_THREADS] = 0u;
            __syncwarp();
            const uint32_t e_eff = st.first ? 0u : st.e;        // window w of the round starts at e_eff - w (first round: window 0 at 0)
            const unsigned long long my_words = (unsigned long long)c.words;
            const uint4* fwd = a.fwd;
            auto load = [fwd](uint64_t idx) { return ldg_half(fwd, idx); };
            const uint64_t seed_mask = (1ull << (2u * a.seed_K)) - 1ull;
            for (uint32_t k0 = 0; k0 < total; k0 += 32u * IPL) {
                bool on[IPL];
                uint32_t owner[IPL], w[IPL], tA[IPL], tn[IPL];
                uint64_t code[IPL];
                uint32_t fhit[IPL], ftrue[IPL], fredo[IPL], fnl[IPL], fnh[IPL];
#pragma unroll
                for (int j = 0; j < IPL; ++j) {                 // the pairs' k-mer codes and table fetches, all in flight together
                    const uint32_t idx = k0 + 32u * j + lane;
                    on[j] = idx < total;
                    const uint32_t it = on[j] ? items[idx] : 0u;
                    owner[j] = it & 31u; w[j] = it >> 5;
                    const uint32_t* ow = (const uint32_t*)__shfl_sync(FULL, my_words, owner[j]);
                    const uint32_t cpos = __shfl_sync(FULL, e_eff, owner[j]) - w[j];
                    code[j] = 0; tA[j] = 0; tn[j] = 0;
                    fhit[j] = ftrue[j] = fredo[j] = fnl[j] = fnh[j] = 0u;
                    if (on[j]) {
                        auto rd = [ow](uint64_t x) { return __ldg(ow + x); };
                        code[j] = kmer_code(rd, cpos, c.K);
                        if (METHOD == GSM_METHOD_LUT) {         // one 8-byte gather (LUT.py:15-35 as a dense table)
                            const uint2 t = __ldg(a.lut + code[j]);
                            tA[j] = t.x; tn[j] = t.y;
                        } else if (ARITH == 2) {                // the k-mer's true bounds straight from the dense table
                            const uint2 t = __ldg(a.rmi_bounds + code[j]);
                            tA[j] = t.x; tn[j] = t.y;
                        } else {                                // seed-table entry of the window's last seed_K bases
                            const uint4 t = __ldg(a.seed_tab + (code[j] & seed_mask));
                            tA[j] = t.x; tn[j] = t.y;
                        }
                    }
                }
                if (METHOD == GSM_METHOD_LUT) {
#pragma unroll
                    for (int j = 0; j < IPL; ++j)
                        if (on[j]) {
                            win.put_for((int)owner[j] - (int)lane, w[j], tA[j], tA[j] + tn[j] - 1u);
                            fhit[j] = tn[j] != 0u;
                        }
                } else {
                    double pred[IPL];                           // while the fetches travel: the model predictions (parameters are L2-resident)
                    rmi_predict_n<IPL>(a.rmi, code, pred);
#pragma unroll
                    for (int j = 0; j < IPL; ++j)
                        if (on[j]) {
                            uint32_t A = tA[j], n = tn[j];
                            if (ARITH != 2) {
                                for (uint32_t p = c.K - a.seed_K; p > 0; --p) {        // K - seed_K backward steps
                                    const uint32_t ch = (uint32_t)(code[j] >> (2u * (c.K - p))) & 3u;
                                    const StepOut r = step_single(load, A, A + n, ch, a.meta.C[ch], a.meta.prim_f);
                                    A = r.lo_new; n = r.cnt_new;
                                }
                            }
                            int64_t lo, hi;                     // the error-bounded search replayed on row numbers
                            if (rmi_arith_lookup(a.rmi, RmiGallop::row_of(pred[j], a.meta.n_rows), A, n, a.meta.n_rows, lo, hi)) {
                                win.put_for((int)owner[j] - (int)lane, w[j], (uint32_t)lo, (uint32_t)hi);
                                ftrue[j] = 1u; fhit[j] = hi >= lo; fnl[j] = lo < 0; fnh[j] = hi < 0;
                            } else {
                                fredo[j] = 1u;
                            }
                        }
                }
#pragma unroll
                for (int j = 0; j < IPL; ++j) {
                    // the pairs of one owner are neighbours in the list: combine their bits before touching its masks
                    const uint32_t peers = __match_any_sync(FULL, on[j] ? owner[j] : 32u);
                    const uint32_t bit = 1u << w[j];
                    const bool lead = on[j] && lane == (uint32_t)(__ffs(peers) - 1);
                    uint32_t* const om = wm + ((int)owner[j] - (int)lane);
                    uint32_t v = __reduce_or_sync(peers, fhit[j] ? bit : 0u);
                    if (lead && v) atomicOr(om + WM_HIT * SELECT_THREADS, v);
                    if (METHOD == GSM_METHOD_RMI) {
                        v = __reduce_or_sync(peers, ftrue[j] ? bit : 0u);
                        if (lead && v) atomicOr(om + WM_TRUE * SELECT_THREADS, v);
                        v = __reduce_or_sync(peers, fredo[j] ? bit : 0u);
                        if (lead && v) atomicOr(om + WM_REDO * SELECT_THREADS, v);
                        if (__any_sync(FULL, (fnl[j] | fnh[j]) != 0u)) {              // negative rows: rare
                            v = __reduce_or_sync(peers, fnl[j] ? bit : 0u);
                            if (lead && v) atomicOr(om + WM_NEG_LO * SELECT_THREADS, v);
                            v = __reduce_or_sync(peers, fnh[j] ? bit : 0u);
                            if (lead && v) atomicOr(om + WM_NEG_HI * SELECT_THREADS, v);
                        }
                    }
                }
            }
            __syncwarp();
            whit = wm[WM_HIT * SELECT_THREADS];
            if (METHOD == GSM_METHOD_LUT) {
                wtrue = vis;
            } else {
                wtrue = wm[WM_TRUE * SELECT_THREADS];
                redo = wm[WM_REDO * SELECT_THREADS];
                win.neg_lo = wm[WM_NEG_LO * SELECT_THREADS];
                win.neg_hi = wm[WM_NEG_HI * SELECT_THREADS];
            }
        } else if (ARITH == 0 && a.rmi.n_none != 0) {
            // probe-based error-bounded search (select_logic.cuh, RmiGallop / RmiLower / RmiUpper): each phase runs over ALL
            // windows of the round as one lock-step loop with straight-line per-probe code
            uint32_t todo = 0, lbm = 0, ubm = 0;
            uint64_t wcode[MAX_SEED_K];
            int64_t wlo[MAX_SEED_K], whi[MAX_SEED_K];
            for (uint32_t i = 0; i < nwin; ++i) {           // codes and model predictions, one converged counted loop
                const uint32_t cpos = st.first ? 0u : st.e - i;
                if (have && (st.first || (i < st.plen && cpos + c.K <= c.L))) {
                    wcode[i] = c.window_code(cpos);
                    wlo[i] = (iv_t)RmiGallop::predicted_row(a.rmi, wcode[i], a.meta.n_rows);
                    todo |= 1u << i;
                }
            }
            const int64_t nb = (int64_t)a.n_bases;
            const uint32_t nr = a.meta.n_rows;
            int64_t sv;
            uint64_t c64;
            {
                RmiGallop ga;                                // phase A: bracket around the prediction
                phase_loop(todo, ga,
                           [&](int w) { ga.begin(a.rmi, wcode[w], (int64_t)wlo[w], nr, nb); },
                           [&](int w) {
                               if (ga.hazard) redo |= 1u << w;
                               else { wlo[w] = (iv_t)ga.lower; whi[w] = (iv_t)ga.upper; lbm |= 1u << w; }
                           },
                           [&]() { c.probe_row(ga.row(), sv, c64); ga.feed(a.rmi, sv, c64); });
            }
            wtrue = lbm;                                     // no hazard: the bounds found below are the k-mer's true interval
            {
                RmiLower lb;                                 // phase B: first row >= q
                phase_loop(lbm, lb,
                           [&](int w) { lb.begin(a.rmi, wcode[w], (uint32_t)wlo[w], (uint32_t)whi[w], nr, nb); },
                           [&](int w) {
                               wlo[w] = (iv_t)lb.hi;
                               if (lb.hi_eq) ubm |= 1u << w;              // hit: whi[w] still holds the bracket's upper end
                               else whi[w] = (iv_t)((int64_t)lb.hi - 1);  // absent: lo = hi + 1
                           },
                           [&]() { c.probe_row(lb.row(), sv, c64); lb.feed(sv, c64); });
            }
            {
                RmiUpper ub;                                 // phase C: last row == q
                phase_loop(ubm, ub,
                           [&](int w) { ub.begin(a.rmi, wcode[w], (uint32_t)wlo[w], (uint32_t)whi[w], nr, nb); },
                           [&](int w) { whi[w] = (iv_t)ub.lo; },
                           [&]() { c.probe_row(ub.row(), sv, c64); ub.feed(sv, c64); });
                whit |= ubm;
            }
            for (uint32_t m = lbm; m != 0u; m &= m - 1u) { const uint32_t w = __ffs(m) - 1; win.put(w, (iv_t)wlo[w], (iv_t)whi[w]); }
        } else {
            redo = vis;
        }
        if (METHOD == GSM_METHOD_RMI && __any_sync(FULL, redo != 0)) {
            const LiteralOut r = literal_lookups<METHOD>(a, c.words, win, redo, st.first ? 0u : st.e, st.first, whit);
            whit = r.whit; win.neg_lo = r.neg_lo; win.neg_hi = r.neg_hi;
            if (r.raised) c.raised = true;
        }
        __syncwarp();
        // ---------------- pass 2: the frame machine of this round -> its winner
        typename Sel::Cand w{};
        bool run = have && !c.raised;
        if (run) w = Sel::round_decide(c, st, win, whit, wtrue);
        __syncwarp();
        // ---------------- pass 3: the winner's interval -- from its window, the match list, or (rare) an explicit backward
        // search, one lock-step loop
        iv_t rlo = 0, rhi = 0;
        uint32_t slo = 0, scnt = 0, sp = 0;
        bool search = run && w.valid() && Sel::resolve(c, w, win, rlo, rhi);
        if (search) {
            // a backward search of up to |SMEM| dependent bucket fetches would hold the other 31 reads of the warp up: the
            // record goes out with its rows open and k_resolve_lazy (one thread per search) fills them in afterwards
            const unsigned long long q = atomicAdd(&a.counters[4], 1ull);
            if (q < a.fix_cap) {
                a.fix[q] = make_uint4(c.rid, c.n_rec, w.ij, 0u);
                search = false;
            }
        }
        if (search) c.interval_begin(w.i(), w.j(), slo, scnt, sp);
        while (__any_sync(FULL, search)) {
            if (search) {
                if (sp > w.i() && scnt != 0u) c.interval_step(slo, scnt, sp);
                else { rlo = (iv_t)slo; rhi = (iv_t)(slo + scnt - 1u); search = false; }
            }
        }
        if (have) {
            if (PREFETCH && st.first && rid + nthreads < a.n_reads) {          // once per read
                prefetch_l2(a.reads + (size_t)nx_chunk * 4);
                prefetch_l2(a.mem_pool + nx_off);
                prefetch_l2(a.mem_pool + nx_off + 8);
            }
            if (c.raised) close_read(GSM_READ_REF_RAISES);
            else Sel::round_commit(c, st, w, rlo, rhi);
        }
        __syncwarp();
    }
}

// The explicit backward searches k_select_seeded deferred (winners whose interval is neither a seed tuple nor on the
// match list), one thread per search: rows of record `ordinal` of read `rid` <- SA interval of q[i:j).  A read that was
// closed without records (the reference raises, pool overflow) has fewer records than the ordinal says: skipped.
template <int METHOD>
__global__ void __launch_bounds__(SELECT_THREADS) k_resolve_lazy(const __grid_constant__ SelectArgs a) {
    const unsigned long long queued = a.counters[4];
    const unsigned long long n = queued < a.fix_cap ? queued : a.fix_cap;
    for (unsigned long long q = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += (unsigned long long)gridDim.x * blockDim.x) {
        const uint4 f = a.fix[q];
        const uint32_t rid = f.x;
        if (f.y >= a.rec_cnt[rid]) continue;
        DevSelCtx<METHOD> c{a, a.reads + (size_t)__ldg(a.chunk_off + rid) * 4, nullptr, nullptr, 0u, __ldg(a.len + rid), a.K, 0u, 0u, rid, 0u, false, false, false};
        uint32_t lo, cnt;
        c.interval(f.z & 0xFFFFu, f.z >> 16, lo, cnt);
        uint4* r = a.rec_tmp + a.rec_tmp_off[rid] + f.y;
        r->z = lo; r->w = lo + cnt - 1u;
    }
}

// ===================================================================================== scan + gather
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__device__ __forceinline__ unsigned long long block_exclusive_scan(unsigned long long v, unsigned long long* total) {
    __shared__ unsigned long long warp_sums[SCAN_THREADS / 32];
    __shared__ unsigned long long tot;
    const uint32_t lane = threadIdx.x & 31u, wid = threadIdx.x >> 5;
    unsigned long long x = v;
    for (int d = 1; d < 32; d <<= 1) {
        unsigned long long y = __shfl_up_sync(FULL, x, d);
        if (lane >= (uint32_t)d) x += y;
    }
    if (lane == 31) warp_sums[wid] = x;
    __syncthreads();
    if (wid == 0) {
        unsigned long long s = lane < SCAN_THREADS / 32 ? warp_sums[lane] : 0ull;
        for (int d = 1; d < 32; d <<= 1) {
            unsigned long long y = __shfl_up_sync(FULL, s, d);
            if (lane >= (uint32_t)d) s += y;
        }
        if (lane < SCAN_THREADS / 32) warp_sums[lane] = s;
        if (lane == SCAN_THREADS / 32 - 1) tot = s;
    }
    __syncthreads();
    unsigned long long base = wid ? warp_sums[wid - 1] : 0ull;
    *total = tot;
    unsigned long long r = base + x - v;
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_tiles(const uint32_t* cnt, uint64_t n, unsigned long long* off, unsigned long long* tile_sums) {
    const uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE + (uint64_t)threadIdx.x * SCAN_ITEMS;
    unsigned long long v[SCAN_ITEMS], sum = 0;
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        v[i] = (base + i < n) ? cnt[base + i] : 0u;
        sum += v[i];
    }
    unsigned long long total;
    unsigned long long ex = block_exclusive_scan(sum, &total);
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i) {
        if (base + i < n) off[base + i] = ex;
        ex += v[i];
    }
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_top(unsigned long long* tile_sums, uint64_t n_tiles, unsigned long long* grand_total) {
    unsigned long long carry = 0;
    for (uint64_t b = 0; b < n_tiles; b += SCAN_THREADS) {
        unsigned long long v = (b + threadIdx.x < n_tiles) ? tile_sums[b + threadIdx.x] : 0ull;
        unsigned long long total;
        unsigned long long ex = block_exclusive_scan(v, &total);
        if (b + threadIdx.x < n_tiles) tile_sums[b + threadIdx.x] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) *grand_total = carry;
}

__global__ void k_gather_advance(unsigned long long* base, const unsigned long long* rank_counts, uint32_t world) {
    unsigned long long t = 0;
    for (uint32_t r = 0; r < world; ++r) t += rank_counts[r];
    *base += t;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_add(unsigned long long* off, uint64_t n, const unsigned long long* tile_sums, const unsigned long long* grand_total) {
    const uint64_t base = (uint64_t)blockIdx.x * SCAN_TILE + (uint64_t)threadIdx.x * SCAN_ITEMS;
    const unsigned long long add = tile_sums[blockIdx.x];
#pragma unroll
    for (int i = 0; i < SCAN_ITEMS; ++i)
        if (base + i < n) off[base + i] += add;
    if (blockIdx.x == 0 && threadIdx.x == 0) off[n] = *grand_total;
}

// Records in (read, emission) order.  `out` may be another GPU's memory (gsm_peer_open): then these stores ARE the
// gather of the multi-GPU path, over NVLink.  The batch's first record goes to out[*base + sum(rank_counts[0..rank))]:
// rank_counts = the all-gathered per-rank record counts of this batch, *base = records of earlier batches (both device
// memory, either may be NULL = 0), so no host round trip sits between the selection and the write.
__global__ void k_gather_records(const uint4* rec_tmp, const uint32_t* tmp_off, const uint32_t* cnt, const unsigned long long* off,
                                 uint64_t n_reads, uint4* out, unsigned long long out_cap, unsigned long long* counters,
                                 const unsigned long long* rank_counts, uint32_t rank, const unsigned long long* base,
                                 const uint4* mem_pool, const uint32_t* mem_off, const uint32_t* mem_cnt, uint32_t read_id_base) {
    // four lanes per read: records are 16 bytes, a read has a handful of them
    const uint64_t q = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 2;
    const uint32_t ql = threadIdx.x & 3u;
    if (q >= n_reads) return;
    unsigned long long first = base ? *base : 0ull;
    for (uint32_t r = 0; rank_counts && r < rank; ++r) first += rank_counts[r];
    const uint32_t n = cnt[q];
    const unsigned long long dst = first + off[q];
    if (dst + n > out_cap) { if (ql == 0 && n) atomicOr(&counters[2], 4ull); return; }
    const uint32_t src = tmp_off[q];
    if (counters[5] != 0ull && (mem_cnt[q] & MEMS_PICKED)) {
        // BWA-SMEM on a list the sweep picked from (k_select_bwa_picked): src = the picks; record k = the k-th picked entry
        const uint32_t nm = mem_cnt[q] & MEMS_COUNT;
        const uint32_t* seg = reinterpret_cast<const uint32_t*>(mem_pool + mem_off[q]);
        for (uint32_t k = ql; k < n; k += 4) {
            const uint32_t b = __fns(src, 0u, (int)k + 1);
            const uint32_t lo = seg[nm + b];
            out[dst + k] = make_uint4(read_id_base + (uint32_t)q, seg[b], lo, lo + seg[2u * nm + b] - 1u);
        }
        return;
    }
    for (uint32_t k = ql; k < n; k += 4) out[dst + k] = rec_tmp[(size_t)src + k];
}

// ===================================================================================== batched primitives
struct BackArgs {
    const uint4* fwd;
    IndexMeta meta;
    const uint32_t* reads;
    const uint32_t* chunk_off;
    const uint32_t* len;
    uint64_t n_reads;
    uint32_t* lo;
    uint32_t* cnt;
};

// exact_match_back_prop (reference SMEM/ExactMatch.py:132-151): one lane pair per read.
__global__ void __launch_bounds__(128) k_backsearch(const BackArgs a) {
    const uint64_t q = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    const uint32_t ql = threadIdx.x & 1u;
    const bool valid = q < a.n_reads;
    uint32_t L = 0;
    const uint32_t* w = a.reads;
    if (valid) { L = __ldg(a.len + q); w = a.reads + (size_t)__ldg(a.chunk_off + q) * 4; }
    uint32_t lo = 0, cnt = a.meta.n_rows;
    int32_t p = (int32_t)L - 1;
    for (;;) {
        const bool act = valid && p >= 0 && cnt != 0;
        if (!__any_sync(FULL, act)) break;
        uint32_t ch = 0;
        if (act) ch = (__ldg(w + (p >> 4)) >> (30u - 2u * ((uint32_t)p & 15u))) & 3u;
        StepOut r = pair_step(a.fwd, lo, lo + cnt, ch, a.meta.C[ch], a.meta.prim_f, ql, act);
        if (act) { lo = r.lo_new; cnt = r.cnt_new; --p; }
    }
    if (valid && ql == 0) { a.lo[q] = lo; a.cnt[q] = cnt; }
}

// exact_match_back_prop_add_one (reference SMEM/ExactMatch.py:155-171)
__global__ void __launch_bounds__(128) k_add_one(const uint4* fwd, IndexMeta meta, uint64_t n, const uint8_t* base, uint32_t* lo, uint32_t* cnt) {
    const uint64_t q = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    const uint32_t ql = threadIdx.x & 1u;
    const bool act = q < n && cnt[q] != 0;
    uint32_t l = 0, c = 0, ch = 0;
    if (act) { l = lo[q]; c = cnt[q]; ch = base[q] & 3u; }
    StepOut r = pair_step(fwd, l, l + c, ch, meta.C[ch], meta.prim_f, ql, act);
    if (act && ql == 0) { lo[q] = r.lo_new; cnt[q] = r.cnt_new; }
}

// get_position(s) (reference SMEM/ExactMatch.py:191-199)
__global__ void k_sa_lookup(const uint32_t* sa, uint64_t n_rows, uint64_t n, const uint32_t* rows, uint32_t* pos) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) pos[i] = rows[i] < n_rows ? __ldg(sa + rows[i]) : 0u;
}

// LUT.generate_lut (reference SMEM/LUT.py:15-35) as a dense table: one thread per k-mer code.
// Sampled suffix array (the "2-bit BWT + sampled SA" index of BASELINE.json configs[3]): ssa[i] = suffix_array[i * S].
__global__ void k_sa_sample(const uint32_t* sa, uint64_t n_rows, uint32_t S, uint32_t* ssa) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i * S < n_rows) ssa[i] = __ldg(sa + i * S);
}

// row -> 1-based text position without the full suffix array: walk LF until a sampled row (or the '$' row) is reached.
// ExactMatch.get_position(s) (ExactMatch.py:191-199); expected (S-1)/2 bucket fetches per row.
__global__ void __launch_bounds__(128) k_locate_sampled(const uint4* fwd, IndexMeta meta, const uint32_t* ssa, uint32_t S, uint64_t n,
                                                         const uint32_t* rows, uint32_t* pos) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    auto load = [fwd](uint64_t idx) { return ldg_half(fwd, idx); };
    uint32_t r = __ldg(rows + i), t = 0;
    if (r >= meta.n_rows) { pos[i] = 0u; return; }
    for (;;) {
        if (r == meta.prim_f) { pos[i] = 1u + t; return; }
        if (r % S == 0u) { pos[i] = __ldg(ssa + r / S) + t; return; }
        r = lf_single(load, r, meta.C, meta.prim_f);
        ++t;
    }
}

__global__ void k_lut_build(const uint4* fwd, IndexMeta meta, uint32_t K, uint64_t n_codes, uint2* table) {
    const uint64_t code = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (code >= n_codes) return;
    auto load = [fwd](uint64_t idx) { return ldg_half(fwd, idx); };
    uint32_t lo = 0, cnt = meta.n_rows;
    for (uint32_t t = 0; t < K && cnt; ++t) {
        const uint32_t c = (uint32_t)(code >> (2 * t)) & 3u;      // backward search: last base first
        StepOut r = step_single(load, lo, lo + cnt, c, meta.C[c], meta.prim_f);
        lo = r.lo_new; cnt = r.cnt_new;
    }
    table[code] = make_uint2(lo, cnt);
}

// Seed table of the sweep kernel: per K-mer code the rows of the k-mer on the text index, its count, and the rows
// of the reversed k-mer on the reversed-text index -- the state (k, P0, cnt) a forward extension has after K steps.
__global__ void k_seed_build(const uint4* fwd, const uint4* rev, IndexMeta meta, uint32_t K, uint64_t n_codes, uint4* table) {
    const uint64_t code = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (code >= n_codes) return;
    auto lf = [fwd](uint64_t idx) { return ldg_half(fwd, idx); };
    auto lr = [rev](uint64_t idx) { return ldg_half(rev, idx); };
    uint32_t lo = 0, cnt = meta.n_rows, rlo = 0, rcnt = meta.n_rows;
    for (uint32_t t = 0; t < K; ++t) {                                        // through empty intervals too: lo ends as the insertion point
        const uint32_t c = (uint32_t)(code >> (2 * t)) & 3u;                  // last base first
        const StepOut r = step_single(lf, lo, lo + cnt, c, meta.C[c], meta.prim_f);
        lo = r.lo_new; cnt = r.cnt_new;
    }
    for (uint32_t t = 0; t < K && rcnt && cnt; ++t) {
        const uint32_t c = (uint32_t)(code >> (2 * (K - 1 - t))) & 3u;        // first base first
        const StepOut r = step_single(lr, rlo, rlo + rcnt, c, meta.C[c], meta.prim_r);
        rlo = r.lo_new; rcnt = r.cnt_new;
    }
    table[code] = make_uint4(lo, cnt, cnt ? rlo : 0u, 0u);
}

// bounds[code] = {first row >= the K-mer, its occurrences}: what kmer_bounds_seeded computes per window, for every code.
// With a seed table (seed_K <= K) a thread starts from the entry of its code's last seed_K bases (consecutive codes:
// consecutive entries) and takes the remaining K - seed_K backward steps, through empty intervals too.
__global__ void k_bounds_build(const uint4* fwd, IndexMeta meta, uint32_t K, uint64_t n_codes, const uint4* seed_tab, uint32_t seed_K,
                               uint2* table) {
    const uint64_t code = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (code >= n_codes) return;
    auto load = [fwd](uint64_t idx) { return ldg_half(fwd, idx); };
    uint32_t lo = 0, cnt = meta.n_rows, t = 0;
    if (seed_tab) {
        const uint4 e = __ldg(seed_tab + (code & ((1ull << (2u * seed_K)) - 1ull)));
        lo = e.x; cnt = e.y; t = seed_K;
    }
    for (; t < K; ++t) {
        const uint32_t c = (uint32_t)(code >> (2 * t)) & 3u;                  // last base first
        const StepOut r = step_single(load, lo, lo + cnt, c, meta.C[c], meta.prim_f);
        lo = r.lo_new; cnt = r.cnt_new;
    }
    table[code] = make_uint2(lo, cnt);
}

// RMI_LUT.get_suffix_rmi (reference SMEM/RMI_LUT.py:67-78) for a batch of codes
__global__ void k_rmi_lookup(const uint32_t* sa, const uint32_t* text, uint64_t n_rows, uint64_t n_bases, RmiModel m, uint64_t n,
                             const uint64_t* codes, double* pred, int64_t* lo, int64_t* hi, uint8_t* status) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    auto sal = [sa](uint64_t r) { return __ldg(sa + r); };
    auto txl = [text](uint64_t w) { return __ldg(text + w); };
    SaTextProbe<decltype(sal), decltype(txl)> pr{sal, txl};
    RmiTable<decltype(pr)> t{pr, (int64_t)n_rows, (int64_t)n_bases, m.K, false};
    double p; int64_t l, h;
    t.lookup(m, codes[i], p, l, h);
    pred[i] = p; lo[i] = l; hi[i] = h;
    status[i] = t.raised ? GSM_READ_REF_RAISES : GSM_READ_OK;
}

// rows whose suffix is shorter than K (RMI_LUT.get_ref_seq returns None there): out[0] = count, out[1..] = rows
__global__ void k_none_rows(const uint32_t* sa, uint64_t n_rows, uint32_t K, uint32_t* out) {
    const uint64_t row = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_rows) return;
    if ((uint64_t)__ldg(sa + row) - 1u + K > n_rows - 1u) {
        const uint32_t slot = atomicAdd(out, 1u);
        if (slot < 32u) out[1 + slot] = (uint32_t)row;
    }
}

// {suffix_array[row], code of the 32 bases at that suffix}: makes RMI_LUT.get_ref_seq one 16-byte fetch.
__global__ void k_rmi_probe_build(const uint32_t* sa, const uint32_t* text, uint64_t n_rows, uint4* out) {
    const uint64_t row = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_rows) return;
    const uint32_t s = __ldg(sa + row);
    auto txl = [text](uint64_t w) { return __ldg(text + w); };
    const uint64_t code = kmer_code(txl, (uint64_t)(s - 1), 32);
    out[row] = make_uint4(s, (uint32_t)(code >> 32), (uint32_t)code, 0u);
}

// Random aligned 64-byte gather with the rank kernels' access shape (lane pair = 2 x 32 B).
// dependent != 0: each pair runs a pointer chase (latency-bound, like one FM chain);
// dependent == 0: independent fetches (the bandwidth ceiling for 64-byte random access).
__global__ void __launch_bounds__(128) k_gather_probe(const uint4* buf, uint64_t n_buckets, uint32_t iters, uint32_t dependent, unsigned long long* sink) {
    const uint64_t gq = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    const uint32_t g = threadIdx.x & 1u;
    uint64_t state = gq * 0x9E3779B97F4A7C15ull + 0x1234567ull;
    uint32_t acc = 0;
    for (uint32_t it = 0; it < iters; ++it) {
        state = state * 6364136223846793005ull + 1442695040888963407ull;
        uint64_t idx = (state >> 17) % n_buckets;
        Half v = ldg_half(buf, idx * 2 + g);
        uint32_t x = v.c0 ^ v.c1 ^ v.l0 ^ v.l1 ^ v.l2 ^ v.h0 ^ v.h1 ^ v.h2;
        acc += x;
        if (dependent) {
            x ^= __shfl_xor_sync(FULL, x, 1);
            state ^= x;
        }
    }
    if (acc == 0x7FFFFFFFu) atomicAdd(sink, 1ull);
}

// The same ceiling measured without the probe's own bottlenecks (VERDICT r1): U independent fetches in flight per lane,
// power-of-two masking instead of a 64-bit modulo, and the access shapes the kernels really use -- BYTES = 64 (one lane
// reads a whole bucket: two 256-bit loads, k_sweep1 / k_locate_sampled), 32 (one 256-bit load), 16 (one seed-table entry).
template <int BYTES, int U, int PF = 0>      // PF == 1: 64-byte fetches by lane PAIRS (one load instruction, one request per bucket)
__global__ void __launch_bounds__(128) k_gather_probe2(const uint4* buf, uint64_t unit_mask, uint32_t iters, unsigned long long* sink) {
    const uint64_t gt = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t state = gt * 0x9E3779B97F4A7C15ull + 0x1234567ull;
    uint32_t acc = 0;
    for (uint32_t it = 0; it < iters; ++it) {
        uint64_t idx[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            state = state * 6364136223846793005ull + 1442695040888963407ull;
            idx[u] = (state >> 20) & unit_mask;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (BYTES == 16) {
                const uint4 v = ldg_seed(buf + idx[u]);
                acc += v.x ^ v.y ^ v.z ^ v.w;
            } else {
                if (PF == 1) {               // the pair shares the even lane's index: each lane loads one half of that bucket
                    const uint64_t shared_idx = __shfl_sync(0xFFFFFFFFu, idx[u], threadIdx.x & 30u);
                    const Half hp = ldg_half(buf, shared_idx * 2 + (threadIdx.x & 1u));
                    acc += hp.c0 ^ hp.c1 ^ hp.l0 ^ hp.l1 ^ hp.l2 ^ hp.h0 ^ hp.h1 ^ hp.h2;
                    continue;
                }
                const Half h0 = ldg_half(buf, idx[u] * (BYTES / 32));
                acc += h0.c0 ^ h0.c1 ^ h0.l0 ^ h0.l1 ^ h0.l2 ^ h0.h0 ^ h0.h1 ^ h0.h2;
                if (BYTES == 64) {
                    const Half h1 = ldg_half(buf, idx[u] * 2 + 1);
                    acc += h1.c0 ^ h1.c1 ^ h1.l0 ^ h1.l1 ^ h1.l2 ^ h1.h0 ^ h1.h1 ^ h1.h2;
                }
            }
        }
    }
    if (acc == 0x7FFFFFFFu) atomicAdd(sink, 1ull);
}

}  // namespace gsm

// ===================================================================================== C ABI
using namespace gsm;

namespace {

IndexMeta make_meta(const gsm_dev_index* ix) {
    IndexMeta m;
    for (int c = 0; c < 4; ++c) { m.C[c] = ix->C[c]; m.cnt[c] = ix->C[c + 1] - ix->C[c]; }
    m.prim_f = ix->primary_fwd; m.prim_r = ix->primary_rev; m.n_rows = (uint32_t)ix->n_rows;
    return m;
}

int device_ready() {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(GSM_E_NODEVICE, "no CUDA device visible: libgenie_smem has no CPU fallback");
    }
    return GSM_OK;
}

// Which sweep kernel runs a batch: k_sweep1<false> with the read in shared memory for reads up to SWEEP1_SMEM_MAX_LEN
// bases, k_sweep1<true> (bases from global memory, grid sized by the staging budget) for anything longer, up to 65535
// bases; UNIQ when the suffix array and the packed text are on the device (the unique-match shortcut).
using SweepKernel = void (*)(const SweepArgs);
bool sweep_long(uint32_t max_len) { return max_len > SWEEP1_SMEM_MAX_LEN; }
SweepKernel sweep_kernel(bool long_reads, bool uniq) {
    if (long_reads) return uniq ? k_sweep1<true, true> : k_sweep1<true, false>;
    return uniq ? k_sweep1<false, true> : k_sweep1<false, false>;
}

int sweep_grid(uint32_t max_len, int* blocks) {
    int dev = 0, sms = 0;
    GSM_CUDA(cudaGetDevice(&dev));
    GSM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const bool long_reads = sweep_long(max_len);
    const size_t smem = sweep1_smem_bytes(max_len, long_reads);
    int a[2] = {0, 0};                  // the grid must be resident for either instantiation (with / without the text shortcut)
    for (int uniq = 0; uniq < 2; ++uniq) {
        const SweepKernel k = sweep_kernel(long_reads, uniq != 0);
        GSM_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        GSM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a[uniq], k, SWEEP1_THREADS, smem));
    }
    const int per_sm = a[0] < a[1] ? a[0] : a[1];
    if (per_sm < 1) return fail(GSM_E_CAPACITY, "read length too large for the sweep kernel's shared memory");
    *blocks = sms * per_sm;
    if (long_reads) {                   // long reads: as many blocks as the staging budget allows (2 x max_len x 16 B per lane)
        const uint64_t fit = SWEEP1_LONG_SCRATCH / ((uint64_t)SWEEP1_THREADS * 2ull * max_len * 16ull);
        if ((uint64_t)*blocks > fit) *blocks = fit < 1 ? 1 : (int)fit;
    }
    return GSM_OK;
}

uint64_t sweep_scratch_bytes(int blocks, uint32_t max_len) { return (uint64_t)blocks * SWEEP1_THREADS * 2ull * max_len * 16ull; }

uint32_t select_stage_stride(uint32_t max_len) { return max_len < SELECT_STAGE ? max_len : SELECT_STAGE; }

int select_grid(int* blocks) {          // upper bound over the selection kernels: sizes the per-thread record staging
    int dev = 0, sms = 0;
    GSM_CUDA(cudaGetDevice(&dev));
    GSM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    *blocks = sms * 8;
    return GSM_OK;
}

// resident grid of one selection kernel: a persistent grid-stride kernel must not spill into a second wave
template <typename Kern>
int resident_grid(Kern kern, int threads, size_t smem, int cap, int* blocks) {
    int dev = 0, sms = 0, per_sm = 0;
    GSM_CUDA(cudaGetDevice(&dev));
    GSM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    GSM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
    if (per_sm < 1) per_sm = 1;
    *blocks = sms * per_sm < cap ? sms * per_sm : cap;
    return GSM_OK;
}

template <int METHOD, int ARITH>
int launch_seeded(const SelectArgs& se, int cap, cudaStream_t stream) {
    int grid = cap;
    const size_t smem = select_smem_bytes(se.K);                          // at most 44 KB (K <= 32)
    const int st = resident_grid(k_select_seeded<METHOD, ARITH>, SELECT_THREADS, smem, cap, &grid);
    if (st) return st;
    k_select_seeded<METHOD, ARITH><<<grid, SELECT_THREADS, smem, stream>>>(se);
    return GSM_OK;
}

}  // namespace

uint64_t gsm::scan_tmp_bytes(uint64_t n) { return ((n + SCAN_TILE - 1) / SCAN_TILE + 2) * 8ull; }

int gsm::scan_counts(const uint32_t* cnt, uint64_t n, uint64_t* off, void* tmp, uint64_t tmp_bytes, void* stream) {
    cudaStream_t s = (cudaStream_t)stream;
    if (n == 0) {
        GSM_CUDA(cudaMemsetAsync(off, 0, sizeof(uint64_t), s));
        return GSM_OK;
    }
    if (tmp_bytes < scan_tmp_bytes(n)) return fail(GSM_E_CAPACITY, "scan_tmp too small");
    const uint64_t n_tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    unsigned long long* tiles = (unsigned long long*)tmp;
    k_scan_tiles<<<(unsigned)n_tiles, SCAN_THREADS, 0, s>>>(cnt, n, (unsigned long long*)off, tiles);
    k_scan_top<<<1, SCAN_THREADS, 0, s>>>(tiles, n_tiles, tiles + n_tiles);
    k_scan_add<<<(unsigned)n_tiles, SCAN_THREADS, 0, s>>>((unsigned long long*)off, n, tiles, tiles + n_tiles);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

extern "C" {

int gsm_smem_workspace_info(uint64_t n_reads, uint32_t max_len, gsm_workspace_info* out) {
    if (!out || max_len == 0 || max_len > 65535) return fail(GSM_E_INVALID, "gsm_smem_workspace_info: max_len must be in 1..65535");
    int st = device_ready();
    if (st) return st;
    int sb = 0, lb = 0;
    if ((st = sweep_grid(max_len, &sb))) return st;
    if ((st = select_grid(&lb))) return st;
    const uint64_t sweep_bytes = sweep_scratch_bytes(sb, max_len);
    const uint64_t sel_bytes = (uint64_t)lb * SELECT_THREADS * (uint64_t)select_stage_stride(max_len) * 16ull;
    out->quad_scratch_bytes = sweep_bytes > sel_bytes ? sweep_bytes : sel_bytes;
    out->scan_tmp_bytes = ((n_reads + SCAN_TILE - 1) / SCAN_TILE + 2) * 8ull;
    out->grid_blocks = (uint32_t)sb;
    out->block_threads = SWEEP1_THREADS;
    return GSM_OK;
}

int gsm_backsearch_batch(const gsm_dev_index* ix, const gsm_dev_reads* rd, uint32_t* lo, uint32_t* cnt, void* stream) {
    if (!ix || !rd || !lo || !cnt) return fail(GSM_E_INVALID, "null");
    int st = device_ready();
    if (st) return st;
    if (rd->n_reads == 0) return GSM_OK;
    BackArgs a{(const uint4*)ix->fwd_buckets, make_meta(ix), (const uint32_t*)rd->packed, rd->chunk_off, rd->len, rd->n_reads, lo, cnt};
    const uint64_t threads = rd->n_reads * 2;
    k_backsearch<<<(unsigned)((threads + 127) / 128), 128, 0, (cudaStream_t)stream>>>(a);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

int gsm_backsearch_add_one_batch(const gsm_dev_index* ix, uint64_t n, const uint8_t* base, uint32_t* lo, uint32_t* cnt, void* stream) {
    if (!ix || !base || !lo || !cnt) return fail(GSM_E_INVALID, "null");
    int st = device_ready();
    if (st) return st;
    if (n == 0) return GSM_OK;
    k_add_one<<<(unsigned)((n * 2 + 127) / 128), 128, 0, (cudaStream_t)stream>>>((const uint4*)ix->fwd_buckets, make_meta(ix), n, base, lo, cnt);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

int gsm_sa_lookup_batch(const gsm_dev_index* ix, uint64_t n, const uint32_t* rows, uint32_t* pos, void* stream) {
    if (!ix || !ix->sa || !rows || !pos) return fail(GSM_E_INVALID, "gsm_sa_lookup_batch needs the suffix array on the device");
    int st = device_ready();
    if (st) return st;
    if (n == 0) return GSM_OK;
    k_sa_lookup<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ix->sa, ix->n_rows, n, rows, pos);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

int gsm_sa_sample_build(const gsm_dev_index* ix, uint32_t sample, uint32_t* ssa, void* stream) {
    if (!ix || !ix->sa || !ssa || sample == 0) return fail(GSM_E_INVALID, "gsm_sa_sample_build: needs the full suffix array on the device and sample >= 1");
    int st = device_ready();
    if (st) return st;
    const uint64_t n = (ix->n_rows + sample - 1) / sample;
    k_sa_sample<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ix->sa, ix->n_rows, sample, ssa);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

int gsm_locate_sampled_batch(const gsm_dev_index* ix, const uint32_t* ssa, uint32_t sample, uint64_t n, const uint32_t* rows, uint32_t* pos,
                             void* stream) {
    if (!ix || !ix->fwd_buckets || !ssa || sample == 0 || (n && (!rows || !pos))) return fail(GSM_E_INVALID, "gsm_locate_sampled_batch: null");
    int st = device_ready();
    if (st) return st;
    if (n == 0) return GSM_OK;
    k_locate_sampled<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>((const uint4*)ix->fwd_buckets, make_meta(ix), ssa, sample, n, rows, pos);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

int gsm_lut_build(const gsm_dev_index* ix, uint32_t K, uint32_t* table, void* stream) {
    if (!ix || !table || K < 1 || K > 16) return fail(GSM_E_INVALID, "gsm_lut_build: K must be in 1..16");
    int st = device_ready();
    if (st) return st;
    const uint64_t n_codes = 1ull << (2 * K);
    k_lut_build<<<(unsigned)((n_codes + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const uint4*)ix->fwd_buckets, make_meta(ix), K, n_codes, (uint2*)table);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

int gsm_device_l2_fetch_granularity(int32_t set_bytes, uint32_t* current) {
    int st = device_ready();
    if (st) return st;
    if (set_bytes > 0) GSM_CUDA(cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)set_bytes));
    size_t v = 0;
    GSM_CUDA(cudaDeviceGetLimit(&v, cudaLimitMaxL2FetchGranularity));
    if (current) *current = (uint32_t)v;
    return GSM_OK;
}

int gsm_l2_persist(const void* ptr, uint64_t bytes, void* stream) {
    int st = device_ready();
    if (st) return st;
    int dev = 0, max_win = 0, max_persist = 0;
    GSM_CUDA(cudaGetDevice(&dev));
    GSM_CUDA(cudaDeviceGetAttribute(&max_win, cudaDevAttrMaxAccessPolicyWindowSize, dev));
    GSM_CUDA(cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, dev));
    cudaStreamAttrValue v;
    memset(&v, 0, sizeof(v));
    if (ptr && bytes) {
        if (max_win <= 0 || max_persist <= 0) return fail(GSM_E_INVALID, "gsm_l2_persist: the device has no persisting L2");
        const uint64_t carve = bytes < (uint64_t)max_persist ? bytes : (uint64_t)max_persist;
        GSM_CUDA(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, (size_t)carve));
        v.accessPolicyWindow.base_ptr = const_cast<void*>(ptr);
        v.accessPolicyWindow.num_bytes = (size_t)(bytes < (uint64_t)max_win ? bytes : (uint64_t)max_win);
        v.accessPolicyWindow.hitRatio = bytes <= carve ? 1.0f : (float)carve / (float)bytes;
        v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        v.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    }   // else: an empty window removes the policy from the stream
    GSM_CUDA(cudaStreamSetAttribute((cudaStream_t)stream, cudaStreamAttributeAccessPolicyWindow, &v));
    if (!(ptr && bytes)) GSM_CUDA(cudaCtxResetPersistingL2Cache());
    return GSM_OK;
}

int gsm_seed_table_build(const gsm_dev_index* ix, uint32_t K, void* table, void* stream) {
    if (!ix || !table || !ix->fwd_buckets || !ix->rev_buckets) return fail(GSM_E_INVALID, "gsm_seed_table_build: needs both bucket arrays");
    if (K < 1 || K > 14) return fail(GSM_E_INVALID, "gsm_seed_table_build: K must be in 1..14");
    int st = device_ready();
    if (st) return st;
    const uint64_t n_codes = 1ull << (2 * K);
    k_seed_build<<<(unsigned)((n_codes + 127) / 128), 128, 0, (cudaStream_t)stream>>>((const uint4*)ix->fwd_buckets, (const uint4*)ix->rev_buckets,
                                                                                    make_meta(ix), K, n_codes, (uint4*)table);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

static int fill_rmi(const gsm_dev_rmi* rmi, RmiModel* m, uint64_t n_rows) {
    memset(m, 0, sizeof(*m));
    if (!rmi || !rmi->level_sizes || !rmi->coef || !rmi->intercept) return fail(GSM_E_INVALID, "RMI parameters missing");
    if (rmi->n_levels < 1 || rmi->n_levels > 8 || rmi->K < 1 || rmi->K > 32) return fail(GSM_E_INVALID, "RMI: 1..8 levels, K in 1..32");
    m->K = rmi->K; m->n_levels = rmi->n_levels; m->coef = rmi->coef; m->intercept = rmi->intercept;
    m->stride = rmi->param_stride ? rmi->param_stride : 1u;
    uint32_t off = 0;
    for (uint32_t l = 0; l < rmi->n_levels; ++l) { m->level_size[l] = rmi->level_sizes[l]; m->level_off[l] = off; off += rmi->level_sizes[l]; }
    if (rmi->none_rows && rmi->n_none_rows) {
        if (rmi->n_none_rows != rmi->K) return fail(GSM_E_INVALID, "RMI: none_rows must hold exactly K rows (gsm_rmi_none_rows)");
        rmi_set_none_rows(*m, rmi->none_rows, rmi->n_none_rows, n_rows);
    }
    return GSM_OK;
}

int gsm_rmi_none_rows(const gsm_dev_index* ix, uint32_t K, uint32_t* rows_host, uint32_t* scratch, void* stream) {
    if (!ix || !ix->sa || !rows_host || !scratch || K < 1 || K > 32) return fail(GSM_E_INVALID, "gsm_rmi_none_rows: needs sa on the device, K in 1..32");
    int st = device_ready();
    if (st) return st;
    if (ix->n_rows <= K) return fail(GSM_E_INVALID, "gsm_rmi_none_rows: reference shorter than K");
    cudaStream_t s_ = (cudaStream_t)stream;
    GSM_CUDA(cudaMemsetAsync(scratch, 0, 33 * sizeof(uint32_t), s_));
    k_none_rows<<<(unsigned)((ix->n_rows + 255) / 256), 256, 0, s_>>>(ix->sa, ix->n_rows, K, scratch);
    GSM_CUDA(cudaGetLastError());
    uint32_t h[33];
    GSM_CUDA(cudaMemcpyAsync(h, scratch, sizeof(h), cudaMemcpyDeviceToHost, s_));
    GSM_CUDA(cudaStreamSynchronize(s_));
    if (h[0] != K) return fail(GSM_E_INVALID, "gsm_rmi_none_rows: the suffix array does not hold exactly K short suffixes");
    std::sort(h + 1, h + 1 + K);
    for (uint32_t t = 0; t < K; ++t) rows_host[t] = h[1 + t];
    return GSM_OK;
}

int gsm_rmi_bounds_build(const gsm_dev_index* ix, uint32_t K, void* bounds, void* stream) {
    if (!ix || !ix->fwd_buckets || !bounds || K < 1 || K > 16) return fail(GSM_E_INVALID, "gsm_rmi_bounds_build: needs the rank buckets and K in 1..16");
    int st = device_ready();
    if (st) return st;
    const uint64_t n_codes = 1ull << (2 * K);
    const bool seeded = ix->seed_table && ix->seed_K >= 1 && ix->seed_K <= K;
    k_bounds_build<<<(unsigned)((n_codes + 255) / 256), 256, 0, (cudaStream_t)stream>>>((const uint4*)ix->fwd_buckets, make_meta(ix), K, n_codes,
                                                                                       seeded ? (const uint4*)ix->seed_table : nullptr,
                                                                                       seeded ? ix->seed_K : 0u, (uint2*)bounds);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

int gsm_rmi_hazard_scan(const gsm_dev_index* ix, const gsm_dev_rmi* rmi, uint32_t* codes, uint64_t cap, uint64_t* count_dev,
                        uint64_t* n_found, void* stream) {
    if (!ix || !rmi || !rmi->bounds || !codes || !count_dev || !n_found || cap == 0)
        return fail(GSM_E_INVALID, "gsm_rmi_hazard_scan: needs the bounds table, a code buffer and a device counter");
    if (rmi->K < 1 || rmi->K > 15) return fail(GSM_E_INVALID, "gsm_rmi_hazard_scan: K in 1..15 (32-bit codes)");
    int st = device_ready();
    if (st) return st;
    RmiModel m;
    if ((st = fill_rmi(rmi, &m, ix->n_rows))) return st;
    if (m.n_none == 0u) return fail(GSM_E_INVALID, "gsm_rmi_hazard_scan: needs none_rows (gsm_rmi_none_rows)");
    cudaStream_t s_ = (cudaStream_t)stream;
    const uint64_t n_codes = 1ull << (2 * rmi->K);
    int dev = 0, sms = 148;
    GSM_CUDA(cudaGetDevice(&dev));
    GSM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    uint64_t blocks = (n_codes + 255) / 256;
    if (blocks > (uint64_t)sms * 64) blocks = (uint64_t)sms * 64;
    GSM_CUDA(cudaMemsetAsync(count_dev, 0, sizeof(uint64_t), s_));
    k_rmi_hazard_scan<<<(unsigned)blocks, 256, 0, s_>>>(m, (const uint2*)rmi->bounds, n_codes, (uint32_t)ix->n_rows, codes, cap,
                                                       (unsigned long long*)count_dev);
    GSM_CUDA(cudaGetLastError());
    GSM_CUDA(cudaMemcpyAsync(n_found, count_dev, sizeof(uint64_t), cudaMemcpyDeviceToHost, s_));
    GSM_CUDA(cudaStreamSynchronize(s_));
    return GSM_OK;
}

int gsm_rmi_hazard_hash(const uint32_t* codes, uint64_t n, uint32_t* slots, uint32_t n_slots) {
    if ((!codes && n) || !slots) return fail(GSM_E_INVALID, "gsm_rmi_hazard_hash: null");
    if (!hz_build(codes, n, slots, n_slots))
        return fail(GSM_E_INVALID, "gsm_rmi_hazard_hash: n_slots must be a power of two in [2 n + 2, 2^24] and no code may be 0xFFFFFFFF");
    return GSM_OK;
}

int gsm_rmi_probe_build(const gsm_dev_index* ix, void* probe, void* stream) {
    if (!ix || !ix->sa || !ix->text2bit || !probe) return fail(GSM_E_INVALID, "gsm_rmi_probe_build needs sa + text on the device");
    int st = device_ready();
    if (st) return st;
    k_rmi_probe_build<<<(unsigned)((ix->n_rows + 255) / 256), 256, 0, (cudaStream_t)stream>>>(ix->sa, ix->text2bit, ix->n_rows, (uint4*)probe);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

int gsm_rmi_lookup_batch(const gsm_dev_index* ix, const gsm_dev_rmi* rmi, uint64_t n, const uint64_t* codes, double* pred,
                         int64_t* lo, int64_t* hi, uint8_t* status, void* stream) {
    if (!ix || !ix->sa || !ix->text2bit || !codes || !pred || !lo || !hi || !status) return fail(GSM_E_INVALID, "gsm_rmi_lookup_batch: null argument (needs sa + text on the device)");
    int st = device_ready();
    if (st) return st;
    RmiModel m;
    if ((st = fill_rmi(rmi, &m, ix->n_rows))) return st;
    if (n == 0) return GSM_OK;
    k_rmi_lookup<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(ix->sa, ix->text2bit, ix->n_rows, ix->n_rows - 1, m, n, codes, pred, lo, hi, status);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

static int smem_check(const gsm_dev_index* ix, const gsm_dev_reads* rd, gsm_workspace* ws, int* sb, int* lb) {
    if (!ix || !rd || !ws) return fail(GSM_E_INVALID, "null");
    if (!ix->fwd_buckets || !ix->rev_buckets) return fail(GSM_E_INVALID, "the SMEM kernels need both BWT directions on the device");
    if (rd->max_len == 0 || rd->max_len > 65535) return fail(GSM_E_INVALID, "max_len must be in 1..65535");
    if (rd->n_reads >= (1ull << 32)) return fail(GSM_E_INVALID, "at most 2^32-1 reads per batch");
    if (ws->mem_cap >= (1ull << 32) || ws->rec_cap >= (1ull << 32)) return fail(GSM_E_INVALID, "pool capacities must be < 2^32 entries");
    int st = device_ready();
    if (st) return st;
    if ((st = sweep_grid(rd->max_len, sb))) return st;
    if ((st = select_grid(lb))) return st;
    const uint64_t need_sweep = sweep_scratch_bytes(*sb, rd->max_len);
    const uint64_t need_sel = (uint64_t)*lb * SELECT_THREADS * (uint64_t)select_stage_stride(rd->max_len) * 16ull;
    if (ws->quad_scratch_bytes < need_sweep || ws->quad_scratch_bytes < need_sel) return fail(GSM_E_CAPACITY, "quad_scratch too small (see gsm_smem_workspace_info)");
    const uint64_t n_tiles = (rd->n_reads + SCAN_TILE - 1) / SCAN_TILE;
    if (ws->scan_tmp_bytes < (n_tiles + 2) * 8) return fail(GSM_E_CAPACITY, "scan_tmp too small");
    return GSM_OK;
}

int gsm_smem_sweep(const gsm_dev_index* ix, const gsm_dev_reads* rd, gsm_workspace* ws, void* stream_) {
    int sb = 0, lb = 0;
    int st = smem_check(ix, rd, ws, &sb, &lb);
    if (st) return st;
    cudaStream_t stream = (cudaStream_t)stream_;
    GSM_CUDA(cudaMemsetAsync(ws->counters, 0, 8 * sizeof(uint64_t), stream));
    if (rd->n_reads == 0) return GSM_OK;
    SweepArgs sa;
    sa.fwd = (const uint4*)ix->fwd_buckets; sa.rev = (const uint4*)ix->rev_buckets; sa.meta = make_meta(ix);
    sa.reads = (const uint4*)rd->packed; sa.chunk_off = rd->chunk_off; sa.len = rd->len; sa.n_reads = (uint32_t)rd->n_reads;
    sa.max_len = rd->max_len;
    sa.seed_tab = (const uint4*)ix->seed_table; sa.seed_K = ix->seed_table ? ix->seed_K : 0u;
    if (sa.seed_tab && (sa.seed_K < 1 || sa.seed_K > 16)) return fail(GSM_E_INVALID, "seed table K must be in 1..16");
    sa.mem_pool = (uint4*)ws->mem_pool; sa.mem_cap = ws->mem_cap; sa.mem_off = ws->mem_off; sa.mem_cnt = ws->mem_cnt;
    sa.scratch = (uint4*)ws->quad_scratch; sa.counters = (unsigned long long*)ws->counters;
    sa.sa = ix->sa; sa.text = ix->text2bit; sa.n_bases = (uint32_t)(ix->n_rows - 1);
    const bool long_reads = sweep_long(rd->max_len);
    sweep_kernel(long_reads, ix->sa && ix->text2bit)<<<sb, SWEEP1_THREADS, sweep1_smem_bytes(rd->max_len, long_reads), stream>>>(sa);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

int gsm_option_rmi_prefilter(int on) {
    const int before = g_rmi_prefilter;
    if (on >= 0) g_rmi_prefilter = on ? 1 : 0;
    return before;
}

int gsm_option_lut_frame_machine(int on) {
    const int before = g_lut_frame_machine;
    if (on >= 0) g_lut_frame_machine = on ? 1 : 0;
    return before;
}

int gsm_smem_select(int method, const gsm_dev_index* ix, const gsm_dev_reads* rd, uint32_t min_len, uint32_t K, const uint32_t* lut,
                    const gsm_dev_rmi* rmi, gsm_workspace* ws, void* stream_) {
    int sb = 0, lb = 0;
    int st = smem_check(ix, rd, ws, &sb, &lb);
    if (st) return st;
    if (method < 0 || method > 2) return fail(GSM_E_INVALID, "unknown method");
    if (method == GSM_METHOD_LUT && (!lut || K < 1 || K > 16)) return fail(GSM_E_INVALID, "LUT method needs a table and K in 1..16");
    RmiModel rm;
    memset(&rm, 0, sizeof(rm));
    if (method == GSM_METHOD_RMI) {
        if ((st = fill_rmi(rmi, &rm, ix->n_rows))) return st;
        if (!ix->sa || !ix->text2bit) return fail(GSM_E_INVALID, "RMI method needs the suffix array and packed text on the device");
        K = rmi->K;
    }
    cudaStream_t stream = (cudaStream_t)stream_;
    if (rd->n_reads == 0) {
        GSM_CUDA(cudaMemsetAsync(ws->rec_off, 0, sizeof(uint64_t), stream));
        return GSM_OK;
    }
    SelectArgs se;
    se.fwd = (const uint4*)ix->fwd_buckets; se.meta = make_meta(ix); se.n_bases = ix->n_rows - 1; se.sa = ix->sa; se.text = ix->text2bit; se.probe = (method == GSM_METHOD_RMI && rmi) ? (const uint4*)rmi->probe : nullptr;
    se.reads = (const uint32_t*)rd->packed; se.chunk_off = rd->chunk_off; se.len = rd->len; se.n_reads = (uint32_t)rd->n_reads;
    // LUT-SMEM emits exactly the records of BWA-SMEM with min_len 1 for every read of at least K bases (DESIGN.md section 3:
    // each round of get_smems_lut returns the longest maximal match covering the previous SMEM's end, ties to the smaller end,
    // which is get_SMEMS's pick): unless the frame machine is asked for (gsm_option_lut_frame_machine) the records are the
    // sweep's picks, and K only decides which reads are too short.
    const bool lut_as_picks = method == GSM_METHOD_LUT && g_lut_frame_machine == 0;
    if (lut_as_picks) { method = GSM_METHOD_BWA; min_len = 1; }
    else if (method == GSM_METHOD_BWA) K = 0;
    se.max_len = rd->max_len; se.read_id_base = rd->read_id_base; se.min_len = min_len; se.K = K; se.lut = (const uint2*)lut; se.rmi = rm;
    se.rmi_bounds = (method == GSM_METHOD_RMI && rmi && rm.n_none != 0u && K <= 16) ? (const uint2*)rmi->bounds : nullptr;
    se.seed_tab = (const uint4*)ix->seed_table; se.seed_K = ix->seed_table ? ix->seed_K : 0u;
    se.mem_pool = (uint4*)ws->mem_pool; se.mem_off = ws->mem_off; se.mem_cnt = ws->mem_cnt; se.stage = (uint4*)ws->quad_scratch; se.stage_stride = select_stage_stride(rd->max_len);
    se.rec_tmp = (uint4*)ws->rec_tmp; se.rec_cap = ws->rec_cap; se.rec_tmp_off = ws->rec_tmp_off; se.rec_cnt = ws->rec_cnt;
    se.read_status = ws->read_status; se.counters = (unsigned long long*)ws->counters;
    se.fix = nullptr; se.fix_cap = 0;
    se.hz_slots = nullptr; se.hz_mask = 0u; se.only_pending = 0u;
    if (method != GSM_METHOD_BWA) {           // deferred explicit searches queue in the last eighth of the record pool (at most one per read)
        const uint64_t reserve = ws->rec_cap / 8 < rd->n_reads ? ws->rec_cap / 8 : rd->n_reads;
        se.rec_cap = ws->rec_cap - reserve;
        se.fix = (uint4*)ws->rec_tmp + se.rec_cap; se.fix_cap = reserve;
    }
    GSM_CUDA(cudaMemsetAsync((unsigned long long*)ws->counters + 1, 0, sizeof(uint64_t), stream));
    GSM_CUDA(cudaMemsetAsync((unsigned long long*)ws->counters + 4, 0, sizeof(uint64_t), stream));
    int grid = lb;
    if (method == GSM_METHOD_BWA) {
        if ((st = resident_grid(k_select<GSM_METHOD_BWA>, SELECT_THREADS, 0, lb, &grid))) return st;
        // reads whose picks the sweep made need no pass over their lists; the others queue up (4 read numbers per 16-byte
        // slot of the record pool's last eighth) for the one-thread-per-read kernel
        const uint64_t reserve = ws->rec_cap / 8;
        if (reserve * 4 >= rd->n_reads) {
            se.rec_cap = ws->rec_cap - reserve;
            uint32_t* queue = (uint32_t*)((uint4*)ws->rec_tmp + se.rec_cap);
            GSM_CUDA(cudaMemsetAsync((unsigned long long*)ws->counters + 4, 0, 3 * sizeof(uint64_t), stream));    // queue length, mode, records
            k_select_bwa_picked<<<(unsigned)((rd->n_reads + 255) / 256), 256, 0, stream>>>(se, queue);
            k_select<GSM_METHOD_BWA><<<grid, SELECT_THREADS, 0, stream>>>(se, queue);
            k_select_bwa_finish<<<1, 1, 0, stream>>>((unsigned long long*)ws->counters);
            GSM_CUDA(cudaMemsetAsync((unsigned long long*)ws->counters + 5, 1, 1, stream));                        // mode: picked reads' records come from their lists
        } else {
            GSM_CUDA(cudaMemsetAsync((unsigned long long*)ws->counters + 5, 0, sizeof(uint64_t), stream));
            k_select<GSM_METHOD_BWA><<<grid, SELECT_THREADS, 0, stream>>>(se, nullptr);
        }
    } else {
        GSM_CUDA(cudaMemsetAsync((unsigned long long*)ws->counters + 5, 0, sizeof(uint64_t), stream));
        const bool arith = rm.n_none != 0u && se.seed_K != 0u && se.seed_K <= K;       // lookups from the seed table: no probes
        // RMI-SMEM pre-filter (with the bounds table and the model's hazard set): reads without a hazard window emit the
        // BWA-SMEM records with min_len 1 (select_logic.cuh, "hazard codes of a model"), so they go through k_select<BWA>;
        // the frame machine then runs only the reads left at READ_PENDING.  The read queue borrows the deferred-search queue's
        // place (4 read numbers per 16-byte slot) and is consumed before k_select_seeded starts filling that one.
        if (method == GSM_METHOD_RMI && g_rmi_prefilter != 0 && se.rmi_bounds && rmi->hazard_slots && rmi->hazard_n_slots >= 2u &&
            (rmi->hazard_n_slots & (rmi->hazard_n_slots - 1u)) == 0u && K <= 15u && se.fix_cap * 4ull >= rd->n_reads) {
            se.hz_slots = rmi->hazard_slots; se.hz_mask = rmi->hazard_n_slots - 1u;
            SelectArgs sb_ = se;                       // the BWA-SMEM selection of the queued reads: min_len 1, K flags reads shorter than K
            sb_.min_len = 1u;
            int grid_b = lb;
            if ((st = resident_grid(k_select<GSM_METHOD_BWA>, SELECT_THREADS, 0, lb, &grid_b))) return st;
            uint32_t* queue = (uint32_t*)se.fix;
            k_rmi_prefilter<<<(unsigned)((rd->n_reads + 255) / 256), 256, 0, stream>>>(se, queue);
            k_select<GSM_METHOD_BWA><<<grid_b, SELECT_THREADS, 0, stream>>>(sb_, queue);
            GSM_CUDA(cudaGetLastError());
            GSM_CUDA(cudaMemsetAsync((unsigned long long*)ws->counters + 4, 0, sizeof(uint64_t), stream));       // the queue is consumed
            se.only_pending = 1u;
        }
        if (method == GSM_METHOD_LUT) st = launch_seeded<GSM_METHOD_LUT, 0>(se, lb, stream);
        else if (se.rmi_bounds) st = launch_seeded<GSM_METHOD_RMI, 2>(se, lb, stream);
        else if (arith) st = launch_seeded<GSM_METHOD_RMI, 1>(se, lb, stream);
        else st = launch_seeded<GSM_METHOD_RMI, 0>(se, lb, stream);
        if (st) return st;
        int dev = 0, sms = 148;
        GSM_CUDA(cudaGetDevice(&dev));
        GSM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        if (method == GSM_METHOD_LUT) k_resolve_lazy<GSM_METHOD_LUT><<<sms * 8, SELECT_THREADS, 0, stream>>>(se);
        else k_resolve_lazy<GSM_METHOD_RMI><<<sms * 8, SELECT_THREADS, 0, stream>>>(se);
    }
    GSM_CUDA(cudaGetLastError());
    const uint64_t n_tiles = (rd->n_reads + SCAN_TILE - 1) / SCAN_TILE;
    unsigned long long* tiles = (unsigned long long*)ws->scan_tmp;
    k_scan_tiles<<<(unsigned)n_tiles, SCAN_THREADS, 0, stream>>>(ws->rec_cnt, rd->n_reads, (unsigned long long*)ws->rec_off, tiles);
    k_scan_top<<<1, SCAN_THREADS, 0, stream>>>(tiles, n_tiles, tiles + n_tiles);
    k_scan_add<<<(unsigned)n_tiles, SCAN_THREADS, 0, stream>>>((unsigned long long*)ws->rec_off, rd->n_reads, tiles, tiles + n_tiles);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

int gsm_smem_batch(int method, const gsm_dev_index* ix, const gsm_dev_reads* rd, uint32_t min_len, uint32_t K, const uint32_t* lut,
                   const gsm_dev_rmi* rmi, gsm_workspace* ws, void* stream) {
    int st = gsm_smem_sweep(ix, rd, ws, stream);
    if (st) return st;
    return gsm_smem_select(method, ix, rd, min_len, K, lut, rmi, ws, stream);
}

int gsm_smem_collect(const gsm_dev_reads* rd, gsm_workspace* ws, gsm_record* out, uint64_t out_cap, void* stream) {
    if (!rd || !ws || (!out && out_cap)) return fail(GSM_E_INVALID, "null");
    int st = device_ready();
    if (st) return st;
    if (rd->n_reads == 0) return GSM_OK;
    const uint64_t threads = rd->n_reads * 4;
    k_gather_records<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (const uint4*)ws->rec_tmp, ws->rec_tmp_off, ws->rec_cnt, (const unsigned long long*)ws->rec_off, rd->n_reads, (uint4*)out, out_cap,
        (unsigned long long*)ws->counters, nullptr, 0u, nullptr,
        (const uint4*)ws->mem_pool, ws->mem_off, ws->mem_cnt, rd->read_id_base);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

int gsm_smem_collect_gathered(const gsm_dev_reads* rd, gsm_workspace* ws, gsm_record* out, uint64_t out_cap, const uint64_t* counts_dev,
                              uint32_t rank, const uint64_t* base_dev, void* stream) {
    if (!rd || !ws || (!out && out_cap)) return fail(GSM_E_INVALID, "null");
    int st = device_ready();
    if (st) return st;
    if (rd->n_reads == 0) return GSM_OK;
    const uint64_t threads = rd->n_reads * 4;
    k_gather_records<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (const uint4*)ws->rec_tmp, ws->rec_tmp_off, ws->rec_cnt, (const unsigned long long*)ws->rec_off, rd->n_reads, (uint4*)out, out_cap,
        (unsigned long long*)ws->counters, (const unsigned long long*)counts_dev, rank, (const unsigned long long*)base_dev,
        (const uint4*)ws->mem_pool, ws->mem_off, ws->mem_cnt, rd->read_id_base);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

int gsm_gather_advance(uint64_t* base_dev, const uint64_t* counts_dev, uint32_t world, void* stream) {
    if (!base_dev || !counts_dev || world == 0) return fail(GSM_E_INVALID, "gsm_gather_advance: null");
    int st = device_ready();
    if (st) return st;
    k_gather_advance<<<1, 1, 0, (cudaStream_t)stream>>>((unsigned long long*)base_dev, (const unsigned long long*)counts_dev, world);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

int gsm_gather_probe2(const void* buf, uint64_t bytes, uint64_t n_fetch, uint32_t fetch_bytes, uint32_t in_flight, uint64_t* sink, uint64_t* n_done,
                      void* stream) {
    const uint32_t pf = fetch_bytes == 66 ? 1u : 0u;      // 66: 64-byte fetches by lane pairs (one request per bucket, half as many buckets per instruction)
    if (pf) fetch_bytes = 64;
    if (!buf || !sink || bytes < 64 || (fetch_bytes != 16 && fetch_bytes != 32 && fetch_bytes != 64) || (in_flight != 1 && in_flight != 4 && in_flight != 8))
        return fail(GSM_E_INVALID, "gsm_gather_probe2: fetch_bytes in {16, 32, 64, 66}, in_flight in {1, 4, 8}");
    int st = device_ready();
    if (st) return st;
    int dev = 0, sms = 0;
    GSM_CUDA(cudaGetDevice(&dev));
    GSM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    uint64_t units = bytes / fetch_bytes, pow2 = 1;
    while (pow2 * 2 <= units) pow2 *= 2;                  // the largest power of two of units: index by mask
    const uint64_t threads = (uint64_t)sms * 16 * 128;
    uint32_t iters = (uint32_t)((n_fetch + threads * in_flight - 1) / (threads * in_flight));
    if (iters == 0) iters = 1;
    cudaStream_t s = (cudaStream_t)stream;
    const uint4* b = (const uint4*)buf;
    unsigned long long* sk = (unsigned long long*)sink;
    const unsigned grid = (unsigned)(sms * 16);
#define GSM_PROBE2(B, U) k_gather_probe2<B, U><<<grid, 128, 0, s>>>(b, pow2 - 1, iters, sk)
    if (fetch_bytes == 16) { if (in_flight == 1) GSM_PROBE2(16, 1); else if (in_flight == 4) GSM_PROBE2(16, 4); else GSM_PROBE2(16, 8); }
    else if (fetch_bytes == 32) { if (in_flight == 1) GSM_PROBE2(32, 1); else if (in_flight == 4) GSM_PROBE2(32, 4); else GSM_PROBE2(32, 8); }
    else if (pf == 1) k_gather_probe2<64, 4, 1><<<grid, 128, 0, s>>>(b, pow2 - 1, iters * in_flight / 4 + 1, sk);
    else { if (in_flight == 1) GSM_PROBE2(64, 1); else if (in_flight == 4) GSM_PROBE2(64, 4); else GSM_PROBE2(64, 8); }
#undef GSM_PROBE2
    GSM_CUDA(cudaGetLastError());
    if (n_done) *n_done = pf ? threads / 2 * 4ull * (iters * in_flight / 4 + 1) : threads * in_flight * iters;
    return GSM_OK;
}

int gsm_gather_probe(const void* buf, uint64_t bytes, uint64_t n_fetch, uint32_t dependent, uint64_t* sink, uint64_t* n_done, void* stream) {
    if (!buf || !sink || bytes < 64) return fail(GSM_E_INVALID, "null");
    int st = device_ready();
    if (st) return st;
    int dev = 0, sms = 0;
    GSM_CUDA(cudaGetDevice(&dev));
    GSM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const uint64_t quads = (uint64_t)sms * 16 * 64;      // 16 blocks x 128 threads per SM, one chain per lane pair
    uint32_t iters = (uint32_t)((n_fetch + quads - 1) / quads);
    if (iters == 0) iters = 1;
    k_gather_probe<<<sms * 16, 128, 0, (cudaStream_t)stream>>>((const uint4*)buf, bytes / 64, iters, dependent, (unsigned long long*)sink);
    GSM_CUDA(cudaGetLastError());
    if (n_done) *n_done = quads * iters;
    return GSM_OK;
}

}  // extern "C"
