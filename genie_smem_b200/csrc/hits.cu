// sm_100a kernels of the hit expansion: SMEM records -> capped occurrence positions in per-sequence coordinates
// (gsm_hits_count / gsm_hits_locate, include/genie_smem.h; per-hit arithmetic in hits_logic.cuh).
//
//   * k_hits_count: one thread per record, one 16-byte load; the counts are scanned by the record scan of kernels.cu.
//   * k_hits_locate: load-balanced over HITS (a record has 0 .. max_occ of them).  A block takes a tile of HIT_TILE
//     consecutive hits, finds the tile's first record with one warp-wide 32-way search of hit_off, stages the tile's
//     records and their hit offsets in shared memory, and every thread finds the record of each of its hits with a short
//     search there, starting where its previous hit's search ended (its hits ascend).  Consecutive lanes take consecutive
//     hits, so with step == 1 a warp reads consecutive suffix-array words (full SA) and writes 512 contiguous bytes.
//     Positions: one suffix-array load (full SA) or the LF walk of k_locate_sampled (sampled SA).  Sequence: a binary
//     search of the start table, from shared memory when it has at most HIT_SMEM_CONTIGS entries AND costs the kernel no
//     resident block, else through L1 / L2.  Measured on B200 (1 Gbp, 221 M hits, profiles/hits_bench_1gbp.json): a table
//     that lowers the occupancy of the latency-bound LF walk loses more than the shared-memory search gains.
#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "../../include/genie_smem.h"
#include "host_common.hpp"
#include "hits_logic.cuh"

namespace gsm {

#define GSM_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess)                                                                 \
            return fail(GSM_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));       \
    } while (0)

namespace {

constexpr int HIT_THREADS = 128;
constexpr int HIT_ITEMS = 4;
constexpr int HIT_TILE = HIT_THREADS * HIT_ITEMS;      // hits per tile
constexpr int HIT_MIN_BLOCKS = 8;                       // register budget of the full-SA variant: 64 per thread
constexpr int HIT_MIN_BLOCKS_LF = 16;                   // LF-walk variant: 32 registers, 2,048 threads per SM (latency-bound like k_locate_sampled)
constexpr uint32_t HIT_SMEM_CONTIGS = 8192;             // start tables up to this many entries (32 KB) sit in shared memory
constexpr int COUNT_THREADS = 256;

struct HitArgs {
    const uint4* fwd;
    const uint32_t* sa;           // full suffix array (1-based values), or NULL: LF walk to the sampled rows
    const uint32_t* ssa;
    uint32_t S;
    uint32_t C[4];
    uint32_t prim_f;
    uint32_t n_bases;
    const uint32_t* start;        // sequence table (n_entries = sequences + 1), NULL = one sequence
    uint32_t n_entries;
    uint32_t max_occ, min_len;
    const uint4* recs;
    const unsigned long long* hit_off;
    unsigned long long rec_begin, rec_end;
    uint4* out;
    unsigned long long out_cap;
    unsigned long long* status;
};

// one 32-byte half of a rank bucket: a single 256-bit read-only load (as in sweep_device.cuh)
__device__ __forceinline__ Half ldg_half(const uint4* halves_base, size_t half_index) {
    Half h;
    asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(h.c0), "=r"(h.c1), "=r"(h.l0), "=r"(h.l1), "=r"(h.l2), "=r"(h.h0), "=r"(h.h1), "=r"(h.h2)
                 : "l"(halves_base + half_index * 2));
    return h;
}

__global__ void __launch_bounds__(COUNT_THREADS) k_hits_count(const uint4* recs, uint64_t n, uint32_t max_occ, uint32_t min_len, uint32_t* cnt) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint4 r = __ldg(recs + i);
    cnt[i] = hit_count(hit_rows(r.z, r.w), hit_len(r.y), max_occ, min_len);
}

// last r in [lo, hi) with hit_off[r] <= h, given hit_off[lo] <= h (one thread)
__device__ __forceinline__ uint64_t last_le(const unsigned long long* off, uint64_t lo, uint64_t hi, unsigned long long h) {
    while (hi - lo > 1) {
        const uint64_t mid = lo + (hi - lo) / 2;
        if (off[mid] <= h) lo = mid;
        else hi = mid;
    }
    return lo;
}

template <bool FULL_SA, bool SMEM_TAB>
__global__ void __launch_bounds__(HIT_THREADS, FULL_SA ? HIT_MIN_BLOCKS : HIT_MIN_BLOCKS_LF) k_hits_locate(const HitArgs a) {
    __shared__ uint4 s_rec[HIT_TILE];
    __shared__ uint32_t s_off[HIT_TILE + 1];     // hit_off[r0 + j] - first hit of the tile, clamped to [0, HIT_TILE + 1]
    __shared__ unsigned long long s_r0, s_r0n;   // first record of this tile / of the next one (s_next: found in the staging)
    __shared__ uint32_t s_k0, s_k0n, s_next;     // ordinal of that tile's first hit in its first record
    extern __shared__ uint32_t s_start[];        // SMEM_TAB: the start table
    if (SMEM_TAB)
        for (uint32_t i = threadIdx.x; i < a.n_entries; i += blockDim.x) s_start[i] = a.start ? __ldg(a.start + i) : (i ? a.n_bases : 0u);
    const unsigned long long base = a.hit_off[a.rec_begin], total = a.hit_off[a.rec_end] - base;
    if (blockIdx.x == 0 && threadIdx.x == 0 && total > a.out_cap) atomicOr(a.status, 1ull);
    const unsigned long long n_hits = total < a.out_cap ? total : a.out_cap;
    auto load_b = [&a](uint64_t i) { return ldg_half(a.fwd, i); };
    // each block takes a contiguous run of tiles: only its first tile searches hit_off, the next tile's first record is
    // read off the staged offsets of the current one
    const unsigned long long n_tiles = (n_hits + HIT_TILE - 1) / HIT_TILE, per = (n_tiles + gridDim.x - 1) / gridDim.x;
    const unsigned long long t_end = (blockIdx.x + 1ull) * per < n_tiles ? (blockIdx.x + 1ull) * per : n_tiles;
    uint64_t r0 = 0;
    uint32_t k0 = 0;
    bool known = false;
    for (unsigned long long t = blockIdx.x * per; t < t_end; ++t) {
        const unsigned long long t0 = t * HIT_TILE, tb = base + t0;
        if (!known) {                            // block-uniform
            if (threadIdx.x < 32) {              // warp 0: 32-way search for the last record with hit_off <= tb
                const uint32_t lane = threadIdx.x;
                uint64_t lo = a.rec_begin, hi = a.rec_end;
                while (hi - lo > 1) {
                    const uint64_t step = (hi - lo + 31) / 32, pr = lo + lane * step;
                    const bool le = pr < hi && a.hit_off[pr] <= tb;
                    const uint32_t k = 31u - __clz(__ballot_sync(0xFFFFFFFFu, le));     // lane 0 probes lo: always true
                    lo += k * step;
                    hi = hi < lo + step ? hi : lo + step;
                }
                if (lane == 0) { s_r0 = lo; s_k0 = (uint32_t)(tb - a.hit_off[lo]); }
            }
            __syncthreads();
            r0 = s_r0;
            k0 = s_k0;
        }
        const uint32_t n_stage = a.rec_end - r0 < (uint64_t)HIT_TILE ? (uint32_t)(a.rec_end - r0) : (uint32_t)HIT_TILE;
        for (uint32_t j = threadIdx.x; j <= n_stage; j += HIT_THREADS) {
            if (j < n_stage) s_rec[j] = __ldg(a.recs + r0 + j);
            const unsigned long long o = a.hit_off[r0 + j];
            s_off[j] = o <= tb ? 0u : (o - tb > (unsigned long long)HIT_TILE ? (uint32_t)HIT_TILE + 1u : (uint32_t)(o - tb));
        }
        __syncthreads();
        if (threadIdx.x == 0) {                  // the record holding hit tb + HIT_TILE, if it is staged
            s_next = s_off[n_stage] > (uint32_t)HIT_TILE;
            if (s_next) {
                uint32_t lo = 0, hi = n_stage;
                while (hi - lo > 1) {
                    const uint32_t mid = (lo + hi) >> 1;
                    if (s_off[mid] <= (uint32_t)HIT_TILE) lo = mid;
                    else hi = mid;
                }
                s_r0n = r0 + lo;
                s_k0n = lo ? (uint32_t)HIT_TILE - s_off[lo] : k0 + (uint32_t)HIT_TILE;
            }
        }
        uint32_t jlo = 0;
#pragma unroll 1
        for (int it = 0; it < HIT_ITEMS; ++it) {
            const uint32_t h = threadIdx.x + it * HIT_THREADS;
            if (t0 + h >= n_hits) break;
            uint64_t r;
            uint4 rec;
            uint32_t k;
            if (s_off[n_stage] > h) {            // staged: last j in [jlo, n_stage) with s_off[j] <= h
                uint32_t hi = n_stage;
                while (hi - jlo > 1) {
                    const uint32_t mid = (jlo + hi) >> 1;
                    if (s_off[mid] <= h) jlo = mid;
                    else hi = mid;
                }
                r = r0 + jlo;
                rec = s_rec[jlo];
                k = jlo ? h - s_off[jlo] : h + k0;
            } else {                             // past the staged records (a run of records without hits): through L2
                r = last_le(a.hit_off, r0 + n_stage, a.rec_end, tb + h);
                rec = __ldg(a.recs + r);
                k = (uint32_t)(tb + h - a.hit_off[r]);
            }
            const uint32_t cnt = hit_rows(rec.z, rec.w), len = hit_len(rec.y);
            uint32_t row = hit_row(rec.z, k, hit_step(cnt, a.max_occ)), pos;
            if (FULL_SA) {
                pos = __ldg(a.sa + row);
            } else {                             // k_locate_sampled's walk: LF until a sampled row or the '$' row
                uint32_t t = 0;
                for (;;) {
                    if (row == a.prim_f) { pos = 1u + t; break; }
                    if (row % a.S == 0u) { pos = __ldg(a.ssa + row / a.S) + t; break; }
                    row = lf_single(load_b, row, a.C, a.prim_f);
                    ++t;
                }
            }
            const bool sampled = hit_sampled(cnt, a.max_occ);
            U4 o;
            if (SMEM_TAB) o = make_hit([](uint32_t i) { return s_start[i]; }, a.n_entries, (uint32_t)r, pos - 1u, len, sampled);
            else o = make_hit([&a](uint32_t i) { return __ldg(a.start + i); }, a.n_entries, (uint32_t)r, pos - 1u, len, sampled);
            a.out[t0 + h] = make_uint4(o.x, o.y, o.z, o.w);
        }
        __syncthreads();
        known = s_next != 0u;
        r0 = s_r0n;
        k0 = s_k0n;
    }
}

template <bool FULL_SA, bool SMEM_TAB>
int launch_locate(const HitArgs& a, cudaStream_t stream) {
    const size_t smem = SMEM_TAB ? (size_t)a.n_entries * 4u : 0u;
    int dev = 0, sms = 0, per_sm = 0;
    GSM_CUDA(cudaGetDevice(&dev));
    GSM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    GSM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_hits_locate<FULL_SA, SMEM_TAB>, HIT_THREADS, smem));
    if (per_sm < 1) per_sm = 1;
    // a resident grid striding over tiles; it cannot need more tiles than out_cap holds
    const unsigned long long by_cap = (a.out_cap + HIT_TILE - 1) / HIT_TILE;
    const unsigned long long resident = (unsigned long long)sms * per_sm;
    const unsigned grid = (unsigned)(by_cap < 1 ? 1 : (by_cap < resident ? by_cap : resident));
    k_hits_locate<FULL_SA, SMEM_TAB><<<grid, HIT_THREADS, smem, stream>>>(a);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

// resident blocks per SM of one instantiation
template <bool FULL_SA, bool SMEM_TAB>
int blocks_per_sm(size_t smem, int* per_sm) {
    GSM_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, k_hits_locate<FULL_SA, SMEM_TAB>, HIT_THREADS, smem));
    return GSM_OK;
}

// the start table goes to shared memory when it is small enough and costs no resident block (always without a table: 8 bytes)
template <bool FULL_SA>
int launch_locate_any(const HitArgs& a, cudaStream_t stream) {
    bool smem_tab = a.start == nullptr;
    if (!smem_tab && a.n_entries <= HIT_SMEM_CONTIGS) {
        int with = 0, without = 0, st;
        if ((st = blocks_per_sm<FULL_SA, true>((size_t)a.n_entries * 4u, &with))) return st;
        if ((st = blocks_per_sm<FULL_SA, false>(0, &without))) return st;
        smem_tab = with >= without;
    }
    return smem_tab ? launch_locate<FULL_SA, true>(a, stream) : launch_locate<FULL_SA, false>(a, stream);
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

}  // namespace
}  // namespace gsm

using namespace gsm;

extern "C" {

int gsm_hits_workspace_info(uint64_t n_recs, uint64_t* bytes) {
    if (!bytes) return fail(GSM_E_INVALID, "gsm_hits_workspace_info: null");
    *bytes = scan_tmp_bytes(n_recs);
    return GSM_OK;
}

int gsm_hits_count(const gsm_record* recs, uint64_t n_recs, uint32_t max_occ, uint32_t min_len, uint32_t* counts, uint64_t* hit_off,
                   void* scan_tmp, uint64_t scan_tmp_bytes_, void* stream) {
    if (!hit_off || (n_recs && (!recs || !counts || !scan_tmp))) return fail(GSM_E_INVALID, "gsm_hits_count: null");
    if (n_recs && scan_tmp_bytes_ < scan_tmp_bytes(n_recs)) return fail(GSM_E_CAPACITY, "gsm_hits_count: scan_tmp too small (see gsm_hits_workspace_info)");
    int st = device_ready();
    if (st) return st;
    cudaStream_t s = (cudaStream_t)stream;
    if (n_recs)
        k_hits_count<<<(unsigned)((n_recs + COUNT_THREADS - 1) / COUNT_THREADS), COUNT_THREADS, 0, s>>>((const uint4*)recs, n_recs, max_occ, min_len,
                                                                                                        counts);
    GSM_CUDA(cudaGetLastError());
    return scan_counts(counts, n_recs, hit_off, scan_tmp, scan_tmp_bytes_, stream);
}

int gsm_hits_locate(const gsm_dev_index* ix, const uint32_t* ssa, uint32_t sample, const gsm_dev_contigs* contigs, const gsm_record* recs,
                    const uint64_t* hit_off, uint64_t rec_begin, uint64_t rec_end, uint32_t max_occ, uint32_t min_len, gsm_hit* out, uint64_t out_cap,
                    uint64_t* status8, void* stream) {
    if (!ix || !hit_off || !status8 || (!out && out_cap) || rec_end < rec_begin || (rec_end > rec_begin && !recs))
        return fail(GSM_E_INVALID, "gsm_hits_locate: null pointer or empty record range");
    if (!ix->sa && (!ssa || sample == 0 || !ix->fwd_buckets))
        return fail(GSM_E_INVALID, "gsm_hits_locate: neither the suffix array nor a sampled one is on the device");
    if (contigs && (!contigs->start || contigs->n == 0 || contigs->n >= 0xFFFFFFFFull))
        return fail(GSM_E_INVALID, "gsm_hits_locate: the sequence table needs n >= 1 sequences and n + 1 start entries");
    int st = device_ready();
    if (st) return st;
    if (rec_end == rec_begin) return GSM_OK;
    HitArgs a;
    a.fwd = (const uint4*)ix->fwd_buckets;
    a.sa = ix->sa;
    a.ssa = ssa;
    a.S = sample ? sample : 1u;
    for (int c = 0; c < 4; ++c) a.C[c] = ix->C[c];
    a.prim_f = ix->primary_fwd;
    a.n_bases = (uint32_t)(ix->n_rows - 1);
    a.start = contigs ? contigs->start : nullptr;
    a.n_entries = contigs ? (uint32_t)(contigs->n + 1) : 2u;
    a.max_occ = max_occ;
    a.min_len = min_len;
    a.recs = (const uint4*)recs;
    a.hit_off = (const unsigned long long*)hit_off;
    a.rec_begin = rec_begin;
    a.rec_end = rec_end;
    a.out = (uint4*)out;
    a.out_cap = out_cap;
    a.status = (unsigned long long*)status8;
    cudaStream_t s = (cudaStream_t)stream;
    return ix->sa ? launch_locate_any<true>(a, s) : launch_locate_any<false>(a, s);
}

}  // extern "C"
