// sm_100a kernels of the seed chaining: located hits -> BWA-MEM's co-linear chains, per slot
// (gsm_chain_seeds / gsm_chains_collect, include/genie_smem.h; per-seed rule in chain_logic.cuh).
//
//   * k_chain_slots: one lane per slot.  The lane walks its slot's records and their hits in order and keeps the slot's
//     ordered chain table in shared memory, CHAIN_CAP chains of 15 words each, lane-interleaved (no bank conflicts, no
//     synchronisation: lanes share nothing).  A slot that needs more chains is appended to an overflow list and stopped.
//   * k_chain_slots_global: the overflow list, one lane per slot, the same per-slot code with the table in global scratch
//     indexed by the slot's first hit.  A slot never has more chains than hits, so that region always has room.
//   * Either way the finished slot writes its chains in output order to the chain scratch (again at its first hit), its
//     count, and remaps its hits' creation-order ids to output order with one more pass over its hits.
//   * The counts are scanned by the record scan of kernels.cu; k_chain_write copies each slot's chains to the caller's
//     buffer at chain_off[slot].
// Every slot is chained by exactly one lane from the same inputs, so the output does not depend on the grid or on the
// order in which the overflow list was filled.
#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "../../include/genie_smem.h"
#include "chain_logic.cuh"
#include "hits_logic.cuh"
#include "host_common.hpp"

namespace gsm {

#define GSM_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess)                                                                 \
            return fail(GSM_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));       \
    } while (0)

namespace {

constexpr int CHAIN_THREADS = 64;
constexpr uint32_t CHAIN_CAP = 8;                                  // chains per slot on the fast path
constexpr int CHAIN_FIELDS = 3 + CHAIN_STATE_WORDS;                // sorted {contig, pos, id} + the state of chain `id`
constexpr int WRITE_THREADS = 256;

struct ChainArgs {
    const uint4* recs;
    const unsigned long long* rec_off;
    unsigned long long n_slots;
    const uint4* hits;
    const unsigned long long* hit_off;
    uint32_t w, max_gap;
    uint32_t* hit_chain;
    uint32_t* chain_cnt;
    uint4* chains;                   // scratch: chain k of a slot at [2 (first hit + k), +2)
    uint32_t* state;                 // slow path: CHAIN_STATE_WORDS per chain id, at the slot's first hit
    uint32_t* order;                 // slow path: ids in (contig, pos) order, at the slot's first hit
    uint32_t* overflow;              // slots the fast path could not hold
    unsigned long long* n_overflow;  // slots on the list (the slow path pops them)
};

// Workspace layout (all offsets 256-byte aligned)
struct ChainLayout {
    uint64_t chains, state, order, overflow, counter, scan, total;
};

uint64_t up256(uint64_t x) { return (x + 255u) & ~255ull; }

ChainLayout chain_layout(uint64_t n_slots, uint64_t n_hits) {
    ChainLayout l;
    l.chains = 0;
    l.state = l.chains + up256(n_hits * 32u);
    l.order = l.state + up256(n_hits * 4u * CHAIN_STATE_WORDS);
    l.overflow = l.order + up256(n_hits * 4u);
    l.counter = l.overflow + up256(n_slots * 4u);
    l.scan = l.counter + 256u;
    l.total = l.scan + up256(scan_tmp_bytes(n_slots));
    return l;
}

// The fast path's table: word f of sorted entry / chain k of this lane at base[(f * CHAIN_CAP + k) * CHAIN_THREADS + lane]
struct SmemTable {
    uint32_t* base;
    uint32_t n;
    __device__ uint32_t& at(int f, uint32_t k) const { return base[(f * CHAIN_CAP + k) * CHAIN_THREADS]; }
    __device__ uint64_t key(uint32_t i) const { return chain_key(at(0, i), at(1, i)); }
    __device__ uint32_t id(uint32_t i) const { return at(2, i); }
    __device__ ChainState load(uint32_t id) const {
        return chain_load([this, id](int f) { return at(3 + f, id); });
    }
    __device__ void store(uint32_t id, const ChainState& c) const {
        chain_store(c, [this, id](int f, uint32_t v) { at(3 + f, id) = v; });
    }
    __device__ void insert(uint32_t i, const ChainState& c) {
        for (uint32_t k = n; k > i; --k) {
            at(0, k) = at(0, k - 1u);
            at(1, k) = at(1, k - 1u);
            at(2, k) = at(2, k - 1u);
        }
        at(0, i) = c.contig;
        at(1, i) = c.pos;
        at(2, i) = n;
        store(n, c);
        ++n;
    }
    // after the output: the rank of chain `id` replaces its first state word
    __device__ void set_rank(uint32_t id, uint32_t k) const { at(3, id) = k; }
    __device__ uint32_t rank(uint32_t id) const { return at(3, id); }
};

// The slow path's table in global scratch: state[id * CHAIN_STATE_WORDS ...], order[i] = id at sorted position i
struct GlobalTable {
    uint32_t* state;
    uint32_t* order;
    uint32_t n;
    __device__ uint64_t key(uint32_t i) const {
        const uint32_t* c = state + (uint64_t)order[i] * CHAIN_STATE_WORDS;
        return chain_key(c[0], c[1]);
    }
    __device__ uint32_t id(uint32_t i) const { return order[i]; }
    __device__ ChainState load(uint32_t id) const {
        const uint32_t* p = state + (uint64_t)id * CHAIN_STATE_WORDS;
        return chain_load([p](int f) { return p[f]; });
    }
    __device__ void store(uint32_t id, const ChainState& c) const {
        uint32_t* p = state + (uint64_t)id * CHAIN_STATE_WORDS;
        chain_store(c, [p](int f, uint32_t v) { p[f] = v; });
    }
    __device__ void insert(uint32_t i, const ChainState& c) {
        for (uint32_t k = n; k > i; --k) order[k] = order[k - 1u];
        order[i] = n;
        store(n, c);
        ++n;
    }
    __device__ void set_rank(uint32_t id, uint32_t k) const { state[(uint64_t)id * CHAIN_STATE_WORDS] = k; }
    __device__ uint32_t rank(uint32_t id) const { return state[(uint64_t)id * CHAIN_STATE_WORDS]; }
};

// mem_chain over slot s: every hit gets its creation-order id.  false: the table reached cap chains (slot unfinished).
template <typename Tab>
__device__ __forceinline__ bool chain_slot(const ChainArgs& a, uint64_t s, Tab& t, uint32_t cap) {
    const uint64_t r0 = a.rec_off[s], r1 = a.rec_off[s + 1];
    uint64_t h = r0 < r1 ? a.hit_off[r0] : 0u;
    for (uint64_t r = r0; r < r1; ++r) {
        const uint4 rec = __ldg(a.recs + r);
        const uint64_t h1 = a.hit_off[r + 1];
        const uint32_t qbeg = rec.y & 0xFFFFu, len = hit_len(rec.y);
        for (; h < h1; ++h) {
            const uint4 hit = __ldg(a.hits + h);
            uint32_t id = CHAIN_NONE;
            if (!(hit.w & HIT_SPANS)) {          // BWA skips a seed that bridges two sequences (rid < 0)
                ChainSeed sd;
                sd.qbeg = qbeg;
                sd.len = len;
                sd.rbeg = hit.z;
                sd.contig = hit.y;
                id = chain_step(t, sd, a.w, a.max_gap, cap);
                if (id == CHAIN_FULL) return false;
            }
            a.hit_chain[h] = id;
        }
    }
    return true;
}

// The finished slot: chains in output order to the scratch at its first hit, its count, ids remapped to output order.
template <typename Tab>
__device__ __forceinline__ void chain_finish(const ChainArgs& a, uint64_t s, Tab& t) {
    const uint64_t r0 = a.rec_off[s], r1 = a.rec_off[s + 1];
    a.chain_cnt[s] = t.n;
    if (t.n == 0u) return;
    const uint64_t h0 = a.hit_off[r0], h1 = a.hit_off[r1];
    bool same = true;
    for (uint32_t k = 0; k < t.n; ++k) {
        const uint32_t id = t.id(k);
        uint32_t o[8];
        chain_output(t.load(id), (uint32_t)s, o);
        a.chains[2 * (h0 + k)] = make_uint4(o[0], o[1], o[2], o[3]);
        a.chains[2 * (h0 + k) + 1] = make_uint4(o[4], o[5], o[6], o[7]);
        same &= id == k;
    }
    if (same) return;                            // created in output order: the ids are final
    for (uint32_t k = 0; k < t.n; ++k) t.set_rank(t.id(k), k);
    for (uint64_t h = h0; h < h1; ++h) {
        const uint32_t v = a.hit_chain[h];
        if (v != CHAIN_NONE) a.hit_chain[h] = (v & CHAIN_CONTAINED) | t.rank(v & ~CHAIN_CONTAINED);
    }
}

__global__ void __launch_bounds__(CHAIN_THREADS) k_chain_slots(const ChainArgs a) {
    __shared__ uint32_t s_tab[CHAIN_FIELDS * CHAIN_CAP * CHAIN_THREADS];
    const uint64_t s = (uint64_t)blockIdx.x * CHAIN_THREADS + threadIdx.x;
    if (s >= a.n_slots) return;
    SmemTable t{s_tab + threadIdx.x, 0u};
    if (chain_slot(a, s, t, CHAIN_CAP)) chain_finish(a, s, t);
    else a.overflow[atomicAdd(a.n_overflow, 1ull)] = (uint32_t)s;
}

__global__ void __launch_bounds__(CHAIN_THREADS) k_chain_slots_global(const ChainArgs a) {
    for (;;) {                                   // lanes pop the list: slots on this path differ widely in size
        const long long i = (long long)atomicAdd(a.n_overflow, ~0ull);
        if (i <= 0) break;
        const uint64_t s = a.overflow[i - 1];
        const uint64_t r0 = a.rec_off[s];
        const uint64_t h0 = r0 < a.rec_off[s + 1] ? a.hit_off[r0] : 0u;
        GlobalTable t{a.state + h0 * CHAIN_STATE_WORDS, a.order + h0, 0u};
        chain_slot(a, s, t, 0xFFFFFFFFu);        // never full: a slot has at most as many chains as hits
        chain_finish(a, s, t);
    }
}

__global__ void __launch_bounds__(WRITE_THREADS) k_chain_write(const unsigned long long* rec_off, unsigned long long n_slots,
                                                               const unsigned long long* hit_off, const unsigned long long* chain_off,
                                                               const uint4* chains, uint4* out, unsigned long long out_cap,
                                                               unsigned long long* status) {
    const uint64_t s = (uint64_t)blockIdx.x * WRITE_THREADS + threadIdx.x;
    if (s == 0 && chain_off[n_slots] > out_cap) atomicOr(status, 1ull);
    if (s >= n_slots) return;
    const unsigned long long o = chain_off[s], n = chain_off[s + 1] - o;
    if (n == 0) return;
    const uint64_t h0 = hit_off[rec_off[s]];
    for (uint64_t k = 0; k < n && o + k < out_cap; ++k) {
        out[2 * (o + k)] = chains[2 * (h0 + k)];
        out[2 * (o + k) + 1] = chains[2 * (h0 + k) + 1];
    }
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

int gsm_chains_workspace_info(uint64_t n_slots, uint64_t n_hits, uint64_t* bytes) {
    if (!bytes) return fail(GSM_E_INVALID, "gsm_chains_workspace_info: null");
    *bytes = chain_layout(n_slots, n_hits).total;
    return GSM_OK;
}

int gsm_chain_seeds(const gsm_record* recs, const uint64_t* rec_off, uint64_t n_slots, const gsm_hit* hits, const uint64_t* hit_off,
                    uint64_t n_hits, uint32_t w, uint32_t max_gap, uint32_t* hit_chain, uint32_t* chain_cnt, uint64_t* chain_off,
                    void* workspace, uint64_t workspace_bytes, void* stream) {
    if (!chain_off || (n_slots && (!recs || !rec_off || !hit_off || !chain_cnt || !workspace)) || (n_hits && (!hits || !hit_chain)))
        return fail(GSM_E_INVALID, "gsm_chain_seeds: null");
    if (n_slots >= 0xFFFFFFFFull) return fail(GSM_E_INVALID, "gsm_chain_seeds: slot indices must fit in 32 bits");
    const ChainLayout l = chain_layout(n_slots, n_hits);
    if (n_slots && workspace_bytes < l.total) return fail(GSM_E_CAPACITY, "gsm_chain_seeds: workspace too small (see gsm_chains_workspace_info)");
    int st = device_ready();
    if (st) return st;
    cudaStream_t s = (cudaStream_t)stream;
    if (n_slots) {
        char* ws = (char*)workspace;
        ChainArgs a;
        a.recs = (const uint4*)recs;
        a.rec_off = (const unsigned long long*)rec_off;
        a.n_slots = n_slots;
        a.hits = (const uint4*)hits;
        a.hit_off = (const unsigned long long*)hit_off;
        a.w = w;
        a.max_gap = max_gap;
        a.hit_chain = hit_chain;
        a.chain_cnt = chain_cnt;
        a.chains = (uint4*)(ws + l.chains);
        a.state = (uint32_t*)(ws + l.state);
        a.order = (uint32_t*)(ws + l.order);
        a.overflow = (uint32_t*)(ws + l.overflow);
        a.n_overflow = (unsigned long long*)(ws + l.counter);
        GSM_CUDA(cudaMemsetAsync(a.n_overflow, 0, 8, s));
        k_chain_slots<<<(unsigned)((n_slots + CHAIN_THREADS - 1) / CHAIN_THREADS), CHAIN_THREADS, 0, s>>>(a);
        int dev = 0, sms = 0;
        GSM_CUDA(cudaGetDevice(&dev));
        GSM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        // the overflow count is only known on the device: a fixed grid strides over the list
        const uint64_t by_slots = (n_slots + CHAIN_THREADS - 1) / CHAIN_THREADS, most = (uint64_t)sms * 8u;
        k_chain_slots_global<<<(unsigned)(by_slots < most ? by_slots : most), CHAIN_THREADS, 0, s>>>(a);
        GSM_CUDA(cudaGetLastError());
    }
    return scan_counts(chain_cnt, n_slots, chain_off, (char*)workspace + l.scan, n_slots ? workspace_bytes - l.scan : 0, stream);
}

int gsm_chains_collect(const uint64_t* rec_off, uint64_t n_slots, const uint64_t* hit_off, uint64_t n_hits, const uint64_t* chain_off,
                       const void* workspace, uint64_t workspace_bytes, gsm_chain* out, uint64_t out_cap, uint64_t* status8, void* stream) {
    if (!chain_off || !status8 || (!out && out_cap) || (n_slots && (!rec_off || !hit_off || !workspace)))
        return fail(GSM_E_INVALID, "gsm_chains_collect: null");
    const ChainLayout l = chain_layout(n_slots, n_hits);
    if (n_slots && workspace_bytes < l.total) return fail(GSM_E_CAPACITY, "gsm_chains_collect: workspace too small (see gsm_chains_workspace_info)");
    int st = device_ready();
    if (st) return st;
    if (n_slots == 0) return GSM_OK;
    cudaStream_t s = (cudaStream_t)stream;
    k_chain_write<<<(unsigned)((n_slots + WRITE_THREADS - 1) / WRITE_THREADS), WRITE_THREADS, 0, s>>>(
        (const unsigned long long*)rec_off, n_slots, (const unsigned long long*)hit_off, (const unsigned long long*)chain_off,
        (const uint4*)((const char*)workspace + l.chains), (uint4*)out, out_cap, (unsigned long long*)status8);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

}  // extern "C"
