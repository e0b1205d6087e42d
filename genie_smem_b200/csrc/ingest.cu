// Read ingest on the device (SURVEY 8f N2): ASCII (or code) reads -> the 2-bit packed, 16-byte aligned batch
// layout of include/genie_smem.h.  The reference takes one Python string per call (ExactMatch.load_query,
// SMEM/ExactMatch.py:104-108; SMEM.get_SMEMS(query, ...), SMEM/SMEM.py:456); a pipeline hands over raw read
// bytes, which cross PCIe once (1 byte/base) and are packed here at HBM speed instead of by a host loop.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <string>

#include "../../include/genie_smem.h"
#include "host_common.hpp"
#include "strand_logic.cuh"

namespace gsm {

#define GSM_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e__ = (call);                                                               \
        if (e__ != cudaSuccess)                                                                 \
            return fail(GSM_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));       \
    } while (0)

namespace {

// One warp per read, one lane per 16-base output word (grid-stride over reads).  The pad words of a read's last
// 16-byte chunk are zeroed.  A non-ACGT byte records the smallest offending read index in *bad.
__global__ void __launch_bounds__(256) k_pack_reads(const uint8_t* bases, const unsigned long long* base_off, uint32_t fixed_len,
                                                    const uint32_t* chunk_off, uint64_t n_reads, int ascii, uint32_t* packed,
                                                    uint32_t* len_out, unsigned long long* bad) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warp0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t r = warp0; r < n_reads; r += n_warps) {
        uint64_t b0;
        uint32_t L;
        if (base_off) {
            b0 = base_off[r];
            L = (uint32_t)(base_off[r + 1] - b0);
        } else {
            b0 = r * (uint64_t)fixed_len;
            L = fixed_len;
        }
        uint32_t* dst = packed + (uint64_t)chunk_off[r] * 4u;
        const uint32_t n_words = ((L + 63u) / 64u) * 4u;
        if (len_out && lane == 0) len_out[r] = L;
        for (uint32_t w = lane; w < n_words; w += 32u) {
            uint32_t v = 0;
            const uint32_t t0 = w * 16u;
            for (uint32_t t = 0; t < 16u && t0 + t < L; ++t) {
                uint32_t c = bases[b0 + t0 + t];
                if (ascii) c = c == 'A' ? 0u : c == 'C' ? 1u : c == 'G' ? 2u : c == 'T' ? 3u : 4u;
                if (c > 3u) {
                    atomicMin(bad, (unsigned long long)r);
                    c = 0;
                }
                v |= c << (30u - 2u * t);
            }
            dst[w] = v;
        }
    }
}

// Fixed-length reads (the FASTQ case): a block takes PACK_R consecutive reads = one contiguous byte range, stages it in
// shared memory with coalesced 16-byte loads, and every thread packs whole 16-base words from there -- all lanes busy,
// global traffic at full sector efficiency (the per-read kernel above keeps 12 of 32 lanes busy on byte loads).
constexpr int PACK_THREADS = 256;

__global__ void __launch_bounds__(PACK_THREADS) k_pack_reads_fixed(const uint8_t* bases, uint32_t L, uint32_t reads_per_block, const uint32_t* chunk_off,
                                                                   uint64_t n_reads, int ascii, uint32_t* packed, uint32_t* len_out,
                                                                   unsigned long long* bad) {
    extern __shared__ uint4 s_raw[];
    uint8_t* sb = reinterpret_cast<uint8_t*>(s_raw);
    const uint64_t r0 = (uint64_t)blockIdx.x * reads_per_block;
    if (r0 >= n_reads) return;
    const uint32_t R = (uint32_t)((n_reads - r0) < reads_per_block ? (n_reads - r0) : reads_per_block);
    // absolute byte range of this block's reads, widened to whole aligned 16-byte units (device allocations are at least
    // 256-byte aligned and sized, so the widened range never leaves the caller's allocation)
    const uintptr_t p0 = reinterpret_cast<uintptr_t>(bases) + r0 * L, p1 = p0 + (uintptr_t)R * L;
    const uintptr_t a0 = p0 & ~(uintptr_t)15;
    const uint32_t n16 = (uint32_t)((p1 - a0 + 15) >> 4);
    for (uint32_t i = threadIdx.x; i < n16; i += PACK_THREADS) s_raw[i] = __ldg(reinterpret_cast<const uint4*>(a0) + i);
    __syncthreads();
    const uint32_t skew = (uint32_t)(p0 - a0);
    const uint32_t wpr = ((L + 63u) / 64u) * 4u;                           // output words per read
    for (uint32_t w = threadIdx.x; w < R * wpr; w += PACK_THREADS) {
        const uint32_t r = w / wpr, k = w - r * wpr;
        const uint8_t* src = sb + skew + (size_t)r * L + k * 16u;
        uint32_t v = 0;
        for (uint32_t t = 0; t < 16u && k * 16u + t < L; ++t) {
            uint32_t c = src[t];
            if (ascii) c = c == 'A' ? 0u : c == 'C' ? 1u : c == 'G' ? 2u : c == 'T' ? 3u : 4u;
            if (c > 3u) {
                atomicMin(bad, (unsigned long long)(r0 + r));
                c = 0;
            }
            v |= c << (30u - 2u * t);
        }
        packed[(uint64_t)chunk_off[r0 + r] * 4u + k] = v;
        if (len_out && k == 0) len_out[r0 + r] = L;
    }
}

// ---------------------------------------------------------------------------------------------- FASTQ on the device
// A 4-line FASTQ held in device memory is cut into records here instead of on the host cores (the host scanner manages a
// few million reads/s; the search kernels take > 100 M reads/s): line ends are counted per 16 KB tile, the tile counts are
// prefix-summed by the caller, and a second pass gives every newline its global line number: line 4r ends where read
// r's bases begin, line 4r+1 ends where they end.  Replaces the one-string-per-file query path of the reference
// (ExactMatch.load_query, ExactMatch.py:104-108) for sequencer output.
constexpr uint32_t FQ_TILE = 16384;          // bytes per block
constexpr uint32_t FQ_THREADS = 256;         // 64 bytes per thread

__device__ __forceinline__ uint32_t count_nl16(uint4 v) {
    return __popc(__vcmpeq4(v.x, 0x0A0A0A0Au) & 0x01010101u) + __popc(__vcmpeq4(v.y, 0x0A0A0A0Au) & 0x01010101u) +
           __popc(__vcmpeq4(v.z, 0x0A0A0A0Au) & 0x01010101u) + __popc(__vcmpeq4(v.w, 0x0A0A0A0Au) & 0x01010101u);
}

// newlines in this thread's 64-byte piece [p, p+64) of buf (clipped to n); buf is 16-byte aligned
__device__ __forceinline__ uint32_t piece_newlines(const uint8_t* buf, uint64_t p, uint64_t n) {
    uint32_t c = 0;
    if (p + 64 <= n) {
        const uint4* q = reinterpret_cast<const uint4*>(buf + p);
#pragma unroll
        for (int i = 0; i < 4; ++i) c += count_nl16(__ldg(q + i));
    } else {
        for (uint64_t i = p; i < n; ++i) c += buf[i] == '\n';
    }
    return c;
}

__global__ void __launch_bounds__(FQ_THREADS) k_fq_count(const uint8_t* buf, uint64_t n, uint32_t* tile_counts) {
    __shared__ uint32_t warp_sum[FQ_THREADS / 32];
    const uint64_t p = (uint64_t)blockIdx.x * FQ_TILE + (uint64_t)threadIdx.x * 64u;
    uint32_t c = p < n ? piece_newlines(buf, p, n) : 0u;
    for (int d = 16; d; d >>= 1) c += __shfl_xor_sync(0xFFFFFFFFu, c, d);
    if ((threadIdx.x & 31u) == 0) warp_sum[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (uint32_t w = 0; w < FQ_THREADS / 32; ++w) t += warp_sum[w];
        tile_counts[blockIdx.x] = t;
    }
}

// err[0]: smallest byte offset at which the 4-line structure is violated (a record not starting with '@', a third line
// not starting with '+'), ~0 if none
__global__ void __launch_bounds__(FQ_THREADS) k_fq_records(const uint8_t* buf, uint64_t n, const unsigned long long* tile_prefix, uint64_t n_records,
                                                           unsigned long long* seq_start, unsigned long long* seq_end, unsigned long long* err) {
    __shared__ uint32_t scan[FQ_THREADS];
    const uint64_t p = (uint64_t)blockIdx.x * FQ_TILE + (uint64_t)threadIdx.x * 64u;
    const uint32_t mine = p < n ? piece_newlines(buf, p, n) : 0u;
    scan[threadIdx.x] = mine;
    __syncthreads();
    for (uint32_t d = 1; d < FQ_THREADS; d <<= 1) {          // inclusive Hillis-Steele scan of 256 counts
        const uint32_t v = threadIdx.x >= d ? scan[threadIdx.x - d] : 0u;
        __syncthreads();
        scan[threadIdx.x] += v;
        __syncthreads();
    }
    if (mine == 0u) return;
    unsigned long long line = tile_prefix[blockIdx.x] + scan[threadIdx.x] - mine;      // number of the first line that ends in this piece
    const uint64_t end = p + 64 < n ? p + 64 : n;
    for (uint64_t i = p; i < end; ++i) {
        if (buf[i] != '\n') continue;
        const unsigned long long r = line >> 2;
        const uint32_t k = (uint32_t)(line & 3u);
        if (r < n_records) {
            if (k == 0u) seq_start[r] = i + 1;
            else if (k == 1u) {
                seq_end[r] = (i > 0 && buf[i - 1] == '\r') ? i - 1 : i;
                if (i + 1 < n && buf[i + 1] != '+') atomicMin(err, (unsigned long long)i + 1);
            } else if (k == 3u && i + 1 < n && buf[i + 1] != '@') atomicMin(err, (unsigned long long)i + 1);
        }
        ++line;
    }
}

// reads scattered in a byte buffer (FASTQ sequence lines): read r = bases[start[r], start[r] + len[r])
__global__ void __launch_bounds__(256) k_pack_reads_scattered(const uint8_t* bases, const unsigned long long* start, const uint32_t* len,
                                                              const uint32_t* chunk_off, uint64_t n_reads, int ascii, uint32_t* packed,
                                                              unsigned long long* bad) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warp0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t r = warp0; r < n_reads; r += n_warps) {
        const uint64_t b0 = start[r];
        const uint32_t L = len[r];
        uint32_t* dst = packed + (uint64_t)chunk_off[r] * 4u;
        const uint32_t n_words = ((L + 63u) / 64u) * 4u;
        for (uint32_t w = lane; w < n_words; w += 32u) {
            uint32_t v = 0;
            const uint32_t t0 = w * 16u;
            for (uint32_t t = 0; t < 16u && t0 + t < L; ++t) {
                uint32_t c = bases[b0 + t0 + t];
                if (ascii) c = c == 'A' ? 0u : c == 'C' ? 1u : c == 'G' ? 2u : c == 'T' ? 3u : 4u;
                if (c > 3u) {
                    atomicMin(bad, (unsigned long long)r);
                    c = 0;
                }
                v |= c << (30u - 2u * t);
            }
            dst[w] = v;
        }
    }
}

// Strand-doubled batch: read r of the input -> slot 2r (the read) and slot 2r+1 (its reverse complement), one warp per
// read, one lane per output word pair (strand_logic.cuh).  Chunk offsets are rebased to the view's first read: slot 2r
// starts at 2 (c[r] - c[0]), slot 2r+1 right after it.  Thread 0 also writes the closing offset and zeroes the pad chunk.
__global__ void __launch_bounds__(256) k_both_strands(const uint32_t* __restrict__ src, const uint32_t* __restrict__ chunk_off,
                                                      const uint32_t* __restrict__ len, uint64_t n_reads, uint32_t* __restrict__ dst,
                                                      uint32_t* __restrict__ chunk_off_out, uint32_t* __restrict__ len_out) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warp0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint32_t c0 = __ldg(chunk_off);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        const uint32_t end = 2u * (__ldg(chunk_off + n_reads) - c0);
        chunk_off_out[2 * n_reads] = end;
        reinterpret_cast<uint4*>(dst)[end] = make_uint4(0u, 0u, 0u, 0u);
    }
    for (uint64_t r = warp0; r < n_reads; r += n_warps) {
        const uint32_t a = __ldg(chunk_off + r) - c0, nch = __ldg(chunk_off + r + 1) - c0 - a;
        const uint32_t L0 = __ldg(len + r);
        const uint32_t L = min(L0, nch * 64u);              // never read past the read's own chunks
        if (lane == 0) {
            chunk_off_out[2 * r] = 2u * a;
            chunk_off_out[2 * r + 1] = 2u * a + nch;
            len_out[2 * r] = L0;
            len_out[2 * r + 1] = L0;
        }
        const uint32_t* s = src + (uint64_t)(a + c0) * 4u;
        uint32_t* fwd = dst + (uint64_t)a * 8u;
        uint32_t* rc = fwd + (uint64_t)nch * 4u;
        for (uint32_t w = lane; w < nch * 4u; w += 32u) {
            const uint32_t m = strand_word_mask(L, w);
            fwd[w] = m ? __ldg(s + w) & m : 0u;
            StrandSrc q;
            uint32_t v = 0u;
            if (strand_rc_src(L, w, &q)) {
                const uint32_t hi = q.q >= 0 ? __ldg(s + q.q) : 0u;
                const uint32_t lo = q.sh ? __ldg(s + q.q + 1) : 0u;
                v = strand_rc_word(hi, lo, q.sh, L, w);
            }
            rc[w] = v;
        }
    }
}

}  // namespace
}  // namespace gsm

using namespace gsm;

extern "C" {

int gsm_pack_reads_device(const void* bases, const uint64_t* base_off, uint32_t fixed_len, const uint32_t* chunk_off, uint64_t n_reads,
                          uint32_t ascii, void* packed, uint32_t* len_out, uint64_t* scratch8, void* stream) {
    if (!bases || !chunk_off || !packed || !scratch8) return fail(GSM_E_INVALID, "gsm_pack_reads_device: null");
    if (!base_off && fixed_len == 0) return fail(GSM_E_INVALID, "gsm_pack_reads_device: base_off is NULL and fixed_len is 0");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(GSM_E_NODEVICE, "no CUDA device");
    if (n_reads == 0) return GSM_OK;
    cudaStream_t st = (cudaStream_t)stream;
    GSM_CUDA(cudaMemsetAsync(scratch8, 0xFF, 8, st));
    if (!base_off && fixed_len <= 2048) {
        // reads per block: 64, fewer for long reads so that the staged bytes fit 40 KB of shared memory
        uint32_t rpb = 64;
        while (rpb > 1 && (uint64_t)rpb * fixed_len + 32 > 40960) rpb >>= 1;
        const size_t smem = (((size_t)rpb * fixed_len + 31) / 16 + 1) * 16;
        const uint64_t blocks = (n_reads + rpb - 1) / rpb;
        if (blocks < (1ull << 31)) {
            k_pack_reads_fixed<<<(unsigned)blocks, PACK_THREADS, smem, st>>>((const uint8_t*)bases, fixed_len, rpb, chunk_off, n_reads, (int)ascii,
                                                                           (uint32_t*)packed, len_out, (unsigned long long*)scratch8);
            GSM_CUDA(cudaGetLastError());
            return GSM_OK;
        }
    }
    const uint64_t warps = n_reads;
    const unsigned grid = (unsigned)std::min<uint64_t>((warps + 7) / 8, 148ull * 32);
    k_pack_reads<<<grid, 256, 0, st>>>((const uint8_t*)bases, (const unsigned long long*)base_off, fixed_len, chunk_off, n_reads, (int)ascii,
                                       (uint32_t*)packed, len_out, (unsigned long long*)scratch8);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

int gsm_fastq_count_device(const void* buf, uint64_t n_bytes, uint32_t* tile_counts, void* stream) {
    if (!buf || !tile_counts) return fail(GSM_E_INVALID, "gsm_fastq_count_device: null");
    if ((reinterpret_cast<uintptr_t>(buf) & 15u) != 0) return fail(GSM_E_INVALID, "gsm_fastq_count_device: buf must be 16-byte aligned");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(GSM_E_NODEVICE, "no CUDA device");
    if (n_bytes == 0) return GSM_OK;
    const uint64_t tiles = (n_bytes + FQ_TILE - 1) / FQ_TILE;
    if (tiles >= (1ull << 31)) return fail(GSM_E_INVALID, "gsm_fastq_count_device: buffer too large for one call");
    k_fq_count<<<(unsigned)tiles, FQ_THREADS, 0, (cudaStream_t)stream>>>((const uint8_t*)buf, n_bytes, tile_counts);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

int gsm_fastq_records_device(const void* buf, uint64_t n_bytes, const uint64_t* tile_prefix, uint64_t n_records, uint64_t* seq_start,
                             uint64_t* seq_end, uint64_t* err8, void* stream) {
    if (!buf || !tile_prefix || !err8 || (n_records && (!seq_start || !seq_end))) return fail(GSM_E_INVALID, "gsm_fastq_records_device: null");
    if ((reinterpret_cast<uintptr_t>(buf) & 15u) != 0) return fail(GSM_E_INVALID, "gsm_fastq_records_device: buf must be 16-byte aligned");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(GSM_E_NODEVICE, "no CUDA device");
    cudaStream_t st = (cudaStream_t)stream;
    GSM_CUDA(cudaMemsetAsync(err8, 0xFF, 8, st));
    if (n_bytes == 0 || n_records == 0) return GSM_OK;
    const uint64_t tiles = (n_bytes + FQ_TILE - 1) / FQ_TILE;
    k_fq_records<<<(unsigned)tiles, FQ_THREADS, 0, st>>>((const uint8_t*)buf, n_bytes, (const unsigned long long*)tile_prefix, n_records,
                                                          (unsigned long long*)seq_start, (unsigned long long*)seq_end, (unsigned long long*)err8);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

int gsm_pack_reads_scattered_device(const void* bases, const uint64_t* seq_start, const uint32_t* seq_len, const uint32_t* chunk_off,
                                    uint64_t n_reads, uint32_t ascii, void* packed, uint64_t* scratch8, void* stream) {
    if (!bases || !seq_start || !seq_len || !chunk_off || !packed || !scratch8) return fail(GSM_E_INVALID, "gsm_pack_reads_scattered_device: null");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(GSM_E_NODEVICE, "no CUDA device");
    cudaStream_t st = (cudaStream_t)stream;
    GSM_CUDA(cudaMemsetAsync(scratch8, 0xFF, 8, st));
    if (n_reads == 0) return GSM_OK;
    const unsigned grid = (unsigned)std::min<uint64_t>((n_reads + 7) / 8, 148ull * 32);
    k_pack_reads_scattered<<<grid, 256, 0, st>>>((const uint8_t*)bases, (const unsigned long long*)seq_start, seq_len, chunk_off, n_reads, (int)ascii,
                                                 (uint32_t*)packed, (unsigned long long*)scratch8);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

int gsm_reads_both_strands_device(const gsm_dev_reads* in, void* packed_out, uint32_t* chunk_off_out, uint32_t* len_out, void* stream) {
    if (!in || !packed_out || !chunk_off_out || !len_out || !in->packed || !in->chunk_off || (in->n_reads && !in->len))
        return fail(GSM_E_INVALID, "gsm_reads_both_strands_device: null");
    // the doubled offsets are at most 2 * n * ceil(max_len / 64) chunks
    const uint64_t n = in->n_reads;
    if (n >= (1ull << 31) || 2ull * n * (((uint64_t)in->max_len + 63) / 64) >= (1ull << 32))
        return fail(GSM_E_CAPACITY, "gsm_reads_both_strands_device: the doubled chunk offsets do not fit in 32 bits");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(GSM_E_NODEVICE, "no CUDA device");
    const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((n + 7) / 8, 148ull * 32));
    k_both_strands<<<grid, 256, 0, (cudaStream_t)stream>>>((const uint32_t*)in->packed, in->chunk_off, in->len, n, (uint32_t*)packed_out,
                                                           chunk_off_out, len_out);
    GSM_CUDA(cudaGetLastError());
    return GSM_OK;
}

/* Result of the validity check of the last gsm_pack_reads_device on this scratch word: GSM_OK, or GSM_E_INVALID
 * naming the first read that holds a non-ACGT byte.  Synchronises the stream. */
int gsm_pack_reads_device_check(const uint64_t* scratch8, void* stream) {
    unsigned long long bad = 0;
    GSM_CUDA(cudaMemcpyAsync(&bad, scratch8, 8, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    GSM_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    if (bad != ~0ull) return fail(GSM_E_INVALID, "non-ACGT base in read " + std::to_string(bad));
    return GSM_OK;
}

}  // extern "C"
