/*
 * genie_smem.h -- C ABI of the B200-native SMEM-seeding engine (libgenie_smem.so).
 *
 * This is the drop-in boundary for GENIE-SMEM's search path.  The reference is pure Python
 * (no FFI of its own), so each entry point cites the reference routine (file:line under
 * /root/reference/SMEM/) it replaces; INTEGRATION.md shows the ctypes stub a maintainer
 * would add to the reference classes.
 *
 * Conventions
 *   - every function returns int status: 0 ok, <0 error (GSM_E_*); nothing throws across
 *     the boundary; gsm_last_error() gives the text of the last failure on this thread;
 *   - plain pointers and sizes only; the caller (torch tensors / numpy arrays) owns every
 *     buffer, the library never allocates device memory;
 *   - `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream);
 *   - rows are 0-based suffix-array rows over n = n_bases + 1 rows (row 0 is the '$'
 *     suffix); an SA interval is reported as (lo, cnt) with cnt == 0 meaning "no match"
 *     (the reference's int -1, ExactMatch.py:149); suffix-array VALUES are 1-based text
 *     positions exactly as ExactMatch.py:66 stores them;
 *   - bases are codes A=0 C=1 G=2 T=3 (LUT.py:39-43); sequences are 2-bit packed MSB-first:
 *     base i sits in bits [30-2*(i%16), 32-2*(i%16)) of 32-bit word i/16, so the top 2K bits of
 *     a window are the k-mer code of LUT.convert_seq_to_num (LUT.py:37-48); every read starts
 *     on a 16-byte boundary of the packed buffer, and packed buffers (reads and text) must be
 *     readable 16 bytes past their last word.
 */
#ifndef GENIE_SMEM_H
#define GENIE_SMEM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GSM_OK 0
#define GSM_E_INVALID (-1)   /* bad argument (non-ACGT base, null pointer, size mismatch) */
#define GSM_E_NOMEM (-2)     /* host allocation failed */
#define GSM_E_CUDA (-3)      /* CUDA runtime error (text in gsm_last_error) */
#define GSM_E_CAPACITY (-4)  /* a caller-provided buffer is too small */
#define GSM_E_NODEVICE (-5)  /* no CUDA device: there is NO CPU fallback */

#define GSM_METHOD_BWA 0 /* SMEM.get_SMEMS      (SMEM.py:456-467) */
#define GSM_METHOD_LUT 1 /* SMEM.get_smems_lut  (SMEM.py:20-192)  */
#define GSM_METHOD_RMI 2 /* SMEM.get_smems_rmi  (SMEM.py:206-384) */

/* per-read status bits written by the SMEM kernels */
#define GSM_READ_OK 0u
#define GSM_READ_REF_RAISES 1u /* the reference raises on this read (RMI last-mile search leaves
                                  the table: RecursionError / IndexError, RMI_LUT.py:136-184) */
#define GSM_READ_TOO_SHORT 2u  /* len < K for LUT/RMI (the reference's behaviour is undefined) */

#define GSM_BUCKET_BYTES 64
#define GSM_BUCKET_SYMS 192

/* ------------------------------------------------------------------ host-side index */
typedef struct gsm_index gsm_index; /* opaque, immutable after build */

typedef struct {
    uint64_t n_bases;
    uint64_t n_rows;       /* n_bases + 1                         (fm_index["ref_size"]) */
    uint64_t n_buckets;    /* 64-byte rank buckets per direction                        */
    uint64_t bucket_bytes; /* n_buckets * 64                                            */
    uint64_t text_words;   /* 32-bit words of the 2-bit packed text incl. 2 pad words    */
    uint32_t count[4];     /* occurrences of A,C,G,T in the text                        */
    uint32_t C[5];         /* first row whose suffix starts with A,C,G,T; C[4]=n_rows
                              (fm_index["count_dic"], ExactMatch.py:92-101)             */
    uint32_t primary_fwd;  /* row of the forward BWT holding '$'                        */
    uint32_t primary_rev;  /* same for the BWT of the reversed text                     */
    uint32_t has_reverse;  /* 1 if the reverse-text BWT was built                       */
    uint32_t reserved;
} gsm_index_info;

/* Build BWT / SA / C of text+'$' with an O(n) suffix sorter.
 * Replaces ExactMatch.create_fm_index (ExactMatch.py:22-33, 52-101: n^2 rotation sort).
 * bases: n_bases ASCII chars from {A,C,G,T}.  flags: bit0 = also build the BWT of the
 * reversed text (needed by the SMEM kernels' forward extension). */
int gsm_index_build(const char* bases, uint64_t n_bases, uint32_t flags, gsm_index** out);

/* Import reference-built arrays (fm_index["suffix_array"], 1-based) instead of sorting:
 * the "same index arrays" clause.  Replaces ExactMatch.load_fm_index (ExactMatch.py:35-41). */
int gsm_index_from_arrays(const char* bases, uint64_t n_bases, const uint32_t* suffix_array_1based,
                          uint32_t flags, gsm_index** out);

int gsm_index_info_get(const gsm_index* idx, gsm_index_info* out);

/* Export in the reference's schema (ExactMatch.py:29-30): suffix_array (1-based, n_rows
 * entries) and bwt (n_rows chars, '$' at the primary row).  Either pointer may be NULL. */
int gsm_index_export(const gsm_index* idx, uint32_t* suffix_array_1based, char* bwt);

/* Fill caller-allocated HOST buffers with the device layouts (the caller then copies them
 * to the GPU).  Any pointer may be NULL to skip that array.
 *   fwd_buckets / rev_buckets : n_buckets * 64 bytes each
 *   sa                        : n_rows uint32 (1-based values, as exported)
 *   text2bit                  : text_words uint32 */
int gsm_index_pack(const gsm_index* idx, void* fwd_buckets, void* rev_buckets, uint32_t* sa,
                   uint32_t* text2bit);

void gsm_index_free(gsm_index* idx);

/* Pack ASCII reads into the device read format.  lens[i] bases each, concatenated in
 * `bases`.  chunk_off (n_reads+1 entries) receives each read's offset in 16-byte chunks;
 * packed must hold chunk_off[n_reads]*16 bytes -- call with packed == NULL to size it.
 * Returns GSM_E_INVALID on a non-ACGT base (the reference raises KeyError there). */
int gsm_pack_reads(const char* bases, const uint32_t* lens, uint64_t n_reads, uint32_t* chunk_off,
                   void* packed);

/* ------------------------------------------------------------------ device-side index build */
/* The same index as gsm_index_build, constructed ON THE GPU (radix sort of 32-mer keys + prefix doubling
 * over the rows that are still tied; BWT planes by ballot; checkpoints by scan) -- seconds at 10^9 bases.
 * Replaces ExactMatch.create_fm_index (ExactMatch.py:22-33, 52-101) for large references; bit-identical
 * arrays to the host builder.  All pointers below are DEVICE memory owned by the caller.
 *
 * gsm_text_pack_device: bases (n_bases bytes: ASCII ACGT if ascii != 0, else codes 0..3) -> text2bit
 *   ((n_bases+15)/16 + 2 words, MSB-first, pad words zeroed).  scratch8: 8 bytes of device scratch.
 *   GSM_E_INVALID on a non-ACGT base (the reference raises KeyError, ExactMatch.py:139).
 * gsm_index_build_device_workspace: bytes of scratch gsm_index_build_device needs (about 36 bytes per base).
 * gsm_index_build_device: text2bit -> sa (n_rows uint32, 1-based values), fwd_buckets and (flags bit0)
 *   rev_buckets (n_buckets * 64 bytes each); *info (HOST) receives sizes, count[], C[], primary rows;
 *   info->reserved = prefix-doubling rounds used.  Synchronises the stream. */
int gsm_text_pack_device(const void* bases, uint64_t n_bases, uint32_t ascii, uint32_t* text2bit, uint64_t* scratch8,
                         void* stream);
int gsm_index_build_device_workspace(uint64_t n_bases, uint32_t flags, uint64_t* bytes);
int gsm_index_build_device(const uint32_t* text2bit, uint64_t n_bases, uint32_t flags, uint32_t* sa, void* fwd_buckets,
                           void* rev_buckets, void* workspace, uint64_t workspace_bytes, gsm_index_info* info,
                           void* stream);

/* ------------------------------------------------------------------ host-side read ingest */
/* Multi-threaded scan of a 4-line FASTQ held in memory (threads == 0: all cores).  gsm_fastq_scan: *n_records = lines / 4;
 * with seq_off / seq_len non-NULL (cap entries) also the offset and length of every sequence line ('\r' stripped).
 * GSM_E_INVALID for a truncated file or records that do not start with '@' / carry no '+' line.  gsm_fastq_gather copies
 * the sequence lines into one contiguous buffer (out may be NULL to get base_off only): base_off[i] = start of read i,
 * n_records + 1 entries -- exactly the (bases, base_off) pair gsm_pack_reads_device takes.  Replaces the one-string-per-
 * file query path (ExactMatch.load_query, ExactMatch.py:104-108). */
int gsm_fastq_scan(const char* buf, uint64_t n_bytes, uint64_t* n_records, uint64_t* seq_off, uint32_t* seq_len, uint64_t cap,
                   uint32_t threads);
int gsm_fastq_gather(const char* buf, const uint64_t* seq_off, const uint32_t* seq_len, uint64_t n_records, char* out,
                     uint64_t* base_off, uint32_t threads);

/* ------------------------------------------------------------------ device-side read ingest */
/* Pack reads ON THE GPU: bases (device; ASCII ACGT if ascii != 0, else codes 0..3), read r = bytes
 * [base_off[r], base_off[r+1]) (device uint64, n_reads+1) or, with base_off == NULL, fixed_len bytes at
 * r*fixed_len; chunk_off (device, n_reads+1, 16-byte chunks: exclusive scan of ceil(len/64)) as in
 * gsm_pack_reads; packed receives chunk_off[n_reads]*16 bytes; len_out (optional, device) the lengths.
 * Fixed-length batches are staged through shared memory with aligned 16-byte loads: the kernel may read up to 15 bytes
 * before and after the byte range, inside the caller's (>= 256-byte aligned) allocation.
 * Replaces the per-string query path (ExactMatch.load_query, ExactMatch.py:104-108) for batches.
 * Asynchronous; gsm_pack_reads_device_check(scratch8) synchronises and returns GSM_E_INVALID if a read
 * held a non-ACGT byte (the reference raises KeyError, ExactMatch.py:139). */
int gsm_pack_reads_device(const void* bases, const uint64_t* base_off, uint32_t fixed_len, const uint32_t* chunk_off,
                          uint64_t n_reads, uint32_t ascii, void* packed, uint32_t* len_out, uint64_t* scratch8,
                          void* stream);
int gsm_pack_reads_device_check(const uint64_t* scratch8, void* stream);

/* FASTQ record cutting ON THE GPU (the host scanner above manages a few million reads/s; the search takes > 100 M/s).
 * buf: the bytes of a 4-line FASTQ in DEVICE memory, 16-byte aligned.  Tiles are GSM_FASTQ_TILE bytes.
 *   gsm_fastq_count_device    tile_counts[t] = line feeds in tile t (ceil(n_bytes / tile) uint32).  The caller prefix-sums them
 *                             (exclusive, uint64: tile_prefix) and reads the total: lines = total (+1 without a final line feed),
 *                             records = lines / 4.
 *   gsm_fastq_records_device  seq_start[r] / seq_end[r] = byte range of record r's sequence line ('\r' stripped); *err8 (device
 *                             uint64) = smallest offset where a record does not begin with '@' or its third line with '+', else ~0.
 *   gsm_pack_reads_scattered_device  gsm_pack_reads_device for reads that are NOT contiguous: read r = bases[seq_start[r],
 *                             seq_start[r] + seq_len[r]); chunk_off as there; scratch8 as there (gsm_pack_reads_device_check).
 * Replaces ExactMatch.load_query (ExactMatch.py:104-108) for sequencer output; all asynchronous on `stream`. */
#define GSM_FASTQ_TILE 16384
int gsm_fastq_count_device(const void* buf, uint64_t n_bytes, uint32_t* tile_counts, void* stream);
int gsm_fastq_records_device(const void* buf, uint64_t n_bytes, const uint64_t* tile_prefix, uint64_t n_records, uint64_t* seq_start,
                             uint64_t* seq_end, uint64_t* err8, void* stream);
int gsm_pack_reads_scattered_device(const void* bases, const uint64_t* seq_start, const uint32_t* seq_len, const uint32_t* chunk_off,
                                    uint64_t n_reads, uint32_t ascii, void* packed, uint64_t* scratch8, void* stream);

/* ------------------------------------------------------------------ device-side views */
typedef struct {
    uint64_t n_rows;
    uint64_t n_buckets;
    const void* fwd_buckets; /* device */
    const void* rev_buckets; /* device, may be NULL for gsm_backsearch_batch / gsm_lut_build */
    const uint32_t* sa;      /* device, 1-based values; needed by RMI and gsm_sa_lookup */
    const uint32_t* text2bit; /* device; needed by RMI */
    uint32_t C[5];
    uint32_t primary_fwd;
    uint32_t primary_rev;
    uint32_t seed_K;          /* K of seed_table (1..14), ignored when seed_table is NULL */
    const void* seed_table;   /* device, optional: gsm_seed_table_build output (4^K x 16 bytes); lets the sweep
                                 kernel replace the first K steps of every extension by one fetch */
} gsm_dev_index;

typedef struct {
    uint64_t n_reads;
    const void* packed;        /* device, 2-bit packed reads */
    const uint32_t* chunk_off; /* device, n_reads + 1 */
    const uint32_t* len;       /* device, n_reads */
    uint32_t max_len;          /* max over len[] */
    uint32_t read_id_base;     /* added to the read index in emitted records (rank sharding) */
} gsm_dev_reads;

/* Strand-doubled batch, built ON THE GPU: the n reads of `in` become 2n slots, interleaved -- slot 2i is read i as given,
 * slot 2i+1 its reverse complement (base k = 3 - base[L-1-k] in the A=0 C=1 G=2 T=3 codes).  Run the SMEM entry points
 * on the doubled batch with read_id_base = 2 * (the original read_id_base): a record's read_id is then
 * 2 * (read_id_base + i) + strand, so read_id >> 1 is the read and read_id & 1 the strand.  Slot 2i gets exactly the
 * records of read i in every field but read_id; slot 2i+1 gets what the method gives for the reverse-complement string,
 * with qstart / qend in ITS coordinates (read[L-qend : L-qstart] on the reverse strand); a palindromic read gets the same
 * records on both strands.  A hit of a strand-1 record at (contig, offset) means RC(read)[qstart:qend] occurs on the
 * forward strand there: the hit entry points do not change.
 *   in:            reads in->packed, in->chunk_off (n+1) and in->len (n); may be a view of reads [lo, hi) with
 *                  chunk_off[0] != 0.  in->max_len bounds the lengths.
 *   chunk_off_out: 2n+1 entries starting at 0: [2r] = 2 (c[r] - c[0]), [2r+1] = (c[r] - c[0]) + (c[r+1] - c[0]).
 *   len_out:       2n entries.
 *   packed_out:    2 (c[n] - c[0]) * 16 + 16 bytes; pad bits and the pad chunk are zero, so the output is byte-identical
 *                  to gsm_pack_reads of the interleaved strings [r0, rc(r0), r1, rc(r1), ...].
 * GSM_E_INVALID for a null pointer, GSM_E_CAPACITY when 2 n ceil(max_len / 64) chunks would not fit in 32 bits.
 * Asynchronous on `stream`. */
int gsm_reads_both_strands_device(const gsm_dev_reads* in, void* packed_out, uint32_t* chunk_off_out, uint32_t* len_out,
                                  void* stream);

/* One emitted SMEM, before the reference's dict collapses duplicate strings.  16 bytes. */
typedef struct {
    uint32_t read_id;
    uint16_t qstart; /* SMEM = read[qstart:qend] */
    uint16_t qend;
    uint32_t sa_lo; /* inclusive rows, the reference's tuple (lo, hi) */
    uint32_t sa_hi;
} gsm_record;

/* RMI parameters (RMI.py:52-69): level_sizes[l] models at level l (level 0 has 1), flattened
 * coef/intercept in level order; prediction = fl(fl(x*coef)+intercept) per level. */
typedef struct {
    uint32_t K;             /* RMI_LUT.prediction_size */
    uint32_t n_levels;
    const uint32_t* level_sizes; /* HOST pointer, n_levels entries */
    const double* coef;          /* device */
    const double* intercept;     /* device */
    const void* probe;           /* device, optional: n_rows x 16 B from gsm_rmi_probe_build, else NULL */
    const uint32_t* none_rows;   /* HOST pointer, optional: the K rows of gsm_rmi_none_rows; enables the error-bounded
                                    fast search (identical bounds, far fewer instructions), else NULL */
    uint32_t n_none_rows;        /* K, or 0 */
    uint32_t param_stride;       /* elements between consecutive models in coef[] / intercept[]: 0 or 1 = two dense arrays;
                                    2 = one interleaved {coef, intercept} array (intercept == coef + 1): one line per model */
    const void* bounds;          /* device, optional: 4^K x 8 B from gsm_rmi_bounds_build (used with none_rows), else NULL */
    const uint32_t* hazard_slots; /* device, optional: hash set of the model's hazard codes (gsm_rmi_hazard_scan +
                                    gsm_rmi_hazard_hash; used with bounds), else NULL */
    uint32_t hazard_n_slots;     /* words in hazard_slots (a power of two), or 0 */
    uint32_t reserved0;
} gsm_dev_rmi;

/* Scratch + output buffers for one SMEM batch; all device memory, all caller-allocated.
 * gsm_smem_workspace_bytes() says how large each must be. */
typedef struct {
    void* mem_pool;        /* classical-SMEM pool, mem_cap entries of 16 bytes */
    uint64_t mem_cap;
    void* quad_scratch;    /* per-resident-quad staging */
    uint64_t quad_scratch_bytes;
    uint32_t* mem_off;     /* n_reads */
    uint32_t* mem_cnt;     /* n_reads: matches per read (low 30 bits); bit 31 = the list is in ascending order and stored field by
                              field, bit 30 = ... and carries the BWA-SMEM picks in place of its first sweep ordinal */
    gsm_record* rec_tmp;   /* unordered record pool, rec_cap entries */
    uint64_t rec_cap;
    uint32_t* rec_tmp_off; /* n_reads */
    uint32_t* rec_cnt;     /* n_reads: records per read (phase-1 result) */
    uint64_t* rec_off;     /* n_reads + 1: exclusive scan of rec_cnt */
    uint8_t* read_status;  /* n_reads: GSM_READ_* */
    uint64_t* counters;    /* 8 x uint64: [0] mems used, [1] records, [2] status bits, [3] next read, [4..7] scratch of the kernels */
    void* scan_tmp;        /* scan scratch */
    uint64_t scan_tmp_bytes;
} gsm_workspace;

typedef struct {
    uint64_t quad_scratch_bytes;
    uint64_t scan_tmp_bytes;
    uint32_t grid_blocks;   /* persistent grid used by the sweep kernel on this device */
    uint32_t block_threads;
} gsm_workspace_info;

int gsm_smem_workspace_info(uint64_t n_reads, uint32_t max_len, gsm_workspace_info* out);

/* ------------------------------------------------------------------ device search */
/* Batched backward search: ExactMatch.exact_match_back_prop (ExactMatch.py:132-151) for every
 * read.  lo[i], cnt[i]: rows [lo, lo+cnt); cnt == 0 <=> the reference returns -1. */
int gsm_backsearch_batch(const gsm_dev_index* idx, const gsm_dev_reads* reads, uint32_t* lo,
                         uint32_t* cnt, void* stream);

/* One backward-search step for a batch of (char, interval) pairs:
 * ExactMatch.exact_match_back_prop_add_one (ExactMatch.py:155-171). In place on lo/cnt. */
int gsm_backsearch_add_one_batch(const gsm_dev_index* idx, uint64_t n, const uint8_t* base,
                                 uint32_t* lo, uint32_t* cnt, void* stream);

/* rows -> 1-based text positions: ExactMatch.get_position(s) (ExactMatch.py:191-199). */
int gsm_sa_lookup_batch(const gsm_dev_index* idx, uint64_t n, const uint32_t* rows, uint32_t* pos,
                        void* stream);

/* Sampled suffix array: ssa[i] = suffix_array[i * sample], ceil(n_rows / sample) entries of device memory (needs idx->sa
 * once; afterwards the 4-byte-per-base suffix array can be dropped unless RMI-SMEM is used).  gsm_locate_sampled_batch:
 * rows -> 1-based text positions by LF-walking to the next sampled row -- ExactMatch.get_position(s)
 * (ExactMatch.py:191-199) with n/sample words instead of n; rows >= n_rows give 0. */
int gsm_sa_sample_build(const gsm_dev_index* idx, uint32_t sample, uint32_t* ssa, void* stream);
int gsm_locate_sampled_batch(const gsm_dev_index* idx, const uint32_t* ssa, uint32_t sample, uint64_t n,
                             const uint32_t* rows, uint32_t* pos, void* stream);

/* Dense k-mer table: entry[code] = {lo, cnt} for every 4^K code, cnt == 0 for absent k-mers.
 * Replaces LUT.generate_lut (LUT.py:15-35); table: 4^K * 8 bytes of device memory. */
int gsm_lut_build(const gsm_dev_index* idx, uint32_t K, uint32_t* table, void* stream);

/* Seed table for the sweep kernel: entry[code] = {rows lo of the k-mer on the text index, count, rows lo of the
 * reversed k-mer on the reversed-text index, 0}, 16 bytes per 4^K code.  The reference's LUT idea (LUT.py:15-35)
 * applied to both directions of the bidirectional extension; results never depend on it. */
int gsm_seed_table_build(const gsm_dev_index* idx, uint32_t K, void* table, void* stream);

/* The three SMEM entry points.  Phase 1 (this call) runs the kernels and leaves per-read
 * record counts in ws->rec_cnt, their exclusive scan in ws->rec_off and the total in
 * ws->counters[1]; phase 2 (gsm_smem_collect) writes the records in (read, emission) order.
 *   BWA: SMEM.get_SMEMS(query, min_len)            (SMEM.py:456-484, 389-443)
 *   LUT: SMEM.get_smems_lut(query), K = lut_size    (SMEM.py:20-192), lut = gsm_lut_build table
 *   RMI: SMEM.get_smems_rmi(query)                  (SMEM.py:206-384, RMI_LUT.py:53-184) */
int gsm_smem_batch(int method, const gsm_dev_index* idx, const gsm_dev_reads* reads, uint32_t min_len,
                   uint32_t K, const uint32_t* lut, const gsm_dev_rmi* rmi, gsm_workspace* ws,
                   void* stream);

/* get_smems_lut (SMEM.py:20-192) emits exactly the records of get_SMEMS (SMEM.py:456-467) with min_len 1 for every read of at
 * least K bases: each round of its frame machine returns the longest maximal match covering the previous SMEM's end, ties to
 * the smaller end (DESIGN.md section 3; checked on 11.5 M adversarial cases of the literal restatement).  By default
 * gsm_smem_select(GSM_METHOD_LUT) therefore takes the records from the sweep's picks and uses K only to flag reads that are too
 * short; on = 1 runs the frame machine itself (k_select_seeded<LUT>: same records, the cross-check), on < 0 only queries.
 * Returns the previous setting.  Process-wide; GSM_LUT_MACHINE=1 in the environment sets the initial value. */
int gsm_option_lut_frame_machine(int on);

/* The two halves of gsm_smem_batch, callable separately (bench.py times them separately).
 * gsm_smem_sweep: every maximal exact match of every read (the FM-index walk, method-independent)
 * into ws->mem_pool / mem_off / mem_cnt.  gsm_smem_select: the reference's record selection for
 * one method over that match list; it may be called several times after one sweep. */
int gsm_smem_sweep(const gsm_dev_index* idx, const gsm_dev_reads* reads, gsm_workspace* ws, void* stream);
int gsm_smem_select(int method, const gsm_dev_index* idx, const gsm_dev_reads* reads, uint32_t min_len,
                    uint32_t K, const uint32_t* lut, const gsm_dev_rmi* rmi, gsm_workspace* ws,
                    void* stream);

int gsm_smem_collect(const gsm_dev_reads* reads, gsm_workspace* ws, gsm_record* out, uint64_t out_cap,
                     void* stream);

/* ------------------------------------------------------------------ multi-GPU: the gather of per-rank records
 * The path shards by reads (rank r searches reads [r*N/G, (r+1)*N/G) against its own replica of the index); its only
 * exchange is the final gather of the per-rank record arrays to one rank (north_star (4), SURVEY 8e).  One process per
 * GPU; the launcher (torchrun, mpirun, ...) only has to carry the 128-byte id from rank 0 to the other ranks.
 *
 * gsm_comm_*: an NCCL communicator owned by the library (libnccl.so.2 is dlopen'ed on first use; GSM_E_INVALID when absent).
 *   gsm_comm_unique_id  rank 0: 128 bytes to broadcast;  gsm_comm_init: every rank, on its current CUDA device.
 * gsm_comm_allgather_u64: n values per rank, device to device (the per-rank record counts: ws->counters + 1).
 * gsm_gather_records: counts[world] (HOST) = records per rank; `send` = this rank's n_send = counts[rank] records
 *   (device); on dst `recv` (device, preallocated, sum(counts) records) receives every rank's records in rank order
 *   (one ncclGroup of exact-size ncclSend / ncclRecv; dst's own shard is a device-to-device copy).  Asynchronous on stream.
 *
 * Peer-memory gather (the fused path): gsm_peer_export names the allocation behind a device pointer of the gathering
 * rank (64-byte CUDA IPC handle + offset of the pointer in it), gsm_peer_open maps it in another process of the same
 * node (NVLink / NVSwitch peer access), gsm_peer_close(ptr, offset) unmaps it.  gsm_smem_collect_gathered is
 * gsm_smem_collect writing record k of this batch to out[*base_dev + sum(counts_dev[0..rank)) + k]: with `out` a peer
 * mapping, each rank's ordered write lands in the gathering rank's HBM and no separate gather pass exists.  counts_dev =
 * output of gsm_comm_allgather_u64 for this batch, base_dev = running total of earlier batches (device; NULL = 0),
 * advanced by gsm_gather_advance(base_dev, counts_dev, world) after each batch. */
typedef struct gsm_comm gsm_comm;
int gsm_comm_unique_id(void* id128);
int gsm_comm_init(const void* id128, int rank, int world, gsm_comm** out);
int gsm_comm_free(gsm_comm* comm);
int gsm_comm_info(const gsm_comm* comm, int* rank, int* world, int* nccl_version);
int gsm_comm_allgather_u64(gsm_comm* comm, const uint64_t* send_dev, uint64_t n, uint64_t* recv_dev, void* stream);
int gsm_gather_records(gsm_comm* comm, const gsm_record* send, uint64_t n_send, const uint64_t* counts, gsm_record* recv,
                       int dst, void* stream);
int gsm_peer_export(const void* dev_ptr, void* handle64, uint64_t* offset);
int gsm_peer_open(const void* handle64, uint64_t offset, void** dev_ptr);
int gsm_peer_close(void* dev_ptr, uint64_t offset);
int gsm_smem_collect_gathered(const gsm_dev_reads* reads, gsm_workspace* ws, gsm_record* out, uint64_t out_cap,
                              const uint64_t* counts_dev, uint32_t rank, const uint64_t* base_dev, void* stream);
int gsm_gather_advance(uint64_t* base_dev, const uint64_t* counts_dev, uint32_t world, void* stream);

/* Optional accelerator for the RMI last-mile search: probe[row] = {suffix_array[row], code of the 32
 * bases at that suffix} (16 bytes), so RMI_LUT.get_ref_seq (RMI_LUT.py:89-92) is ONE fetch instead of
 * a suffix-array read followed by a text read.  probe: n_rows * 16 bytes of device memory. */
int gsm_rmi_probe_build(const gsm_dev_index* idx, void* probe, void* stream);

/* Optional accelerator for the RMI lookups of gsm_smem_select: bounds[code] = {first row whose K-mer >= code, occurrences of
 * the K-mer} (two uint32) for all 4^K codes, K = the model's prediction size (K <= 16; 8.6 GB for K = 15).  The error-bounded
 * search of RMI_LUT.get_suffix_rmi (RMI_LUT.py:67-184) is a function of the prediction and of these true bounds
 * (rmi_arith_lookup), so a window then costs ONE fetch instead of a seed-table fetch plus K - seed_K backward steps.  Uses the
 * index's seed table when present (seed_K <= K) to shorten the build.  Results never depend on it. */
int gsm_rmi_bounds_build(const gsm_dev_index* idx, uint32_t K, void* bounds, void* stream);

/* The rows whose suffix is shorter than K bases (RMI_LUT.get_ref_seq returns None there, RMI_LUT.py:89-92): exactly K
 * rows.  rows_host (HOST, K entries, ascending); scratch: 33 uint32 of device memory.  With them in gsm_dev_rmi the
 * selection kernel can prove, per lookup, that the literal exponential + binary search equals a plain error-bounded
 * binary search, and runs that instead; the literal search remains the path for every lookup it cannot prove. */
int gsm_rmi_none_rows(const gsm_dev_index* idx, uint32_t K, uint32_t* rows_host, uint32_t* scratch, void* stream);

/* RMI-SMEM pre-filter.  What RMI_LUT.get_suffix_rmi (RMI_LUT.py:67-78) returns for a K-mer is a function of its code alone
 * (prediction, true bounds, None rows), and for all but a few codes per million -- the model's HAZARD codes -- it is the
 * k-mer's true interval.  On a read none of whose windows is a hazard, get_smems_rmi (SMEM.py:206-384) makes the very lookups
 * of get_smems_lut (SMEM.py:20-192; the two routines are the same text apart from the lookup) and so emits the records of
 * get_SMEMS with min_len 1 (DESIGN.md section 3): gsm_smem_select(GSM_METHOD_RMI) hands such reads to the BWA-SMEM selection
 * and runs the frame machine on the others only.  Results never depend on it.
 *   gsm_rmi_hazard_scan: every hazard code of `rmi` (needs bounds + none_rows, K <= 15) appended to codes[] (device, cap
 *     entries); *n_found (HOST) = how many there are -- more than cap: not all were stored, do not build the set.
 *     count_dev: 8 bytes of device scratch.  Synchronises the stream.
 *   gsm_rmi_hazard_hash (host only, no GPU needed): open-addressing set of n 32-bit codes in slots[n_slots], n_slots a power
 *     of two in [2 n + 2, 2^24]; upload it and name it in gsm_dev_rmi.hazard_slots / hazard_n_slots.
 *   gsm_option_rmi_prefilter: 1 (default) = use the set when present, 0 = frame machine for every read (the cross-check:
 *     same records), < 0 = query; returns the previous setting.  Process-wide; GSM_RMI_PREFILTER in the environment sets the
 *     initial value. */
int gsm_rmi_hazard_scan(const gsm_dev_index* idx, const gsm_dev_rmi* rmi, uint32_t* codes, uint64_t cap, uint64_t* count_dev,
                        uint64_t* n_found, void* stream);
int gsm_rmi_hazard_hash(const uint32_t* codes, uint64_t n, uint32_t* slots, uint32_t n_slots);
int gsm_option_rmi_prefilter(int on);

/* RMI_LUT.get_suffix_rmi (RMI_LUT.py:67-78) for a batch of K-mer codes: predict + exponential
 * + binary last-mile search.  pred receives the float64 prediction, lo/hi the returned pair
 * (hit <=> hi >= lo as int64), status GSM_READ_REF_RAISES where the reference would raise. */
int gsm_rmi_lookup_batch(const gsm_dev_index* idx, const gsm_dev_rmi* rmi, uint64_t n,
                         const uint64_t* codes, double* pred, int64_t* lo, int64_t* hi,
                         uint8_t* status, void* stream);

/* Random aligned 64-byte gather over `bytes` of device memory with the rank kernels' access
 * shape (4 lanes x 16 B): the measured ceiling the rank kernels are compared with (SURVEY 8d).
 * At least n_fetch buckets are fetched; *n_done receives the exact number.  dependent != 0:
 * every quad chases pointers (one FM chain each); 0: independent fetches.  sink: device u64. */
int gsm_gather_probe(const void* buf, uint64_t bytes, uint64_t n_fetch, uint32_t dependent,
                     uint64_t* sink, uint64_t* n_done, void* stream);

/* The same ceiling with the kernels' real access shapes and enough memory parallelism: every lane keeps `in_flight`
 * (1, 4 or 8) independent fetches of `fetch_bytes` (64 = a whole bucket by one lane: two requests, 66 = a whole bucket by a lane
 * pair: one 64-byte request, 32 = one 256-bit load, 16 = one seed-table entry) outstanding, indices masked to the largest
 * power of two of units in `bytes`. */
int gsm_gather_probe2(const void* buf, uint64_t bytes, uint64_t n_fetch, uint32_t fetch_bytes, uint32_t in_flight,
                      uint64_t* sink, uint64_t* n_done, void* stream);

/* Pin [ptr, ptr+bytes) in the persisting part of the L2 for kernels launched on `stream` (access-policy window; the small,
 * randomly read top of a structure: RMI model parameters, the top of a k-mer table).  ptr == NULL or bytes == 0 removes the
 * window and resets the persisting lines. */
int gsm_l2_persist(const void* ptr, uint64_t bytes, void* stream);

/* L2 fetch granularity of the current device (cudaLimitMaxL2FetchGranularity): the rank kernels read isolated
 * 64-byte buckets, so a 128-byte fetch granularity moves twice the necessary DRAM bytes.  set_bytes > 0 requests
 * 32 / 64 / 128 (a hint to the driver); *current receives the value in force. */
int gsm_device_l2_fetch_granularity(int32_t set_bytes, uint32_t* current);

const char* gsm_last_error(void);
int gsm_version(void);

/* ------------------------------------------------------------------ hits: records -> reference positions
 * Expands SMEM records into capped occurrence positions in per-sequence coordinates: ExactMatch.exact_match /
 * get_positions (ExactMatch.py:174-199) and the positions LUT.lut stores per k-mer (LUT.py:33-35), for a whole batch.
 *
 * Record r = {read_id, qstart, qend, lo, hi}: cnt = hi - lo + 1, len = qend - qstart.  n_hits(r) = 0 if len < min_len,
 * else min(cnt, max_occ) (max_occ == 0: no cap).  Hit k (0 <= k < n_hits) is row lo + k * step, step = cnt / max_occ
 * when cnt > max_occ, else 1 (BWA's mem_collect_seeds rule: hits in suffix-array row order).  Its 0-based text position
 * p = suffix_array[row] - 1 lies in sequence c = upper_bound(start, p) - 1 at offset p - start[c].
 *
 * The reference is the concatenation of n sequences; start (device, n + 1 entries, non-decreasing, start[0] = 0,
 * start[n] = n_bases; empty sequences allowed) gives where each begins.  A NULL gsm_dev_contigs = one sequence. */
typedef struct {
    uint64_t n;             /* sequences */
    const uint32_t* start;  /* device, n + 1 entries */
} gsm_dev_contigs;

#define GSM_HIT_SPANS 1u   /* offset + len > length of the sequence: the match runs into the next sequence */
#define GSM_HIT_SAMPLED 2u /* cnt > max_occ: the hits are an evenly spaced sample of the interval */

typedef struct {
    uint32_t record; /* index of the record in the array passed in */
    uint32_t contig;
    uint32_t offset; /* 0-based, in the sequence */
    uint32_t flags;  /* GSM_HIT_* */
} gsm_hit;

/* Bytes of device scratch gsm_hits_count needs for n_recs records (host arithmetic, no device needed). */
int gsm_hits_workspace_info(uint64_t n_recs, uint64_t* scan_tmp_bytes);

/* Phase 1: counts_u32[r] = n_hits(r) and hit_off_u64 (n_recs + 1 entries) = their exclusive scan, hit_off_u64[n_recs] =
 * the total.  recs, counts_u32, hit_off_u64 and scan_tmp are device memory.  Asynchronous on stream. */
int gsm_hits_count(const gsm_record* recs, uint64_t n_recs, uint32_t max_occ, uint32_t min_len, uint32_t* counts_u32,
                   uint64_t* hit_off_u64, void* scan_tmp, uint64_t scan_tmp_bytes, void* stream);

/* Phase 2: the hits of records [rec_begin, rec_end), hit h at out[h - hit_off[rec_begin]] (device, out_cap entries).
 * Positions come from idx->sa when it is set, else from ssa (gsm_sa_sample_build, every `sample`-th row) by LF walks; with
 * neither, GSM_E_INVALID.  max_occ / min_len must be those given to gsm_hits_count.  Nothing is written at or past out_cap;
 * if the range holds more hits, bit 0 of *status8 (device uint64) is set.  Asynchronous on stream. */
int gsm_hits_locate(const gsm_dev_index* idx, const uint32_t* ssa, uint32_t sample, const gsm_dev_contigs* contigs,
                    const gsm_record* recs, const uint64_t* hit_off, uint64_t rec_begin, uint64_t rec_end, uint32_t max_occ,
                    uint32_t min_len, gsm_hit* out, uint64_t out_cap, uint64_t* status8, void* stream);

/* ------------------------------------------------------------------ chains: located hits -> co-linear seed chains
 * BWA-MEM's mem_chain (test_and_merge, mem_chain_weight) per SLOT: slot s = read s of the batch, or with a strand-doubled
 * batch read s >> 1 on strand s & 1.  The records of slot s are recs[rec_off[s] .. rec_off[s+1]) (the engine's rec_off),
 * the hits of record r are hits[hit_off[r] .. hit_off[r+1]) (gsm_hits_count / gsm_hits_locate).  The slot's seeds are its
 * hits in record order, then hit order; the seed of hit h of record r is qbeg = r.qstart, len = r.qend - r.qstart,
 * rbeg = h.offset on sequence h.contig.  A hit flagged GSM_HIT_SPANS is skipped (BWA's rid < 0).
 *
 * The slot's chains are ordered by (contig, pos), pos = rbeg of the first seed; each seed is tested against `lower`, the
 * chain with the largest key <= (contig, rbeg) -- the one created first when several share it -- by BWA's test_and_merge
 * with 64-bit signed differences: contained (qbeg >= first.qbeg, qbeg + len <= last.qbeg + last.len, and the same on the
 * reference) -> not appended; appended if y = rbeg - last.rbeg >= 0, |x - y| <= w (x = qbeg - last.qbeg),
 * x - last.len < max_gap and y - last.len < max_gap; otherwise, or without `lower`, the seed starts a new chain.  BWA's
 * defaults: w = 100 (-w), max_gap = 10000 (max_chain_gap).
 *
 * Output: the chains of every slot in slot order, within a slot in (contig, pos) order with ties in creation order; a chain's
 * id is its index within its slot in that order.  hit_chain[h] = id of the chain hit h was appended to, GSM_CHAIN_CONTAINED |
 * id when contained, GSM_CHAIN_NONE for a spanning hit. */
#define GSM_CHAIN_NONE 0xFFFFFFFFu
#define GSM_CHAIN_CONTAINED 0x80000000u

typedef struct {
    uint32_t slot;     /* slot in the batch (not the read id) */
    uint32_t contig;
    uint32_t rbeg;     /* rbeg of the first seed */
    uint32_t rend;     /* max rbeg + len over the member seeds */
    uint32_t q;        /* qbeg | qend << 16: min qbeg, max qend over the members; reverse-complement coordinates on a strand-1 slot */
    uint32_t weight;   /* mem_chain_weight: min(non-overlapping query coverage, non-overlapping reference coverage) */
    uint32_t n_seeds;  /* member seeds (contained seeds are not members) */
    uint32_t reserved; /* 0 */
} gsm_chain;

/* Bytes of device workspace for n_slots slots over a hits array of n_hits entries (host arithmetic, no device needed):
 * 84 bytes per hit (a slot's scratch sits at its first hit) plus a few bytes per slot. */
int gsm_chains_workspace_info(uint64_t n_slots, uint64_t n_hits, uint64_t* bytes);

/* Phase 1: chain every slot.  hit_chain (n_hits u32) receives the ids, chain_cnt (n_slots u32) the chains per slot and
 * chain_off (n_slots + 1 u64) their exclusive scan, chain_off[n_slots] = the total.  All pointers are device memory; the
 * workspace is the caller's (gsm_chains_workspace_info) and must be passed unchanged to phase 2.  GSM_E_CAPACITY for a
 * short workspace.  Asynchronous on stream. */
int gsm_chain_seeds(const gsm_record* recs, const uint64_t* rec_off, uint64_t n_slots, const gsm_hit* hits, const uint64_t* hit_off,
                    uint64_t n_hits, uint32_t w, uint32_t max_gap, uint32_t* hit_chain, uint32_t* chain_cnt, uint64_t* chain_off,
                    void* workspace, uint64_t workspace_bytes, void* stream);

/* Phase 2: chain k of the batch to out[k] (device, out_cap entries).  Nothing is written at or past out_cap; if the batch
 * holds more chains, bit 0 of *status8 (device uint64) is set.  Asynchronous on stream. */
int gsm_chains_collect(const uint64_t* rec_off, uint64_t n_slots, const uint64_t* hit_off, uint64_t n_hits, const uint64_t* chain_off,
                       const void* workspace, uint64_t workspace_bytes, gsm_chain* out, uint64_t out_cap, uint64_t* status8, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GENIE_SMEM_H */
