// Per-hit arithmetic of the hit expansion (hits.cu), shared with the host-compiled test (tests/test_hits_host.py).
//
// A record {read_id, qstart, qend, sa_lo, sa_hi} with cnt = sa_hi - sa_lo + 1 rows and len = qend - qstart bases expands
// into n = min(cnt, max_occ) hits (0 when len < min_len; max_occ == 0 = no cap).  Hit k sits at row lo + k * step with
// step = cnt / max_occ when cnt > max_occ, else 1: BWA's mem_collect_seeds rule, so hits come in suffix-array row order.
// Its position p = SA[row] - 1 is placed with the sequence table start[0..n] (start[n] = n_bases, empty sequences allowed):
// sequence c = upper_bound(start, p) - 1, offset p - start[c].
#pragma once
#include <stdint.h>

#include "fm_core.cuh"

namespace gsm {

constexpr uint32_t HIT_SPANS = 1u;     // GSM_HIT_SPANS: the match runs past the end of its sequence
constexpr uint32_t HIT_SAMPLED = 2u;   // GSM_HIT_SAMPLED: the interval had more rows than max_occ

// rows of [lo, hi]; 0 for an inverted interval
GSM_HD uint32_t hit_rows(uint32_t lo, uint32_t hi) { return hi >= lo ? hi - lo + 1u : 0u; }

// len = qend - qstart of a record's second word (qstart | qend << 16); 0 for an inverted range
GSM_HD uint32_t hit_len(uint32_t y) {
    const uint32_t qs = y & 0xFFFFu, qe = y >> 16;
    return qe > qs ? qe - qs : 0u;
}

GSM_HD bool hit_sampled(uint32_t cnt, uint32_t max_occ) { return max_occ != 0u && cnt > max_occ; }

GSM_HD uint32_t hit_count(uint32_t cnt, uint32_t len, uint32_t max_occ, uint32_t min_len) {
    if (len < min_len) return 0u;
    return hit_sampled(cnt, max_occ) ? max_occ : cnt;
}

GSM_HD uint32_t hit_step(uint32_t cnt, uint32_t max_occ) { return hit_sampled(cnt, max_occ) ? cnt / max_occ : 1u; }

// row of hit k: lo + k * step < lo + cnt, so it never leaves the interval
GSM_HD uint32_t hit_row(uint32_t lo, uint32_t k, uint32_t step) { return lo + (uint32_t)((uint64_t)k * step); }

// first i in [0, n_entries) with start(i) > p, minus one: the sequence holding text position p (start(0) == 0 <= p)
template <typename LoadStart>
GSM_HD uint32_t contig_of(LoadStart start, uint32_t n_entries, uint32_t p) {
    uint32_t lo = 0u, hi = n_entries;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (start(mid) <= p) lo = mid + 1u;
        else hi = mid;
    }
    return lo - 1u;
}

// The hit record {record, contig, offset, flags} of text position p (0-based) for a match of len bases.
template <typename LoadStart>
GSM_HD U4 make_hit(LoadStart start, uint32_t n_entries, uint32_t record, uint32_t p, uint32_t len, bool sampled) {
    const uint32_t c = contig_of(start, n_entries, p);
    const uint32_t s = start(c), off = p - s;
    U4 h;
    h.x = record;
    h.y = c;
    h.z = off;
    h.w = ((uint64_t)off + len > (uint64_t)(start(c + 1u) - s) ? HIT_SPANS : 0u) | (sampled ? HIT_SAMPLED : 0u);
    return h;
}

}  // namespace gsm
