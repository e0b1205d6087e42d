// Per-read control of the SMEM sweep kernel, written once for device and for the host-compiled
// logic test (tests/emu).  It enumerates ALL maximal exact matches of a read with a bidirectional
// FM index, the way the reference's forward_extension / backward_extension pair
// (SMEM/SMEM.py:425-443, 389-423) would if each extension cost one FM step instead of a full
// restart of exact_match_back_prop, and if the first K steps of an extension were one table fetch
// (the reference's own LUT idea, SMEM/LUT.py:15-35, applied to both directions):
//
//   sweep(x):  SEEDF one fetch from the seed table gives the intervals of q[x:x+K) on both indexes
//                    (absent k-mer or read end closer than K: plain stepping from one base).
//              FWD   append q[x+K], ... on the reverse-text index while q[x:j] still occurs
//                    (SMEM.py:431-440); remember (j, interval) whenever the occurrence count is
//                    about to change: only those ends can be right-maximal.  Ends j < x+K are not
//                    materialised ("short" candidates): most sweeps never need them.
//              WALK  prepend q[x-1], q[x-2], ... to the LONGEST candidate until it dies
//                    (SMEM.py:396-416): its start s is LS[F(x)].  Every other candidate j has
//                    lb <= LS[j] <= s, where lb = (previous sweep's start) + 1 because that
//                    sweep's forward extension ended exactly at x.  If s == lb they all share
//                    LS = s and none of them is maximal: the sweep is over after the minimum
//                    possible number of steps (the common case inside an exact stretch); a walk
//                    that reaches lb stops there without the failing step.
//              SEQ   otherwise every remaining candidate end j, longest first, gets its own walk:
//                    stored candidates continue from their interval at x-1; short candidates start
//                    from the seed-table entry of q[j-K:j) (SEEDB, one fetch replaces K steps on
//                    wide intervals) or, if that k-mer is absent / would start left of lb, from a
//                    plain backward search at j.  LS is non-decreasing in j, so (LS[j], j) is
//                    maximal iff LS[j] is smaller than the last emitted start, and the first walk
//                    that reaches lb ends the sweep.
//              x = F(x) = end of the longest forward match; repeat until x == L.
//
// With LS[j] = leftmost start of a match ending at j (SURVEY Appendix B) the emitted set is
// {(LS[j], j) : j = L or LS[j+1] > LS[j]}; it determines LS[] and F() completely, and the three
// reference entry points are integer selections over it (select_logic.cuh).
//
// One next()/consume() pair = one FM extension step (at most two bucket fetches) or one seed-table
// fetch.  The pending operation's operands live in registers (P0, cnt, ch), so the top of the
// kernel loop is uniform.
#pragma once
#include "fm_core.cuh"

namespace gsm {

struct IndexMeta {
    uint32_t C[4];      // first row per leading base
    uint32_t cnt[4];    // occurrences per base
    uint32_t prim_f, prim_r;
    uint32_t n_rows;
};

// A maximal-match record as staged per read: 16 bytes.
//   se = start | end << 16, lo = SA lo, cnt = SA count, sweep = sweep ordinal
struct MemEntry {
    uint32_t se, lo, cnt, sweep;
};

// One entry of the seed table (gsm_seed_table_build): the k-mer's rows on the text index, its count, and
// the rows of the reversed k-mer on the reversed-text index.
struct SeedEntry {
    uint32_t fwd_lo, cnt, rev_lo, pad;
};

enum SweepMode : int { M_FETCH = 0, M_FWD = 1, M_WALK = 2, M_SEEDF = 3, M_SEEDB = 4, M_DONE = 5,
                       // unique-match shortcut (needs suffix array, inverse suffix array and packed text; see Ctx::uniq):
                       M_SAF = 6,    // fetch suffix_array[k]: where in the text the unique occurrence of q[x:pos) starts (FWD)
                       M_SAW = 7,    // the same for the longest candidate when the forward phase never needed it (first WALK)
                       M_CMPF = 8,   // compare q[pos..) with the text behind the occurrence, up to SWEEP_CMP_CHUNK bases per fetch
                       M_CMPB = 9,   // compare q[..pos) with the text in front of the occurrence
                       M_ISA = 10 }; // fetch inverse_suffix_array[text position]: the row of the extended match

constexpr uint32_t SWEEP_CMP_CHUNK = 64;   // bases compared per text fetch

// Ctx must provide:
//   bool     fetch(uint32_t& rid, uint32_t& L)          next read (loads its bases), false when none
//   uint32_t base(uint32_t pos)                         2-bit base of the current read
//   uint32_t seed_k()                                   K of the seed table, 0 = no table
//   bool     uniq()                                     unique-match shortcut available: once q[x:pos) occurs exactly once
//                                                       the forward extension follows the TEXT (one suffix-array fetch, then
//                                                       64 bases per compare) instead of one FM step per base.  k_sweep1
//                                                       runs it when the suffix array and the text are on the device.
//   bool     uniq_back()                                also walk unique matches to the LEFT along the text (needs the inverse
//                                                       suffix array; host-compiled test only)
//   uint32_t kmer(uint32_t pos)                         code of q[pos:pos+K) (LUT.convert_seq_to_num, LUT.py:37-48)
//   void     cand_put(uint32_t i, uint32_t j, uint32_t lo, uint32_t cnt)
//   void     cand_get(uint32_t i, uint32_t& j, uint32_t& lo, uint32_t& cnt)
//   void     cand_sync()                                make candidate writes visible to the read's other lanes, if any
//   void     emit(uint32_t idx, MemEntry e)             stage maximal match #idx of this read
//   void     finish(uint32_t rid, uint32_t n_mems)      read complete
// BWA-SMEM selection (get_SMEMS, SMEM.py:456-467 = Selector::run_bwa) as a MAXIMUM over the ordered match list: standing at
// read position p the pick is the entry with the largest key -- entries ending at or before p are out (key 0); an entry
// covering p beats every entry that starts beyond it, the longer one wins, ties go to the earlier entry; if nothing covers
// p the first entry beyond it is taken (what covering_best returns then).  k = position in the ordered list (< 64),
// lengths < 2^16.  The sweep's hand-over reduces these keys over the lanes of a warp (flush_finished), one pick per
// reduction, then continues from the pick's end; tests/emu compares the same loop with Selector::run_bwa.
GSM_HD uint32_t bwa_pick_key(uint32_t start, uint32_t end, uint32_t k, uint32_t p) {
    if (end <= p) return 0u;
    return (start <= p ? 0x80000000u | ((end - start) << 6) : 0u) | (63u - k);
}
GSM_HD uint32_t bwa_pick_of(uint32_t key) { return 63u - (key & 63u); }

template <typename Ctx>
struct Sweeper {
    int mode = M_FETCH;
    uint32_t rid = 0, L = 0;
    uint32_t x = 0, F = 0, lb = 0;
    uint32_t n_mems = 0, sweep_id = 0;
    // pending FM step: rows [P0, P0 + cnt) extended by base ch (FWD: on the reverse-text index);
    // pending seed fetch (M_SEEDF / M_SEEDB): P0 holds the k-mer code
    uint32_t P0 = 0, cnt = 0, ch = 0;
    uint32_t k = 0;            // FWD: rows of q[x:pos) on the text index start here
    uint32_t pos = 0;          // FWD: next base to append; WALK: base being prepended
    uint32_t cur_j = 0;        // WALK: end of the candidate being extended
    uint32_t ncand = 0;        // stored candidates (ends >= x + K when the sweep was seeded)
    uint32_t short_hi = 0;     // short candidates still to walk: ends x+1 .. short_hi (none if <= x)
    uint32_t last_start = 0;
    // Unique-match shortcut.  Once q[x:pos) occurs exactly ONCE, every further extension is decided by the text itself:
    // one suffix-array fetch locates the occurrence (tpos = text index of q[x]), then SWEEP_CMP_CHUNK bases are compared
    // per text fetch instead of one FM step per base; the row of a match extended to the left is one inverse-suffix-array
    // fetch.  Same results by construction: a unique occurrence extends exactly as far as the text around it agrees.
    uint32_t tpos = 0, have_tpos = 0;
    uint32_t aux = 0;          // index of the pending suffix-array / inverse-suffix-array fetch

    GSM_HD bool pending_step() const { return mode == M_FWD || mode == M_WALK; }
    GSM_HD bool pending_seed() const { return mode == M_SEEDF || mode == M_SEEDB; }
    GSM_HD bool pending_word() const { return mode == M_SAF || mode == M_SAW || mode == M_ISA; }
    GSM_HD bool pending_cmp() const { return mode == M_CMPF || mode == M_CMPB; }
    GSM_HD bool on_reverse() const { return mode == M_FWD; }
    // operands of the pending text comparison.  Forward: text[cmp_text() + i] against q[cmp_read() + i]; backward:
    // text[cmp_text() - 1 - i] against q[cmp_read() - 1 - i]; i < min(cmp_max(n_bases), SWEEP_CMP_CHUNK).
    GSM_HD uint32_t cmp_text() const { return mode == M_CMPF ? tpos + (pos - x) : tpos - (x - pos); }
    GSM_HD uint32_t cmp_read() const { return pos; }
    GSM_HD uint32_t cmp_max(uint32_t n_bases) const {
        const uint32_t t = cmp_text();
        const uint32_t a = mode == M_CMPF ? L - pos : pos - lb;
        const uint32_t b = mode == M_CMPF ? n_bases - t : t;
        return a < b ? a : b;
    }

    GSM_HD void emit_match(Ctx& c, uint32_t start, uint32_t end, uint32_t lo, uint32_t n) {
        MemEntry e;
        e.se = start | (end << 16);
        e.lo = lo; e.cnt = n; e.sweep = sweep_id;
        c.emit(n_mems++, e);
        last_start = start;
    }

    // mode M_FETCH doubles as "needs a transition": x >= L means no read is in progress.
    GSM_HD void end_sweep(Ctx& c) {
        lb = x + 1; x = F; sweep_id++;
        mode = M_FETCH;
        if (x >= L) c.finish(rid, n_mems);
    }

    // Start the sweep at x (a read is in progress, x < L).  Leaves a pending operation, or mode == M_FETCH.
    GSM_HD void start_sweep(Ctx& c, const IndexMeta& m) {
        const uint32_t b = c.base(x);
        ncand = 0; short_hi = 0; have_tpos = 0;
        if (m.cnt[b] == 0) {              // base absent from the text (outside the reference's domain): skip it
            lb = x + 1; x++; sweep_id++;
            if (x >= L) c.finish(rid, n_mems);
            return;                       // mode stays M_FETCH
        }
        const uint32_t K = c.seed_k();
        if (K != 0 && x + K <= L) { P0 = c.kmer(x); mode = M_SEEDF; return; }
        fwd_plain(c, m);
    }

    GSM_HD void fwd_plain(Ctx& c, const IndexMeta& m) {
        const uint32_t b = c.base(x);
        k = m.C[b]; P0 = m.C[b]; cnt = m.cnt[b];
        pos = x + 1;
        fwd_continue(c, m);
    }

    // (k, P0, cnt) describe q[x:pos): append q[pos], or close the forward phase at the read end.  A unique occurrence
    // is followed in the text instead (M_SAF -> M_CMPF).
    GSM_HD void fwd_continue(Ctx& c, const IndexMeta& m) {
        if (pos < L) {
            if (cnt == 1u && c.uniq()) { aux = k; mode = M_SAF; return; }
            ch = c.base(pos); mode = M_FWD;
            return;
        }
        c.cand_put(ncand++, pos, k, cnt);
        start_bwd(c, m);
    }

    // forward comparison finished (or impossible): q[x:pos) is the longest forward match
    GSM_HD void uniq_fwd_done(Ctx& c, const IndexMeta& m) {
        c.cand_put(ncand++, pos, k, 1u);
        start_bwd(c, m);
    }
    // q[pos:cur_j) is matched at text index tpos - (x - pos): compare further left, or finish
    GSM_HD void uniq_walk_next(Ctx& c, const IndexMeta& m) {
        mode = M_CMPB;
        if (cmp_max(m.n_rows - 1u) != 0u) return;
        uniq_walk_done(c, m);
    }
    GSM_HD void uniq_walk_done(Ctx& c, const IndexMeta& m) {
        if (pos == x) { walk_end(c, m, x); return; }            // no extension: the interval of the candidate stands
        aux = tpos - (x - pos);                                 // the extended match starts here in the text
        mode = M_ISA;
    }

    // result of the pending suffix-array / inverse-suffix-array fetch
    GSM_HD void consume_word(Ctx& c, const IndexMeta& m, uint32_t v) {
        if (mode == M_ISA) { P0 = v; cnt = 1u; walk_end(c, m, pos); return; }
        tpos = v - 1u;                                          // suffix-array values are 1-based (ExactMatch.py:66)
        have_tpos = 1u;
        if (mode == M_SAF) {
            mode = M_CMPF;
            if (cmp_max(m.n_rows - 1u) == 0u) uniq_fwd_done(c, m);
            return;
        }
        uniq_walk_next(c, m);                                   // M_SAW
    }

    // result of the pending text comparison: `matched` bases agree (already capped by cmp_max and the chunk size)
    GSM_HD void consume_cmp(Ctx& c, const IndexMeta& m, uint32_t matched) {
        if (mode == M_CMPF) {
            pos += matched;
            if (matched == SWEEP_CMP_CHUNK && cmp_max(m.n_rows - 1u) != 0u) return;     // a whole chunk agreed: next chunk
            uniq_fwd_done(c, m);
            return;
        }
        pos -= matched;
        if (matched == SWEEP_CMP_CHUNK && cmp_max(m.n_rows - 1u) != 0u) return;
        uniq_walk_done(c, m);
    }

    // Forward phase over: pop the longest candidate and walk it left.
    GSM_HD void start_bwd(Ctx& c, const IndexMeta& m) {
        c.cand_sync();
        ncand--;
        c.cand_get(ncand, cur_j, P0, cnt);
        F = cur_j;
        last_start = 0xFFFFFFFFu;
        if (x == 0) {                       // nothing to prepend: every candidate starts at 0, the longest wins
            emit_match(c, 0, cur_j, P0, cnt);
            end_sweep(c);
            return;
        }
        if (cnt == 1u && x != lb && c.uniq() && c.uniq_back()) {      // unique occurrence: extend it to the left along the text
            pos = x;
            if (have_tpos) uniq_walk_next(c, m);
            else { aux = P0; mode = M_SAW; }
            return;
        }
        walk_from(c, m, x);
    }

    // (P0, cnt) is the interval of q[start:cur_j): set up the step prepending q[start-1].  False if start is
    // already the lower bound (no match ending beyond x starts left of lb) or the left end of the read.
    GSM_HD bool try_walk(Ctx& c, uint32_t start) {
        if (start == lb || start == 0) return false;
        pos = start - 1;
        ch = c.base(pos);
        mode = M_WALK;
        return true;
    }

    GSM_HD void walk_from(Ctx& c, const IndexMeta& m, uint32_t start) {
        if (!try_walk(c, start)) walk_end(c, m, start);
    }

    // The walked candidate (cur_j, P0, cnt) cannot be extended beyond `start`: it is maximal iff it reaches further
    // left than every longer candidate did.  A walk that stops at lb settles all the shorter candidates too.
    // Then the next candidate (stored ones first, longest first; then the short ends) is set up.
    GSM_HD void walk_end(Ctx& c, const IndexMeta& m, uint32_t start) {
        for (;;) {
            if (start < last_start) emit_match(c, start, cur_j, P0, cnt);
            if (start == lb || (ncand == 0 && short_hi <= x)) { end_sweep(c); return; }
            if (ncand != 0) {                   // stored candidate: continue from its interval at x
                ncand--;
                c.cand_get(ncand, cur_j, P0, cnt);
                start = x;
            } else {                            // short candidate: end in (x, x + K)
                cur_j = short_hi--;
                const uint32_t K = c.seed_k();
                if (cur_j >= K && cur_j - K >= lb) { P0 = c.kmer(cur_j - K); mode = M_SEEDB; return; }
                start = plain_begin(c, m);
            }
            if (try_walk(c, start)) return;
        }
    }

    // backward search of q[..cur_j) from scratch; q[x:cur_j) occurs, so its last base does
    GSM_HD uint32_t plain_begin(Ctx& c, const IndexMeta& m) {
        const uint32_t b = c.base(cur_j - 1);
        P0 = m.C[b]; cnt = m.cnt[b];
        return cur_j - 1;
    }

    // Bring this pair to its next pending operation.  Returns false only when there are no more reads.
    GSM_HD bool next(Ctx& c, const IndexMeta& m) {
        while (mode == M_FETCH) {
            if (x >= L) {                   // no read in progress (initial state: x == L == 0)
                if (!c.fetch(rid, L)) { mode = M_DONE; return false; }
                n_mems = 0; sweep_id = 0; x = 0; lb = 0;
                if (L == 0) { c.finish(rid, 0); continue; }
            }
            start_sweep(c, m);
        }
        return mode != M_DONE;
    }

    // result of the pending seed-table fetch
    GSM_HD void consume_seed(Ctx& c, const IndexMeta& m, const SeedEntry& e) {
        if (mode == M_SEEDF) {
            if (e.cnt == 0) { fwd_plain(c, m); return; }          // q[x:x+K) does not occur: F(x) < x + K
            k = e.fwd_lo; P0 = e.rev_lo; cnt = e.cnt;
            pos = x + c.seed_k();
            short_hi = pos - 1;
            fwd_continue(c, m);
            return;
        }
        // M_SEEDB: seed of the short candidate ending at cur_j
        if (e.cnt == 0) { walk_from(c, m, plain_begin(c, m)); return; }
        P0 = e.fwd_lo; cnt = e.cnt;
        walk_from(c, m, cur_j - c.seed_k());
    }

    // result of the pending FM step
    GSM_HD void consume(Ctx& c, const IndexMeta& m, const StepOut& r) {
        // FWD (append q[pos] to q[x:pos)) and WALK (prepend q[pos] to q[pos+1:cur_j)) share one hot path:
        // take the new interval, move one base, fetch it.  Only the ends of an extension branch.
        const bool fwd = mode == M_FWD;
        if (fwd && r.cnt_new != cnt) c.cand_put(ncand++, pos, k, cnt);     // count about to change: q[x:pos) is a candidate
        if (r.cnt_new != 0) {
            k += r.lt_add; P0 = r.lo_new; cnt = r.cnt_new;
            // one site for both directions: FWD and WALK lanes of a warp fetch their next base together
            const bool more = fwd ? (pos + 1u != L) : (pos != lb && pos != 0u);
            if (more && !(fwd && cnt == 1u && c.uniq())) { pos += fwd ? 1u : 0xFFFFFFFFu; ch = c.base(pos); return; }
            if (fwd) {
                pos++;
                fwd_continue(c, m);                                        // read end, or unique: follow the text
                return;
            }
            walk_end(c, m, pos);                                           // reached the lower bound (or the left end)
            return;
        }
        if (fwd) start_bwd(c, m);
        else walk_end(c, m, pos + 1u);
    }
};

}  // namespace gsm
