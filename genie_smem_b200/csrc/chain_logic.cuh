// Per-seed rule of the seed chaining (chains.cu), shared with the host-compiled test (tests/test_chains_host.py).
//
// BWA-MEM's mem_chain, per slot: seeds (the slot's hits in record order, then in hit order) are visited one by one.  The
// slot's chains are kept ordered by (contig, pos), pos = rbeg of the chain's first seed; `lower` is the chain with the
// largest key <= (seed.contig, seed.rbeg), the one created first among chains sharing that key.  test_and_merge (literal,
// 64-bit signed differences) either finds the seed contained in `lower` (not appended), appends it, or fails; a failed
// merge or a missing `lower` starts a new chain.  mem_chain_weight is kept incrementally: the non-overlapping query and
// reference coverage of the members in member order, each with the running end of its loop.
#pragma once
#include <stdint.h>

#include "fm_core.cuh"

namespace gsm {

constexpr uint32_t CHAIN_NONE = 0xFFFFFFFFu;        // GSM_CHAIN_NONE: a spanning hit, in no chain
constexpr uint32_t CHAIN_CONTAINED = 0x80000000u;   // GSM_CHAIN_CONTAINED: contained in the chain, not a member
constexpr uint32_t CHAIN_FULL = 0x7FFFFFFFu;        // chain_step: the seed needs a new chain and the table is at capacity

struct ChainSeed {
    uint32_t qbeg, len, rbeg, contig;
};

// One chain while its slot is chained: 12 words.
struct ChainState {
    uint32_t contig, pos;    // key; pos = rbeg of the first seed
    uint32_t fq;             // qbeg of the first seed
    uint32_t lq, lr, ll;     // qbeg, rbeg, len of the last member
    uint32_t qmin, qe, re;   // min qbeg, max qbeg + len, max rbeg + len over the members (qe, re: mem_chain_weight's `end`s)
    uint32_t wq, wr, n;      // non-overlapping query / reference coverage, members
};
constexpr int CHAIN_STATE_WORDS = 12;

// ChainState <-> 12 words, word f through ld(f) / st(f, v) (shared or global tables)
template <typename Ld>
GSM_HD ChainState chain_load(Ld ld) {
    ChainState c;
    c.contig = ld(0); c.pos = ld(1); c.fq = ld(2); c.lq = ld(3); c.lr = ld(4); c.ll = ld(5);
    c.qmin = ld(6); c.qe = ld(7); c.re = ld(8); c.wq = ld(9); c.wr = ld(10); c.n = ld(11);
    return c;
}

template <typename St>
GSM_HD void chain_store(const ChainState& c, St st) {
    st(0, c.contig); st(1, c.pos); st(2, c.fq); st(3, c.lq); st(4, c.lr); st(5, c.ll);
    st(6, c.qmin); st(7, c.qe); st(8, c.re); st(9, c.wq); st(10, c.wr); st(11, c.n);
}

GSM_HD uint64_t chain_key(uint32_t contig, uint32_t pos) { return (uint64_t)contig << 32 | pos; }

// mem_chain_weight's two loops, one member further
GSM_HD void chain_add_member(ChainState& c, const ChainSeed& s) {
    const uint32_t qend = s.qbeg + s.len, rend = s.rbeg + s.len;
    if (s.qbeg >= c.qe) c.wq += s.len;
    else if (qend > c.qe) c.wq += qend - c.qe;
    if (s.rbeg >= c.re) c.wr += s.len;
    else if (rend > c.re) c.wr += rend - c.re;
    c.qe = c.qe > qend ? c.qe : qend;
    c.re = c.re > rend ? c.re : rend;
    c.qmin = c.qmin < s.qbeg ? c.qmin : s.qbeg;
    c.lq = s.qbeg;
    c.lr = s.rbeg;
    c.ll = s.len;
    ++c.n;
}

GSM_HD ChainState chain_new(const ChainSeed& s) {
    ChainState c;
    c.contig = s.contig;
    c.pos = s.rbeg;
    c.fq = c.qmin = s.qbeg;
    c.lq = c.lr = c.ll = 0u;
    c.qe = c.re = c.wq = c.wr = c.n = 0u;
    chain_add_member(c, s);
    return c;
}

enum { CHAIN_MERGE_FAIL = 0, CHAIN_MERGE_CONTAINED = 1, CHAIN_MERGE_APPENDED = 2 };

// BWA's test_and_merge without the forward / reverse strand test (hits are on the forward strand)
GSM_HD int chain_test_and_merge(ChainState& c, const ChainSeed& s, uint32_t w, uint32_t max_gap) {
    if (s.contig != c.contig) return CHAIN_MERGE_FAIL;
    const int64_t qb = s.qbeg, rb = s.rbeg, ln = s.len, lq = c.lq, lr = c.lr, ll = c.ll;
    if (qb >= (int64_t)c.fq && qb + ln <= lq + ll && rb >= (int64_t)c.pos && rb + ln <= lr + ll) return CHAIN_MERGE_CONTAINED;
    const int64_t x = qb - lq, y = rb - lr;
    if (y >= 0 && x - y <= (int64_t)w && y - x <= (int64_t)w && x - ll < (int64_t)max_gap && y - ll < (int64_t)max_gap) {
        chain_add_member(c, s);
        return CHAIN_MERGE_APPENDED;
    }
    return CHAIN_MERGE_FAIL;
}

// First sorted position in [0, n) whose key is > k (upper) or >= k (!upper); key(i) = key at sorted position i.
template <typename Key>
GSM_HD uint32_t chain_bound(Key key, uint32_t n, uint64_t k, bool upper) {
    uint32_t lo = 0u, hi = n;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        const uint64_t v = key(mid);
        if (upper ? v <= k : v < k) lo = mid + 1u;
        else hi = mid;
    }
    return lo;
}

// The output record (gsm_chain, 8 words) of a finished chain.
GSM_HD void chain_output(const ChainState& c, uint32_t slot, uint32_t out[8]) {
    const uint32_t w = c.wq < c.wr ? c.wq : c.wr;
    out[0] = slot;
    out[1] = c.contig;
    out[2] = c.pos;
    out[3] = c.re;
    out[4] = (c.qmin & 0xFFFFu) | (c.qe << 16);
    out[5] = w < (1u << 30) ? w : (1u << 30) - 1u;
    out[6] = c.n;
    out[7] = 0u;
}

// One seed of mem_chain against the ordered chain table t of its slot.  Tab provides n (chains), key(i) / id(i) at sorted
// position i, load(id) / store(id, state), and insert(i, state): the new chain gets id n (creation order) at sorted
// position i, after every chain of an equal key.  Returns the seed's chain id (creation order, | CHAIN_CONTAINED when
// contained), or CHAIN_FULL when the seed needs a new chain and the table already holds cap chains (t is unchanged).
template <typename Tab>
GSM_HD uint32_t chain_step(Tab& t, const ChainSeed& s, uint32_t w, uint32_t max_gap, uint32_t cap) {
    const uint32_t n = t.n;
    auto key = [t](uint32_t i) { return t.key(i); };          // a copy: keeps the table in registers
    const uint32_t up = chain_bound(key, n, chain_key(s.contig, s.rbeg), true);
    if (up > 0u) {
        const uint32_t lo = chain_bound(key, up - 1u, t.key(up - 1u), false);    // the first chain of the lower key
        const uint32_t id = t.id(lo);
        ChainState c = t.load(id);
        const int m = chain_test_and_merge(c, s, w, max_gap);
        if (m == CHAIN_MERGE_CONTAINED) return id | CHAIN_CONTAINED;
        if (m == CHAIN_MERGE_APPENDED) {
            t.store(id, c);
            return id;
        }
    }
    if (n >= cap) return CHAIN_FULL;
    t.insert(up, chain_new(s));
    return n;
}

}  // namespace gsm
