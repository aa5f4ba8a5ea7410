// CIR search: exact top-k of every query over a gallery shard, behind ofx_topk_search.
//
// Replaces the trainer / demo idiom  torch.cdist(Q, G) -> torch.topk(k, largest=False)
// (/root/reference/src/trains/trainers/complementary_item_retrieval_trainer.py:240-242,
//  src/demo/app.py:189-190), restated as the arg-max of  q.g - 0.5|g|^2  (or q.g).
//
// Pass 1 (tc_pipeline.cuh, tcgen05 / TMEM / TMA): bf16 Q x G^T tiles of 128 queries x 256
//   gallery rows; the epilogue thread that owns a query row scans the tile straight out of
//   TMEM and keeps that query's running top-K' in shared memory, so the score matrix never
//   reaches HBM.  Work is cut into units = (query block, gallery segment); a unit's list lives
//   on chip for the whole segment sweep and is flushed once.  A per-query global threshold
//   (the best "K'-th best" any finished unit has seen) lets later units reject almost every
//   score with one compare.
// Pass 2: per query, merge the units' lists by (score desc, index asc), re-score the K' best
//   in fp64 from the fp32 queries / gallery, rank by (-score, index), emit the top k.
#include <stdlib.h>

#include "common.h"
#include "tc_pipeline.cuh"

namespace ofx {

constexpr int kSearchBN = 256;
constexpr int kMaxSegments = 64;
// The L2 metric's per-row bias -0.5|g|^2 rides in the contraction itself: every packed gallery
// row carries one extra k-block of 64 bf16 whose first two entries are the bias split into
// bf16 hi + lo parts (16 mantissa bits, error ~1e-5 against ~1e-3 of bf16 score noise), and the
// bf16 copy of a query carries 1, 1 there (0, 0 for the dot metric).  One more k-block in 17
// (+6 % tensor work) removes the bias add -- 64 of the ~100 epilogue instructions per 32-column
// slab (32 shuffles + 32 adds) -- from an epilogue that was the kernel's bottleneck.
constexpr int kAugCols = 64;

// order-preserving float <-> uint32 map (for atomicMax on scores); 0 is below every float
__device__ __forceinline__ uint32_t enc_score(float f) {
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float dec_score(uint32_t e) {
    if (e == 0) return -INFINITY;
    return __uint_as_float((e & 0x80000000u) ? (e & 0x7FFFFFFFu) : ~e);
}
// smallest float strictly greater than x (x finite)
__device__ __forceinline__ float next_up(float x) {
    if (x == 0.f) return __uint_as_float(1u);
    const int b = __float_as_int(x);
    return __int_as_float(x > 0.f ? b + 1 : b - 1);
}

// ---------------------------------------------------------------------------------------
// Unit schedule.  Units u = seg * n_qblocks + qb, CTA c runs units c, c + P, c + 2P, ...
// Units of one segment share their gallery tiles, and all CTAs sweep a segment's tiles in the
// same order at the same pace, so every gallery tile is fetched from HBM once and then hit in
// L2 by the other query blocks.
// ---------------------------------------------------------------------------------------
struct SchedSearch {
    struct Params {
        int n_qgroups, n_tiles, seg_tiles, n_units, cl;
        int* progress; // [n_units] tile index each unit's producer has reached (-1 not started, huge = done), or null
    };
    static constexpr bool kPrefetch = true;
    static constexpr bool kThrottle = true;
    static constexpr int kPfDist = 8;   // query group 0 of every segment prefetches the tile kPfDist ahead into L2
    static constexpr int kWindow = 8;   // a unit may run at most kWindow tiles ahead of the slowest co-scheduled unit of its segment
    static constexpr int kCheck = 8;    // pacing check every kCheck tiles (power of two)
    // Pacing (producer thread only).  The query groups that sweep the same gallery segment share its tiles
    // through L2: whoever touches a tile first pulls it from HBM, the others hit.  Nothing keeps them together,
    // though, and measured at 10 M rows the main sweep read 316 GB from HBM for a 21.8 GB gallery (L2 hit rate
    // 72 %): the units drift further apart than L2 holds.  Every unit publishes the tile it has reached; every
    // kCheck-th tile a unit waits until it is at most kWindow tiles ahead of the slowest unit that was launched in
    // the same round of the same segment.  The slowest unit never waits, so this cannot deadlock.
    __device__ void throttle() {
        if (!p.progress) return;
        volatile int* pr = p.progress;
        if (rank == 0) pr[unit] = last ? 0x3fffffff : it;
        if ((it & (kCheck - 1)) != 0 || it == 0 || last) return;
        const int seg = unit / p.n_qgroups, round = unit / step;
        const int base = seg * p.n_qgroups;
        // bounded: pacing is an optimisation, never a correctness condition -- after ~20 ms of waiting the unit
        // simply goes on (a wedged peer must not be able to hang the sweep)
        for (int spins = 0; spins < (1 << 14); ++spins) {
            int mn = 0x7fffffff;
            if ((p.n_qgroups & 3) == 0) {      // 16-byte loads, all in flight before the first use
                int4 v[16];
                const int n4 = min(p.n_qgroups >> 2, 16);
#pragma unroll
                for (int j = 0; j < 16; ++j)
                    if (j < n4)
                        asm volatile("ld.volatile.global.v4.s32 {%0, %1, %2, %3}, [%4];"
                                     : "=r"(v[j].x), "=r"(v[j].y), "=r"(v[j].z), "=r"(v[j].w) : "l"(p.progress + base + 4 * j));
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    if (j < n4) {
                        const int e[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
#pragma unroll
                        for (int u = 0; u < 4; ++u)
                            if ((base + 4 * j + u) / step == round && e[u] >= 0 && e[u] < mn) mn = e[u];
                    }
                }
                for (int g = 64; g < p.n_qgroups; ++g) {
                    if ((base + g) / step != round) continue;
                    const int x = pr[base + g];
                    if (x >= 0 && x < mn) mn = x;
                }
            } else {
                for (int g = 0; g < p.n_qgroups; ++g) {
                    if ((base + g) / step != round) continue;
                    const int x = pr[base + g];
                    if (x >= 0 && x < mn) mn = x;
                }
            }
            if (it - mn <= kWindow) break;
            __nanosleep(200);
        }
    }
    int pf_n0;
    int m0, n0, unit, step, rank;
    int seg_lo, seg_len, it, qg;
    bool first, last;
    Params p;
    // With clusters (cl > 1) a unit belongs to a cluster: its cl CTAs take cl consecutive query
    // blocks (query group qg) and walk the same gallery tiles in the same order.
    __device__ SchedSearch(const Params& pp, int cta, int n_cta) : p(pp) {
        rank = cta % pp.cl;
        step = n_cta / pp.cl;
        unit = cta / pp.cl - step;
        it = 0;
        seg_lo = seg_len = qg = 0;
        m0 = n0 = 0;
        pf_n0 = -1;
        first = last = false;
    }
    // Every query group walks the segment in the same order; group 0 runs the L2 prefetch kPfDist
    // tiles ahead, so that the other groups (and group 0 itself) hit L2 and each gallery tile
    // crosses HBM once per segment sweep (33 GB instead of 43 GB of DRAM reads at 2 M rows against
    // a sweep that starts every query block at a different tile, +1.5 % throughput).
    // Prefetch leaders besides group 0 (DESIGN.md 4.2): the first unit of a round (its segment's
    // group 0 ran a round earlier), and, in the last kPfDist tiles of a unit, the CTA that leads
    // a segment in the next round pulls in that segment's first tiles.
    __device__ bool next() {
        if (it + 1 < seg_len) {
            ++it;
            first = false;
        } else {
            unit += step;
            if (unit >= p.n_units) return false;
            const int seg = unit / p.n_qgroups;
            qg = unit - seg * p.n_qgroups;
            m0 = (qg * p.cl + rank) * kBM;
            seg_lo = seg * p.seg_tiles;
            seg_len = min(p.n_tiles, seg_lo + p.seg_tiles) - seg_lo;
            it = 0;
            first = true;
        }
        last = it + 1 == seg_len;
        n0 = (seg_lo + it) * kSearchBN;
        const bool lead = qg == 0 || unit % step == 0;
        pf_n0 = (lead && it + kPfDist < seg_len) ? (seg_lo + it + kPfDist) * kSearchBN : -1;
        if (it + kPfDist >= seg_len && unit + step < p.n_units) {
            // nothing left to pull ahead in this segment: warm the first tiles of the segment this CTA
            // leads in the next round, so that round does not start on kPfDist cold tiles
            const int nu = unit + step, nseg = nu / p.n_qgroups;
            const int j = it + kPfDist - seg_len;
            if ((nu - nseg * p.n_qgroups == 0 || nu % step == 0) && nseg * p.seg_tiles + j < p.n_tiles)
                pf_n0 = (nseg * p.seg_tiles + j) * kSearchBN;
        }
        return true;
    }
    // query rows >= m_end and gallery rows >= n_end are not part of the unit (EpiTopK)
    __device__ __forceinline__ int m_end(int n_query) const { return n_query; }
    __device__ __forceinline__ long long n_end(long long n_rows) const { return n_rows; }
};

// ---------------------------------------------------------------------------------------
// Category schedule (ofx_category_search).  The shard's rows are sorted by category, so category c
// is the packed rows [seg_off[c], seg_off[c+1]); its queries are gathered into groups of cl
// consecutive 128-row query blocks.  A unit = (group of category c, tile range inside c's segment),
// read from the work list cat_plan_kernel writes on the device: {m0 = the group's first query row,
// m_end = end of c's live query rows, n_lo, n_hi = the range's packed rows}.  Tiles start at
// n_lo + 256 it (TMA takes any row coordinate, so segments need no padding) and the epilogue masks
// columns >= n_hi: no row of another category is ever admitted.  CTA c runs units c, c + P, ... as
// in SchedSearch; both CTAs of a pair take the same unit (same category, same tiles).
// ---------------------------------------------------------------------------------------
struct SchedCat {
    struct Params {
        const int4* units;    // [n_units] {m0, m_end, n_lo, n_hi}
        const int* n_units;   // written by cat_plan_kernel
        int cl;
    };
    static constexpr bool kPrefetch = false;
    static constexpr bool kThrottle = false;
    int m0, n0, unit, step, rank, it, n_it, total, n_lo, row_end, col_end;
    bool first, last;
    Params p;
    __device__ SchedCat(const Params& pp, int cta, int n_cta) : p(pp) {
        rank = cta % pp.cl;
        step = n_cta / pp.cl;
        unit = cta / pp.cl - step;
        it = n_it = 0;
        m0 = n0 = n_lo = row_end = col_end = 0;
        first = last = false;
        total = *pp.n_units;
    }
    __device__ bool next() {
        if (it + 1 < n_it) {
            ++it;
            first = false;
        } else {
            unit += step;
            if (unit >= total) return false;
            const int4 w = p.units[unit];
            m0 = w.x + rank * kBM;
            row_end = w.y;
            n_lo = w.z;
            col_end = w.w;
            n_it = (w.w - w.z + kSearchBN - 1) / kSearchBN;
            it = 0;
            first = true;
        }
        last = it + 1 == n_it;
        n0 = n_lo + it * kSearchBN;
        return true;
    }
    __device__ __forceinline__ int m_end(int) const { return row_end; }
    __device__ __forceinline__ long long n_end(long long) const { return col_end; }
};

struct SearchPlan {
    int n_qblocks, n_qgroups, cl, n_tiles, n_seg, seg_tiles, n_units, grid;
};

// Pick the segment count that minimises (rounds of units per CTA) x (tiles per unit).
static SearchPlan make_plan(long long n_rows, int n_query, int n_sm) {
    SearchPlan pl{};
    pl.n_qblocks = (n_query + kBM - 1) / kBM;
    pl.cl = pl.n_qblocks < 2 ? 1 : 2;   // CTA pairs; a single query block: nothing to pair
    pl.n_qgroups = (pl.n_qblocks + pl.cl - 1) / pl.cl;
    const int n_cta = n_sm / pl.cl;  // clusters that fit
    pl.n_tiles = static_cast<int>((n_rows + kSearchBN - 1) / kSearchBN);
    long long best = -1;
    for (int s = 1; s <= kMaxSegments && s <= pl.n_tiles; ++s) {
        const int len = (pl.n_tiles + s - 1) / s;
        const int segs = (pl.n_tiles + len - 1) / len;
        const long long rounds = (static_cast<long long>(pl.n_qgroups) * segs + n_cta - 1) / n_cta;
        const long long cost = rounds * len + rounds;  // + flush overhead per unit
        if (best < 0 || cost < best) {
            best = cost;
            pl.n_seg = segs;
            pl.seg_tiles = len;
        }
    }
    if (pl.n_tiles == 0) { pl.n_seg = 0; pl.seg_tiles = 1; }
    pl.n_units = pl.n_qgroups * pl.n_seg;
    pl.grid = (pl.n_units < n_cta ? pl.n_units : n_cta) * pl.cl;
    return pl;
}

// ---------------------------------------------------------------------------------------
// Counting bound shared by all units of a query.
// A unit's list only ever sees its own segment, so its admission gate settles at the kcap-th best of ~1/37 of the
// shard: every (query, segment) pair fills a list from scratch and about one score in a thousand still passes the
// gate -- half of all 32x32 slabs take the divergent insert path, and that, not the MMA, sets the pace of a short
// segment (1.25 M-row shard: tensor pipe 72 % busy, ~120 us lost per unit).  The rows of different segments are
// distinct rows, though: if c rows of the whole shard have been seen with a score >= T, the c-th best score of the
// shard is >= T, whichever units saw them.  So every admitted candidate is also counted (one RED) in a 64-bucket
// histogram of its query, buckets uniform over [lo, lo + 2.5 (top - lo)] with lo / top the kcap-th and the largest
// of the seeding block maxima, and every few tiles a thread reads its query's histogram and raises its gate to
//     min( T(kcap), T(k) - 2 eps )
// T(c) = lower edge of the bucket where the count from the top reaches c.  T(kcap) keeps the lists at the kcap
// best of the SHARD, and T(k) - 2 eps keeps the exactness certificate provable: T(k) <= the k-th best bf16 score
// Sb_k, the k rows above it have exact scores >= Sb_k - eps, hence T_out <= Sb_k - 2 eps < S_k - eps.
// HistQ = {lo, inv_w, w_safe, margin}: bucket(s) = trunc(fl(fl(s - lo) * inv_w)) clamped to [0, 63], and
// w_safe = (1 / inv_w)(1 - 2e-6) rounded down, so lo + j * w_safe (rounded down) is below every score that can
// land in bucket j or higher whatever the two roundings did.
// ---------------------------------------------------------------------------------------
constexpr int kHistBuckets = 64;
constexpr int kSeedSegments = 4;   // sample segments of the seeding sweep (pooled block maxima)
constexpr int kHistRefresh = 16;    // tiles between two reads of the histogram (power of two)

static __device__ __noinline__ float hist_bound(const uint32_t* __restrict__ h, const float4* __restrict__ hq, int m, int k) {
    const float4 q = __ldg(hq);
    unsigned cum = 0;
    int jm = -1, jk = -1;
    // two batches of eight 16-byte loads (all in flight together), upper half of the buckets first
    for (int half = 1; half >= 0 && jm < 0; --half) {
        uint4 v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = __ldcg(reinterpret_cast<const uint4*>(h) + half * 8 + j);
#pragma unroll
        for (int j = 7; j >= 0; --j) {
            const unsigned c[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
#pragma unroll
            for (int u = 3; u >= 0; --u) {
                cum += c[u];
                if (jk < 0 && cum >= static_cast<unsigned>(k)) jk = 4 * (half * 8 + j) + u;
                if (jm < 0 && cum >= static_cast<unsigned>(m)) jm = 4 * (half * 8 + j) + u;
            }
        }
    }
    if (jm < 0) return q.x;      // fewer than m rows counted so far: the seeded bound stands
    const float tm = __fadd_rd(q.x, __fmul_rd(static_cast<float>(jm), q.z));
    const float tk = __fsub_rd(__fadd_rd(q.x, __fmul_rd(static_cast<float>(jk), q.z)), q.w);
    return fmaxf(q.x, fminf(tm, tk));
}

// ---------------------------------------------------------------------------------------
// Fused top-K' epilogue.  Thread <-> accumulator row <-> query.  List slot j of thread t is
// ls[j * 128 + t] / li[j * 128 + t] (conflict-free across a warp).  Sched = SchedSearch (flat
// shard) or SchedCat (category segments); the unit's live query rows and gallery rows come from it.
// ---------------------------------------------------------------------------------------
template <int KCAP, class Sched = SchedSearch>
struct EpiTopK {
    struct Params {
        long long n_rows;
        int n_query;
        uint32_t* thr_enc;         // (n_qblocks * 128) encoded per-query thresholds
        float* cand_s;             // [n_units][cl][128][KCAP]
        int* cand_i;               // [n_units][128][KCAP] shard-local row ids
        int* cand_n;               // [n_units][128]
        int* progress;             // [n_units] scheduler pacing state (see SchedSearch::throttle), not used by the epilogue
        uint32_t* hist;            // [n_query][kHistBuckets] counting bound (see above), or null
        const float4* hq;          // [n_query] HistQ
        int k;
    };
    static constexpr int kSmemBytes = KCAP * 128 * 8 + 1024;      // lists + {lo, inv_w} per thread
    static constexpr int kWarps = 4;

    float* ls;
    int* li;
    int cnt, lpos, lidx;
    float lmin, thr;  // gate: s >= thr (thr = max(shared bound, list minimum once the list is full))
    float gthr;       // the shared bound: thr_enc / counting bound as last read
    bool full;

    __device__ void begin(const Params&, const Sched&, int quarter, int lane, uint8_t* smem) {
        const int t = quarter * 32 + lane;
        ls = reinterpret_cast<float*>(smem) + t;
        li = reinterpret_cast<int*>(smem + KCAP * 128 * 4) + t;
        cnt = 0; lpos = 0; lidx = 0; lmin = 0.f; thr = -INFINITY; gthr = -INFINITY; full = false;
    }

    __device__ void end(const Params&, int) {}
    __device__ void pre_tile(const Params&, const Sched&, int, int, uint8_t*) {}

    // evict candidate = lowest score, highest index among equal scores.  Static + by-value so
    // the per-thread state stays in registers (no `this` escaping into local memory).
    static __device__ __noinline__ float4 find_evict(const float* ls, const int* li) {
        float mn = ls[0];
        int mi = li[0], mp = 0;
#pragma unroll 8
        for (int j = 1; j < KCAP; ++j) {
            const float s = ls[j * 128];
            const int i = li[j * 128];
            if (s < mn || (s == mn && i > mi)) { mn = s; mi = i; mp = j; }
        }
        return make_float4(mn, __int_as_float(mp), __int_as_float(mi), 0.f);
    }
    __device__ __forceinline__ void rescan() {
        const float4 r = find_evict(ls, li);
        lmin = r.x;
        lpos = __float_as_int(r.y);
        lidx = __float_as_int(r.z);
        thr = fmaxf(r.x, gthr);
    }

    // Tiles of a unit arrive in rotated order, so ties are resolved on the index explicitly:
    // a full list takes s only if (s, idx) beats its worst entry under (score desc, index asc).
    __device__ __forceinline__ void insert(float s, int idx) {
        if (!full) {
            ls[cnt * 128] = s;
            li[cnt * 128] = idx;
            if (++cnt == KCAP) { full = true; rescan(); }
        } else if (s > lmin || idx < lidx) {
            ls[lpos * 128] = s;
            li[lpos * 128] = idx;
            rescan();
        }
    }

    // v[i] for a run-time i without spilling v[] to local memory: a 5-level select tree (31 selects)
    static __device__ __forceinline__ float sel32(const float (&v)[32], int i) {
        float a[16], b[8], c4[4];
#pragma unroll
        for (int j = 0; j < 16; ++j) a[j] = (i & 1) ? v[2 * j + 1] : v[2 * j];
#pragma unroll
        for (int j = 0; j < 8; ++j) b[j] = (i & 2) ? a[2 * j + 1] : a[2 * j];
#pragma unroll
        for (int j = 0; j < 4; ++j) c4[j] = (i & 4) ? b[2 * j + 1] : b[2 * j];
        const float d0 = (i & 8) ? c4[1] : c4[0], d1 = (i & 8) ? c4[3] : c4[2];
        return (i & 16) ? d1 : d0;
    }

    __device__ void tile(const Params& p, const Sched& s, uint32_t t_acc, int quarter,
                         int lane, uint8_t*) {
        const int row = s.m0 + quarter * 32 + lane;
        const bool live = row < s.m_end(p.n_query);
        uint32_t* const hrow = p.hist ? p.hist + static_cast<size_t>(row) * kHistBuckets : nullptr;
        float* const hp = reinterpret_cast<float*>(li + KCAP * 128);      // [2][128]: lo, inv_w of this thread's query
        if (s.first) {
            cnt = 0;
            full = false;
            gthr = live ? dec_score(__ldcg(p.thr_enc + row)) : INFINITY;
            thr = gthr;
            if (hrow && live) {
                const float4 q = __ldg(p.hq + row);
                hp[0] = q.x;
                hp[128] = q.y;
            }
        }
        // the first round learns the bound from scratch (it moves as kcap / rows seen): look four times as often
        const int period = s.unit < s.step ? kHistRefresh / 4 : kHistRefresh;
        if (hrow && live && (s.first || (s.it & (period - 1)) == 0)) {
            // every gate a row can be dropped at is folded into thr_enc (the certificate's T_out)
            const float t = hist_bound(hrow, p.hq + row, KCAP, p.k);
            const float g = dec_score(__ldcg(p.thr_enc + row));
            if (t > g) atomicMax(p.thr_enc + row, enc_score(t));
            gthr = fmaxf(gthr, fmaxf(t, g));
            thr = fmaxf(thr, gthr);
        }
        const long long col_lim = s.n_end(p.n_rows) - s.n0;  // columns >= col_lim are padding or another category
#pragma unroll 1
        for (int c = 0; c < kSearchBN; c += 32) {
            uint32_t raw[32];
            tmem_ld_32x32(t_acc + c, raw);
            tmem_ld_wait();
            float v[32];     // scores; the L2 bias is already inside (augmented k-block, see kAugCols)
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(raw[i]);
            float m4[4] = {v[0], v[1], v[2], v[3]};      // four independent max chains instead of one
#pragma unroll
            for (int i = 4; i < 32; ++i) m4[i & 3] = fmaxf(m4[i & 3], v[i]);
            const float mx = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
            if (__any_sync(0xffffffffu, mx >= thr)) {
                // Taken by the whole warp as soon as ONE of its 32 queries has a candidate in this slab.  Every lane
                // builds the bit mask of its own candidates and the lanes then pop theirs TOGETHER: the trip count
                // is the largest number of candidates any one query has in the slab (1, rarely 2), not the number
                // of distinct columns with a candidate anywhere in the warp -- with cold lists (first round) that
                // was 5-6 serialised insertions per slab.
                uint32_t mask = 0;
#pragma unroll
                for (int i = 0; i < 32; ++i) mask |= (v[i] >= thr) ? (1u << i) : 0u;
                const long long room = col_lim - c;
                if (room < 32) mask &= room <= 0 ? 0u : ((1u << static_cast<int>(room)) - 1u);
                while (__any_sync(0xffffffffu, mask != 0u)) {
                    if (mask) {
                        const int i = __ffs(mask) - 1;
                        mask &= mask - 1u;
                        const float sv = sel32(v, i);
                        if (sv >= thr) {          // thr may have risen with this lane's previous insertion
                            if (hrow) {
                                int b = static_cast<int>(__fmul_rn(__fsub_rn(sv, hp[0]), hp[128]));
                                b = max(0, min(kHistBuckets - 1, b));
                                atomicAdd(hrow + b, 1u);
                            }
                            insert(sv, s.n0 + c + i);
                        }
                    }
                }
            }
        }
        if (s.last) {
            const long long slot = (static_cast<long long>(s.unit) * s.p.cl + s.rank) * 128 + quarter * 32 + lane;
            const int n = live ? cnt : 0;
            for (int j = 0; j < n; ++j) {
                p.cand_s[slot * KCAP + j] = ls[j * 128];
                p.cand_i[slot * KCAP + j] = li[j * 128];
            }
            p.cand_n[slot] = n;
            if (live && full) atomicMax(p.thr_enc + row, enc_score(lmin));
        }
    }
};

// ---------------------------------------------------------------------------------------
// Threshold seeding epilogue.  For every query the maxima of NB disjoint blocks of 128 gallery rows are
// NB scores of NB distinct rows, so the m-th largest of them is a lower bound of the m-th best score of
// the whole gallery -- a valid starting threshold for the top-m lists of the main sweep.  The sample is split
// into as many segments as there are idle CTA pairs per query group (2 at 8192 queries, 4 at 4096): the units
// only write their maxima, seed_finish_kernel takes the m-th largest of the POOL (64 -> 128 blocks moves the
// bound from the 0.54 % to the 0.22 % quantile at the same wall time).  Unlike running the real top-k epilogue
// over a sample (the first warm-up: 1.15 ms at 8192 queries, dominated by list insertions into cold lists) this is
// one running maximum per thread per block: ~0.2 ms for 64 blocks per segment, and with NB = 2 m per segment the
// bound (the median of maxima of 128 samples = the 0.54 % quantile) is already tighter than the exact m-th best of
// 4096 rows (0.78 %).
// ---------------------------------------------------------------------------------------
template <int NBMAX>
struct EpiBlockMax {
    struct Params {
        long long n_rows;          // rows swept (multiple of kSearchBN, all real)
        int n_query;
        int* progress;             // scheduler pacing state (SchedSearch::throttle)
        float* bm;                 // [n_query][nb_total] pooled block maxima, segment-major
        int nb_seg, nb_total;      // blocks per sample segment, blocks of all segments
    };
    static constexpr int kMaxBlocks = NBMAX;
    static constexpr int kSmemBytes = kMaxBlocks * 128 * 4;
    static constexpr int kWarps = 4;

    float* ls;
    int nb;

    __device__ void begin(const Params&, const SchedSearch&, int quarter, int lane, uint8_t* smem) {
        ls = reinterpret_cast<float*>(smem) + quarter * 32 + lane;
        nb = 0;
    }
    __device__ void end(const Params&, int) {}
    __device__ void pre_tile(const Params&, const SchedSearch&, int, int, uint8_t*) {}

    __device__ void tile(const Params& p, const SchedSearch& s, uint32_t t_acc, int quarter, int lane, uint8_t*) {
        const int row = s.m0 + quarter * 32 + lane;
        if (s.first) nb = 0;
#pragma unroll 1
        for (int b = 0; b < kSearchBN / 128; ++b) {
            float bm = -INFINITY;
#pragma unroll 1
            for (int c = 0; c < 128; c += 32) {
                uint32_t raw[32];
                tmem_ld_32x32(t_acc + b * 128 + c, raw);
                tmem_ld_wait();
                float m4[4] = {__uint_as_float(raw[0]), __uint_as_float(raw[1]), __uint_as_float(raw[2]), __uint_as_float(raw[3])};
#pragma unroll
                for (int i = 4; i < 32; ++i) m4[i & 3] = fmaxf(m4[i & 3], __uint_as_float(raw[i]));
                bm = fmaxf(bm, fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3])));
            }
            if (nb < kMaxBlocks) ls[nb * 128] = bm;
            ++nb;
        }
        if (s.last) {
            // the unit's block maxima go to the query's pool (segment-major); seed_finish_kernel selects from the
            // pooled maxima of all sample segments
            const int n = min(nb, kMaxBlocks);
            if (row < p.n_query) {
                const int seg = s.unit / s.p.n_qgroups;
                float* out = p.bm + static_cast<size_t>(row) * p.nb_total + static_cast<size_t>(seg) * p.nb_seg;
                for (int j = 0; j < p.nb_seg; ++j) out[j] = j < n ? ls[j * 128] : -INFINITY;
            }
        }
    }
};

// ---------------------------------------------------------------------------------------
// fp32 -> bf16 rows (queries), and gallery packing (bf16 rows + 0.5|g|^2 from the fp32 data)
// ---------------------------------------------------------------------------------------
// queries (nq, dim) fp32 -> (nq, dim + kAugCols) bf16 with the bias selector columns
__global__ void __launch_bounds__(256)
to_bf16_kernel(const float* __restrict__ in, int n_query, int dim, float aug, __nv_bfloat16* __restrict__ out) {
    const int pitch = dim + kAugCols;
    const long long i = (static_cast<long long>(blockIdx.x) * 256 + threadIdx.x) * 4;
    if (i >= static_cast<long long>(n_query) * pitch) return;
    const int row = static_cast<int>(i / pitch), col = static_cast<int>(i - static_cast<long long>(row) * pitch);
    float4 v;
    if (col < dim) v = *reinterpret_cast<const float4*>(in + static_cast<long long>(row) * dim + col);
    else v = col == dim ? make_float4(aug, aug, 0.f, 0.f) : make_float4(0.f, 0.f, 0.f, 0.f);
    __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 u;
    u.x = *reinterpret_cast<uint32_t*>(&a);
    u.y = *reinterpret_cast<uint32_t*>(&b);
    *reinterpret_cast<uint2*>(out + i) = u;
}

// CAT: packed row `row` is gallery row perm[row] (category order), and the maximum of 0.5|g|^2 is kept per
// category (max_hs_bits[n_cat]); rows whose id is outside [0, n_cat) belong to no category and count nowhere.
template <bool CAT>
__global__ void __launch_bounds__(256)
gallery_pack_kernel(const float* __restrict__ g, long long n_rows, int dim,
                    __nv_bfloat16* __restrict__ out, float* __restrict__ half_sqnorm,
                    unsigned int* __restrict__ max_hs_bits, const int* __restrict__ perm = nullptr,
                    const int* __restrict__ cat = nullptr, int n_cat = 0) {
    const long long row = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
    if (row >= n_rows) return;
    const int lane = threadIdx.x & 31;
    const int pitch = dim + kAugCols;
    long long src = row;
    if constexpr (CAT) src = perm[row];
    float ss = 0.f;
    for (int e = lane * 4; e < dim; e += 128) {
        const float4 v = *reinterpret_cast<const float4*>(g + src * dim + e);
        ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
        __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
        uint2 u;
        u.x = *reinterpret_cast<uint32_t*>(&a);
        u.y = *reinterpret_cast<uint32_t*>(&b);
        *reinterpret_cast<uint2*>(out + row * pitch + e) = u;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    if (lane == 0) {
        if constexpr (CAT) {
            const int c = cat[src];
            if (static_cast<unsigned>(c) < static_cast<unsigned>(n_cat)) atomicMax(max_hs_bits + c, __float_as_uint(0.5f * ss));
        } else {
            half_sqnorm[row] = 0.5f * ss;
            atomicMax(max_hs_bits, __float_as_uint(0.5f * ss));     // non-negative floats order like their bit patterns
        }
    }
    // bias columns: -0.5|g|^2 = hi + lo in bf16, then zeros (2 x 4 bytes per lane = 64 columns)
    const float bias = -0.5f * ss;
    const __nv_bfloat16 hi = __float2bfloat16_rn(bias);
    const __nv_bfloat16 lo = __float2bfloat16_rn(bias - __bfloat162float(hi));
    __nv_bfloat162 z = __floats2bfloat162_rn(0.f, 0.f), first;
    first.x = hi; first.y = lo;
    __nv_bfloat162* aug = reinterpret_cast<__nv_bfloat162*>(out + row * pitch + dim);
    aug[lane] = lane == 0 ? first : z;
}

// ---------------------------------------------------------------------------------------
// Pass 2: merge + exact re-rank.  One CTA per query.
// key = enc(score) << 32 | (0xFFFFFFFF - idx): descending key = score desc, index asc.
// ---------------------------------------------------------------------------------------
struct MergeArgs {
    const float* cand_s;
    const int* cand_i;
    const int* cand_n;
    int kcap, n_seg, n_qgroups, cl, n_pad;  // n_pad = pow2 >= n_seg * kcap
    const float* queries;       // (nq, dim) fp32
    const float* gallery_f32;   // (n_rows, dim) fp32 or nullptr (no re-rank: bf16-pass scores)
    int dim, metric, k;
    long long id_offset;
    double* out_score;          // (nq, k)
    long long* out_idx;         // (nq, k)
    const uint32_t* thr_enc;    // per-query encoded threshold left by pass 1 (<= the global kcap-th best)
    const float* max_half_sqnorm;   // max over the shard of 0.5|g|^2 (tail of the packed gallery), for the certificate
    unsigned char* certified;   // (nq) or nullptr: 1 = the returned top-k is PROVEN equal to the exhaustive fp64 result
    unsigned long long* prof;   // OFX_MERGE_PROF=1: [0..3] summed cycles of gather / sort / re-score / rank, [4] CTAs that sorted all keys
    // category search only (merge_rerank_kernel<true>): candidate ids are packed rows
    const int* qpos;            // (nq) query row in the category-grouped query blocks, -1 = no row of its category here
    const int* grp;             // [groups][3] {first unit, unit stride, units} of a group of cl query blocks
    const int* perm;            // packed row -> shard-local row (fp32 rows and returned ids)
    const int* q_cat;           // (nq) category of each query; max_half_sqnorm is per category
};

constexpr int kMergeThreads = 256;
constexpr int kMergeSmall = 512;   // capacity of the selected-key buffer (power of two)
constexpr int kMergeSelect = 128;  // with more candidates than this, select before sorting
constexpr int kMaxRerank = 128;
constexpr int kMaxScored = kMaxRerank + kMergeSmall;   // shortlist + certificate extension

// Rigorous bound on |bf16-pass score - exact score| of ANY gallery row for a query of norm qn, G = max |g|:
//   operands rounded to bf16 (round to nearest, relative error u = 2^-9 each): |q.g - q^.g^| <= (2u + u^2) |q||g|;
//   fp32 accumulation of the K = dim + 64 exact bf16 products in the tensor core: <= K 2^-22 |q^||g^| (truncating
//   adder, factor-two margin);  the L2 bias -0.5|g|^2 as bf16 hi + lo of an fp32 sum: <= (2^-18 + dim 2^-24) 0.5 G^2.
// The certificate below is a worst-case statement; the typical error is ~50x smaller (it grows with sqrt(K), not K).
__device__ __forceinline__ double bf16_score_error_bound(double qn, double half_g2, int dim, int metric) {
    const double u = 1.0 / 512.0;
    const double g = sqrt(2.0 * half_g2);
    double e = (2.0 * u + u * u + (dim + 64) * (1.0 / 4194304.0)) * qn * g * (1.0 + u) * (1.0 + u);
    if (metric == OFX_METRIC_L2) e += (1.0 / 262144.0 + dim * (1.0 / 16777216.0)) * half_g2;
    return e * 1.01;
}

// After the seeding sweep, one warp per query: the m-th largest of the pooled block maxima becomes the query's
// starting threshold, and (hq != null) the parameters of the counting bound are set and its histogram cleared.
__global__ void __launch_bounds__(256)
seed_finish_kernel(const float* __restrict__ queries, int n_query, int dim, int metric, const float* __restrict__ bm,
                   int nb_total, int m, uint32_t* __restrict__ thr_enc, const float* __restrict__ max_half_sqnorm,
                   float4* __restrict__ hq, uint32_t* __restrict__ hist) {
    const int q = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (q >= n_query) return;
    // rank of every pooled maximum by counting (value desc, position asc); nb_total <= 1024
    const float* b = bm + static_cast<size_t>(q) * nb_total;
    float kth = -INFINITY, top = -INFINITY;
    for (int i0 = 0; i0 < nb_total; i0 += 32) {
        const int i = i0 + lane;
        const float v = i < nb_total ? __ldg(b + i) : -INFINITY;
        int rank = 0;
        for (int j = 0; j < nb_total; ++j) {
            const float w = __ldg(b + j);
            rank += (w > v || (w == v && j < i)) ? 1 : 0;
        }
        if (i < nb_total && rank == m - 1) kth = v;
        if (i < nb_total && rank == 0) top = v;
    }
    for (int o = 16; o; o >>= 1) {
        kth = fmaxf(kth, __shfl_xor_sync(0xffffffffu, kth, o));
        top = fmaxf(top, __shfl_xor_sync(0xffffffffu, top, o));
    }
    if (lane == 0 && kth > -INFINITY) atomicMax(thr_enc + q, enc_score(kth));
    if (!hq) return;
    double qq = 0.0;
    for (int c = lane; c < dim; c += 32) {
        const double v = static_cast<double>(__ldg(queries + static_cast<size_t>(q) * dim + c));
        qq += v * v;
    }
    for (int o = 16; o; o >>= 1) qq += __shfl_xor_sync(0xffffffffu, qq, o);
    for (int c = lane; c < kHistBuckets; c += 32) hist[static_cast<size_t>(q) * kHistBuckets + c] = 0u;
    if (lane) return;
    const double eps = bf16_score_error_bound(sqrt(qq) * (1.0 + 1e-9), static_cast<double>(__ldg(max_half_sqnorm)), dim, metric);
    const float lo = kth;
    const float span = (top - lo) * (2.5f / kHistBuckets);
    float4 r;
    r.x = lo;
    if (lo > -INFINITY && span > 0.f && span < INFINITY && 1.f / span < INFINITY) {
        r.y = 1.f / span;
        r.z = __double2float_rd((1.0 / static_cast<double>(r.y)) * (1.0 - 2e-6));
    } else {             // degenerate sample (ties, infinities): every candidate counts in bucket 0, whose edge is lo
        r.y = 0.f;
        r.z = 0.f;
    }
    r.w = __double2float_ru(2.0 * eps * 1.001);
    hq[q] = r;
}

// CAT: the query's lists are those of its group's units (a.grp), not one per gallery segment; candidate ids are
// packed rows, mapped through a.perm to read the fp32 row and to emit the id.  Within a category packed order is
// the original order, so ranking by (score, packed row) is ranking by (score, id).
template <bool CAT>
__global__ void __launch_bounds__(kMergeThreads)
merge_rerank_kernel(const MergeArgs a) {
    extern __shared__ unsigned long long keys[];
    __shared__ double r_score[kMaxScored];
    __shared__ long long r_idx[kMaxScored];
    __shared__ int n_valid;
    __shared__ int n_ext;
    __shared__ double s_kth, s_qq;
    const int q = blockIdx.x, tid = threadIdx.x;
    int qb = q / kBM, r = q % kBM, trow = q, n_seg = a.n_seg, u0 = 0, ustride = 0;
    if constexpr (CAT) {
        const int pos = a.qpos[q];
        if (pos < 0) {       // no row of the query's category in this shard: padding only, trivially exact
            for (int j = tid; j < a.k; j += kMergeThreads) {
                a.out_score[static_cast<long long>(q) * a.k + j] = -INFINITY;
                a.out_idx[static_cast<long long>(q) * a.k + j] = -1;
            }
            if (tid == 0 && a.certified) a.certified[q] = a.gallery_f32 ? 1 : 0;
            return;
        }
        qb = pos / kBM; r = pos % kBM; trow = pos;
        const int* g = a.grp + 3 * (qb / a.cl);
        u0 = g[0]; ustride = g[1]; n_seg = g[2];
    }
    auto src_row = [&](long long idx) -> long long {
        if constexpr (CAT) return a.perm[idx];
        return idx;
    };
    __shared__ int n_small, sel_bin;
    __shared__ unsigned int es_lo, es_hi;
    __shared__ int hist[256];
    if (tid == 0) { n_valid = 0; n_small = 0; es_lo = 0xFFFFFFFFu; es_hi = 0u; sel_bin = -1; n_ext = 0; s_qq = 0.0; }
    hist[tid] = 0;     // kMergeThreads == 256
    __syncthreads();
    const long long tstart = a.prof ? clock64() : 0;
    unsigned long long* small = keys + a.n_pad;
    int mine = 0;
    uint32_t my_lo = 0xFFFFFFFFu, my_hi = 0u;
    for (int e = tid; e < a.n_pad; e += kMergeThreads) {
        const int seg = e / a.kcap, j = e - seg * a.kcap;
        unsigned long long key = 0ull;
        if (seg < n_seg) {
            const long long unit = CAT ? static_cast<long long>(u0) + static_cast<long long>(seg) * ustride
                                       : static_cast<long long>(seg) * a.n_qgroups + qb / a.cl;
            const long long slot = (unit * a.cl + qb % a.cl) * 128 + r;
            if (j < a.cand_n[slot]) {
                const float s = a.cand_s[slot * a.kcap + j];
                const uint32_t idx = static_cast<uint32_t>(a.cand_i[slot * a.kcap + j]);
                const uint32_t es = enc_score(s);
                key = (static_cast<unsigned long long>(es) << 32) | (0xFFFFFFFFu - idx);
                ++mine;
                my_lo = min(my_lo, es);
                my_hi = max(my_hi, es);
            }
        }
        keys[e] = key;
    }
    if (mine) { atomicAdd(&n_valid, mine); atomicMin(&es_lo, my_lo); atomicMax(&es_hi, my_hi); }
    __syncthreads();
    // Selection instead of a full sort.  The n_seg lists of a query hold up to n_seg * kcap candidates, all of
    // them near the top of the score distribution (each unit keeps ITS kcap best), so a score threshold left
    // by pass 1 filters almost nothing once the gallery is cut into many segments (measured: every query fell
    // back to the 2048-key bitonic sort, 55 % of this kernel).  A 256-bin histogram of the encoded scores over
    // [min, max] finds the bin that holds the kcap-th best; only the keys in that bin or above (kcap plus the
    // bin's population, typically < 128) are sorted.
    if (n_valid > kMergeSelect) {
        const unsigned long long span = static_cast<unsigned long long>(es_hi - es_lo) + 1ull;
        for (int e = tid; e < a.n_pad; e += kMergeThreads) {
            const unsigned long long key = keys[e];
            if (key) atomicAdd(&hist[static_cast<int>(((static_cast<unsigned long long>(static_cast<uint32_t>(key >> 32) - es_lo)) << 8) / span)], 1);
        }
        __syncthreads();
        if (tid < 32) {      // suffix sums from the top bin down, 8 bins per lane
            int loc = 0;
#pragma unroll
            for (int i = 0; i < 8; ++i) loc += hist[255 - (tid * 8 + i)];
            int inc = loc;   // inclusive scan over lanes (lane 0 = top 8 bins)
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, inc, o);
                if (tid >= o) inc += v;
            }
            const int before = inc - loc;
            if (before < a.kcap && inc >= a.kcap) {      // exactly one lane: the kcap-th best lies in its 8 bins
                int c = before;
                for (int i = 0; i < 8; ++i) {
                    c += hist[255 - (tid * 8 + i)];
                    if (c >= a.kcap) { sel_bin = 255 - (tid * 8 + i); break; }
                }
            }
        }
        __syncthreads();
        if (sel_bin >= 0) {
            for (int e = tid; e < a.n_pad; e += kMergeThreads) {
                const unsigned long long key = keys[e];
                if (key && static_cast<int>(((static_cast<unsigned long long>(static_cast<uint32_t>(key >> 32) - es_lo)) << 8) / span) >= sel_bin) {
                    const int pos = atomicAdd(&n_small, 1);
                    if (pos < kMergeSmall) small[pos] = key;
                }
            }
        }
        __syncthreads();
    } else if (a.n_pad > kMergeSelect) {     // few candidates in many (mostly empty) lists: compact them
        for (int e = tid; e < a.n_pad; e += kMergeThreads) {
            const unsigned long long key = keys[e];
            if (key) small[atomicAdd(&n_small, 1)] = key;
        }
        if (tid == 0) sel_bin = 0;
        __syncthreads();
    }
    const bool use_small = sel_bin >= 0 && n_small <= kMergeSmall && (n_small >= a.kcap || n_small == n_valid);
    long long tp0 = 0, tp1 = 0, tp2 = 0;
    if (a.prof && tid == 0) { tp1 = clock64(); atomicAdd(a.prof + 0, static_cast<unsigned long long>(tp1 - tstart)); if (!use_small) atomicAdd(a.prof + 4, 1ull); }
    int sort_n = a.n_pad;
    unsigned long long* sk = keys;
    if (use_small) {
        sort_n = 32;
        while (sort_n < n_small) sort_n <<= 1;
        for (int e = n_small + tid; e < sort_n; e += kMergeThreads) small[e] = 0ull;
        sk = small;
        __syncthreads();
    }
    // bitonic sort, descending
    for (int size = 2; size <= sort_n; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int e = tid; e < sort_n / 2; e += kMergeThreads) {
                const int lo = 2 * e - (e & (stride - 1));
                const int hi = lo + stride;
                const bool desc = (lo & size) == 0;
                const unsigned long long x = sk[lo], y = sk[hi];
                if ((x < y) == desc) { sk[lo] = y; sk[hi] = x; }
            }
            __syncthreads();
        }
    }
    if (a.prof && tid == 0) { tp2 = clock64(); atomicAdd(a.prof + 1, static_cast<unsigned long long>(tp2 - tp1)); }
    const int n_total = n_valid;      // every candidate pass 1 kept for this query (all of them are still in keys[])
    __syncthreads();
    if (use_small && tid == 0) n_valid = n_small;
    __syncthreads();
    const int n_r = min(min(n_valid, a.kcap), kMaxRerank);
    const int warp = tid >> 5, lane = tid & 31;
    const unsigned long long key_last = n_r > 0 ? sk[n_r - 1] : 0ull;   // worst (bf16 score, index) of the shortlist
    // the gallery rows of the candidates are cold 4 KB reads scattered over HBM: every warp asks for all of its
    // rows at once (one 128-byte line per lane and row) before it starts on the first
    if (a.gallery_f32) {
        for (int c = warp; c < n_r; c += kMergeThreads / 32) {
            const long long idx = 0xFFFFFFFFu - static_cast<uint32_t>(sk[c] & 0xFFFFFFFFull);
            const float* g = a.gallery_f32 + src_row(idx) * a.dim;
            for (int d = lane * 32; d < a.dim; d += 1024)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(g + d));
        }
    }
    // exact score of one candidate (whole warp), fp64 from the fp32 rows
    auto exact_score = [&](unsigned long long key, long long idx) -> double {
        if (!a.gallery_f32) return static_cast<double>(dec_score(static_cast<uint32_t>(key >> 32)));
        const float* g = a.gallery_f32 + src_row(idx) * a.dim;
        const float* qv = a.queries + static_cast<long long>(q) * a.dim;
        double acc = 0.0, nn = 0.0;
        // eight gallery elements per lane in flight (the row is a cold 4 KB read from HBM; as a rolled loop
        // its 32 iterations were 32 exposed round trips); same element order per lane as before
        for (int d0 = lane; d0 < a.dim; d0 += 256) {
            float gv[8], qq[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int d = d0 + 32 * u;
                gv[u] = d < a.dim ? __ldcs(g + d) : 0.f;
                qq[u] = d < a.dim ? __ldg(qv + d) : 0.f;
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const double gd = static_cast<double>(gv[u]);
                acc = fma(static_cast<double>(qq[u]), gd, acc);
                nn = fma(gd, gd, nn);
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            acc += __shfl_xor_sync(0xffffffffu, acc, o);
            nn += __shfl_xor_sync(0xffffffffu, nn, o);
        }
        return a.metric == OFX_METRIC_L2 ? acc - 0.5 * nn : acc;
    };
    for (int c = warp; c < n_r; c += kMergeThreads / 32) {
        const unsigned long long key = sk[c];
        const long long idx = 0xFFFFFFFFu - static_cast<uint32_t>(key & 0xFFFFFFFFull);
        const double score = exact_score(key, idx);
        if (lane == 0) { r_score[c] = score; r_idx[c] = idx; }
    }
    // |q|^2 for the certificate (fp64, all threads)
    if (a.certified && a.gallery_f32) {
        double qq = 0.0;
        for (int d = tid; d < a.dim; d += kMergeThreads) {
            const double v = static_cast<double>(__ldg(a.queries + static_cast<long long>(q) * a.dim + d));
            qq = fma(v, v, qq);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) qq += __shfl_xor_sync(0xffffffffu, qq, o);
        if (lane == 0) atomicAdd(&s_qq, qq);
    }
    __syncthreads();
    if (a.prof && tid == 0) { tp0 = clock64(); atomicAdd(a.prof + 2, static_cast<unsigned long long>(tp0 - tp2)); }
    // rank of every scored candidate under (score desc, index asc); rank k-1 is the k-th best
    auto rank_and_emit = [&](int n_s) {
        if (tid == 0) s_kth = -INFINITY;
        __syncthreads();
        if (tid < a.k && tid >= n_s) {
            const long long o = static_cast<long long>(q) * a.k + tid;
            a.out_score[o] = -INFINITY; a.out_idx[o] = -1;
        }
        for (int e = tid; e < n_s; e += kMergeThreads) {
            const double se = r_score[e];
            const long long id = r_idx[e];
            int rank = 0;
            for (int j = 0; j < n_s; ++j) {
                const double sj = r_score[j];
                rank += (sj > se) || (sj == se && r_idx[j] < id);
            }
            if (rank < a.k) {
                const long long o = static_cast<long long>(q) * a.k + rank;
                a.out_score[o] = se;
                a.out_idx[o] = a.id_offset + src_row(id);
                if (rank == a.k - 1) s_kth = se;
            }
        }
        __syncthreads();
    };
    rank_and_emit(n_r);
    if (!a.certified) return;
    // ---------------------------------------------------------------- exactness certificate
    // Claim to prove: no gallery row outside the scored set can reach the k-th best exact score S_k.
    //  * rows pass 1 never listed: their bf16 score is <= the final per-query threshold T_out (a unit drops a row
    //    only below its admission gate, and every gate -- seeded bound, a finished unit's list minimum -- is folded
    //    into thr_enc with atomicMax), so their exact score is <= T_out + eps;
    //  * listed rows outside the shortlist: bf16 score <= the shortlist's worst, T_in.  If S_k - eps does not clear
    //    T_in, every listed row with bf16 score >= S_k - eps is re-scored too (the extension below).
    // eps = bf16_score_error_bound(|q|, max 0.5|g|^2).  No re-rank (bf16 ranking requested): nothing is claimed.
    if (!a.gallery_f32) { if (tid == 0) a.certified[q] = 0; return; }
    const float* hs_max = a.max_half_sqnorm;
    if constexpr (CAT) hs_max += a.q_cat[q];        // the category's bound (tighter than the shard's)
    const double eps = bf16_score_error_bound(sqrt(s_qq), static_cast<double>(__ldg(hs_max)), a.dim, a.metric);
    const uint32_t thr_e = a.thr_enc ? __ldcg(a.thr_enc + trow) : 0u;
    const bool gated = thr_e != 0u;                  // some row may have been dropped without being listed
    const double t_out = gated ? static_cast<double>(dec_score(thr_e)) : -INFINITY;
    bool ok = true;
    int n_s = n_r;
    if (n_total > n_r) {
        const double need = s_kth - eps;             // -inf when fewer than k rows were scored: everything listed is needed
        const double t_in = static_cast<double>(dec_score(static_cast<uint32_t>(key_last >> 32)));
        if (!(t_in < need)) {
            // extension: listed candidates below the shortlist whose bf16 score reaches `need` (keys[] still holds
            // every listed candidate; the shortlist is exactly the keys >= key_last)
            for (int e = tid; e < a.n_pad; e += kMergeThreads) {
                const unsigned long long key = keys[e];
                if (key && key < key_last && static_cast<double>(dec_score(static_cast<uint32_t>(key >> 32))) >= need) {
                    const int pos = atomicAdd(&n_ext, 1);
                    if (pos < kMergeSmall) r_idx[n_r + pos] = static_cast<long long>(key);   // parked, replaced by the index below
                }
            }
            __syncthreads();
            if (n_ext > kMergeSmall) ok = false;     // more near-ties than the extension holds: leave it to the exhaustive fallback
            const int n_e = min(n_ext, kMergeSmall);
            for (int c = warp; c < n_e; c += kMergeThreads / 32) {
                const unsigned long long key = static_cast<unsigned long long>(r_idx[n_r + c]);
                const long long idx = 0xFFFFFFFFu - static_cast<uint32_t>(key & 0xFFFFFFFFull);
                const double score = exact_score(key, idx);
                __syncwarp();
                if (lane == 0) { r_score[n_r + c] = score; r_idx[n_r + c] = idx; }
            }
            __syncthreads();
            n_s = n_r + n_e;
            rank_and_emit(n_s);
        }
    }
    if (n_s < a.k) ok = ok && !gated && n_total == n_s;        // fewer than k rows: exact only if nothing was ever dropped
    else if (gated) ok = ok && (t_out < s_kth - eps);
    if (tid == 0) a.certified[q] = ok ? 1 : 0;
}

// ---------------------------------------------------------------------------------------
// Merge of R per-shard lists (after the all-gather): rank by (-score, idx), padding last.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
topk_merge_kernel(const double* __restrict__ scores, const long long* __restrict__ idx, int n_lists,
                  int n_query, int k, double* __restrict__ out_score, long long* __restrict__ out_idx,
                  const int* __restrict__ out_row = nullptr) {
    extern __shared__ unsigned char sm[];
    const int n = n_lists * k;
    double* s = reinterpret_cast<double*>(sm);
    long long* id = reinterpret_cast<long long*>(sm + sizeof(double) * n);
    const int q = blockIdx.x;
    const long long oq = out_row ? out_row[q] : q;      // the exhaustive fallback scatters into the caller's rows
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
        const int l = e / k, j = e - l * k;
        const long long src = (static_cast<long long>(l) * n_query + q) * k + j;
        s[e] = scores[src];
        id[e] = idx[src];
    }
    __syncthreads();
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
        const double se = s[e];
        const long long ie = id[e];
        const bool pad_e = ie < 0;
        int rank = 0;
        for (int j = 0; j < n; ++j) {
            const bool pad_j = id[j] < 0;
            bool better;
            if (pad_e != pad_j) better = pad_e;  // real entries before padding
            else if (pad_e) better = j < e;
            else better = s[j] > se || (s[j] == se && (id[j] < ie || (id[j] == ie && j < e)));
            rank += better;
        }
        if (rank < k) {
            out_score[oq * k + rank] = pad_e ? -INFINITY : se;
            out_idx[oq * k + rank] = pad_e ? -1 : ie;
        }
    }
}

// ---------------------------------------------------------------------------------------
// Exhaustive fp64 search of a few selected queries: the fallback for queries whose tensor-core result could not
// be certified (near-duplicate gallery rows closer than bf16 resolution, ofx_topk_search's out_certified == 0).
// CTA (c, s): row chunk c x group s of up to kExactQ selected queries.  A warp takes one gallery row at a time
// (coalesced 16-byte loads), forms the fp64 dot products with the group's queries (fp32 copies in shared memory)
// and keeps a private top-k per query; the CTA merges its 8 warps' lists and emits one list per (chunk, query);
// topk_merge_kernel then merges the chunks.  Arithmetic and ranking are those of merge_rerank_kernel / the fp64
// oracle: score = q.g (- 0.5 |g|^2), ties to the lowest index.
// ---------------------------------------------------------------------------------------
constexpr int kExactQ = 8;
constexpr int kExactWarps = 8;

// CAT: one selected query per blockIdx.x, and the chunks (blockIdx.y) split the query's category segment
// [seg_off[c], seg_off[c+1]) of packed rows, read through perm, so the cost follows the segment, not the shard.
// Listed ids are packed rows (ascending within the category like the original ids).
struct ExactCat {
    const int* perm;
    const long long* seg_off;
    const int* q_cat;
    int n_cat;
};

template <bool CAT>
__global__ void __launch_bounds__(kExactWarps * 32)
exact_scan_kernel(const float* __restrict__ gallery, long long n_rows, int dim, int metric,
                  const float* __restrict__ queries, const int* __restrict__ sel, int n_sel, int k,
                  long long rows_per_chunk, double* __restrict__ part_s, long long* __restrict__ part_i,
                  const ExactCat xc) {
    extern __shared__ unsigned char sm_raw[];
    float* sq = reinterpret_cast<float*>(sm_raw);                                   // [kExactQ][dim]
    double* ls = reinterpret_cast<double*>(sm_raw + sizeof(float) * kExactQ * dim);  // [warps][kExactQ][k]
    long long* li = reinterpret_cast<long long*>(ls + kExactWarps * kExactQ * k);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // CAT: x = selected query, y = chunk of its segment (grid x takes any number of queries)
    const int chunk = CAT ? blockIdx.y : blockIdx.x, n_chunks = CAT ? gridDim.y : gridDim.x;
    const int q0 = CAT ? blockIdx.x : blockIdx.y * kExactQ, nq = CAT ? 1 : min(kExactQ, n_sel - q0);
    for (int e = threadIdx.x; e < nq * dim; e += blockDim.x)
        sq[e] = queries[static_cast<long long>(sel[q0 + e / dim]) * dim + e % dim];
    for (int e = threadIdx.x; e < kExactWarps * kExactQ * k; e += blockDim.x) { ls[e] = -INFINITY; li[e] = -1; }
    __syncthreads();
    double* my_s = ls + warp * kExactQ * k;
    long long* my_i = li + warp * kExactQ * k;
    double worst_s[kExactQ];      // current worst entry of each private list (lane 0's copy is authoritative)
    int worst_p[kExactQ];
#pragma unroll
    for (int j = 0; j < kExactQ; ++j) { worst_s[j] = -INFINITY; worst_p[j] = 0; }
    long long lo = chunk * rows_per_chunk, hi = min(n_rows, lo + rows_per_chunk);
    if constexpr (CAT) {
        const int c = xc.q_cat[sel[q0]];
        lo = hi = 0;
        if (static_cast<unsigned>(c) < static_cast<unsigned>(xc.n_cat)) {
            const long long s_lo = xc.seg_off[c], s_hi = xc.seg_off[c + 1];
            const long long per = (s_hi - s_lo + n_chunks - 1) / n_chunks;
            lo = s_lo + chunk * per;
            hi = min(s_hi, lo + per);
        }
    }
    for (long long row = lo + warp; row < hi; row += kExactWarps) {
        double acc[kExactQ], nn = 0.0;
#pragma unroll
        for (int j = 0; j < kExactQ; ++j) acc[j] = 0.0;
        long long src = row;
        if constexpr (CAT) src = xc.perm[row];
        for (int d = lane * 4; d < dim; d += 128) {
            const float4 g4 = __ldcs(reinterpret_cast<const float4*>(gallery + src * dim + d));
            const double g[4] = {g4.x, g4.y, g4.z, g4.w};
#pragma unroll
            for (int u = 0; u < 4; ++u) nn = fma(g[u], g[u], nn);
#pragma unroll
            for (int j = 0; j < kExactQ; ++j) {
                if (j < nq) {
                    const float4 q4 = *reinterpret_cast<const float4*>(sq + j * dim + d);
                    acc[j] = fma(static_cast<double>(q4.x), g[0], acc[j]);
                    acc[j] = fma(static_cast<double>(q4.y), g[1], acc[j]);
                    acc[j] = fma(static_cast<double>(q4.z), g[2], acc[j]);
                    acc[j] = fma(static_cast<double>(q4.w), g[3], acc[j]);
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            nn += __shfl_xor_sync(0xffffffffu, nn, o);
#pragma unroll
            for (int j = 0; j < kExactQ; ++j) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], o);
        }
        if (lane == 0) {
#pragma unroll
            for (int j = 0; j < kExactQ; ++j) {
                if (j >= nq) continue;
                const double sc = metric == OFX_METRIC_L2 ? acc[j] - 0.5 * nn : acc[j];
                // rows arrive in ascending index order, so an equal score never displaces an earlier row
                if (sc > worst_s[j] || my_i[j * k + worst_p[j]] < 0) {
                    my_s[j * k + worst_p[j]] = sc;
                    my_i[j * k + worst_p[j]] = row;
                    double ws = my_s[j * k]; long long wi = my_i[j * k]; int wp = 0;
                    for (int t = 1; t < k; ++t) {
                        const double st = my_s[j * k + t]; const long long it = my_i[j * k + t];
                        // worst = an empty slot first, else lowest score, among equals the highest index
                        const bool worse = (wi >= 0) && (it < 0 || st < ws || (st == ws && it > wi));
                        if (worse) { ws = st; wi = it; wp = t; }
                    }
                    worst_s[j] = wi < 0 ? -INFINITY : ws;
                    worst_p[j] = wp;
                }
            }
        }
    }
    __syncthreads();
    // merge the warps' lists: rank by counting over kExactWarps * k entries per query
    const int n = kExactWarps * k;
    for (int e = threadIdx.x; e < nq * n; e += blockDim.x) {
        const int j = e / n, t = e % n, w = t / k, p = t % k;
        const double se = ls[(w * kExactQ + j) * k + p];
        const long long ie = li[(w * kExactQ + j) * k + p];
        if (ie < 0) continue;
        int rank = 0;
        for (int w2 = 0; w2 < kExactWarps; ++w2)
            for (int p2 = 0; p2 < k; ++p2) {
                const long long i2 = li[(w2 * kExactQ + j) * k + p2];
                if (i2 < 0) continue;
                const double s2 = ls[(w2 * kExactQ + j) * k + p2];
                rank += (s2 > se) || (s2 == se && i2 < ie);
            }
        if (rank < k) {
            const long long o = (static_cast<long long>(chunk) * n_sel + q0 + j) * k + rank;
            part_s[o] = se;
            part_i[o] = ie;
        }
    }
}

// CAT: the listed ids are packed rows; the returned id is offset + perm[row]
template <bool CAT>
__global__ void add_offset_kernel(long long* idx, const int* __restrict__ sel, int n_sel, int k, long long offset,
                                  unsigned char* certified, const int* __restrict__ perm) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_sel * k) return;
    const long long o = static_cast<long long>(sel[e / k]) * k + e % k;
    if constexpr (CAT) {
        if (idx[o] >= 0) idx[o] = offset + perm[idx[o]];
    } else {
        if (idx[o] >= 0) idx[o] += offset;
    }
    if (certified && e % k == 0) certified[sel[e / k]] = 1;
}

// ---------------------------------------------------------------------------------------
// Category gallery (ofx_category_gallery_pack): a stable counting sort of the shard's rows by category.
//   cat_count_kernel            rows per category; bin n_cat collects ids outside [0, n_cat) (in no segment)
//   cat_scan_kernel             seg_off = exclusive prefix sums of the bins (one block)
//   cat_sort_kernel             perm: chunks of 1024 rows, each sorted in shared memory by (category, row) and
//                               then placed in chunk order -- a chunk waits until the previous one has advanced the
//                               per-category cursors, so the rows of a category keep their original order.  Chunks
//                               take tickets in the order they start, so the chunk waited on is always running.
//   gallery_pack_kernel<true>   bf16 rows in packed order + per-category maximum of 0.5|g|^2
// ---------------------------------------------------------------------------------------
constexpr int kMaxCategories = 65536;
constexpr int kSortChunk = 1024;
constexpr int kMaxCatRanges = 64;     // units per query group: merge fan-in kMaxCatRanges * kcap <= 8192

__global__ void __launch_bounds__(256)
cat_count_kernel(const int* __restrict__ cat, long long n, int n_cat, int* __restrict__ cnt) {
    const long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
    int c = -1;
    if (i < n) {
        c = cat[i];
        if (static_cast<unsigned>(c) >= static_cast<unsigned>(n_cat)) c = n_cat;
    }
    // one atomic per distinct category of a warp: a dominant category would otherwise serialise on one address
    const unsigned same = __match_any_sync(0xffffffffu, c);
    if (c >= 0 && static_cast<int>(threadIdx.x & 31) == __ffs(same) - 1) atomicAdd(cnt + c, __popc(same));
}

// exclusive prefix sum over the 1024 threads of a block; *total = the sum of all v
__device__ long long block_exscan(long long v, long long* sh, long long* total) {
    const int t = threadIdx.x;
    sh[t] = v;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        const long long x = t >= o ? sh[t - o] : 0;
        __syncthreads();
        sh[t] += x;
        __syncthreads();
    }
    const long long incl = sh[t];
    *total = sh[1023];
    __syncthreads();
    return incl - v;
}

__global__ void __launch_bounds__(1024)
cat_scan_kernel(const int* __restrict__ cnt, int n_bins, long long* __restrict__ seg_off) {
    __shared__ long long sh[1024];
    const int per = (n_bins + 1023) / 1024;
    const int b0 = min(n_bins, static_cast<int>(threadIdx.x) * per), b1 = min(n_bins, b0 + per);
    long long s = 0, total;
    for (int b = b0; b < b1; ++b) s += cnt[b];
    long long o = block_exscan(s, sh, &total);
    for (int b = b0; b < b1; ++b) { seg_off[b] = o; o += cnt[b]; }
}

__global__ void __launch_bounds__(512)
cat_sort_kernel(const int* __restrict__ cat, long long n, int n_cat, const long long* __restrict__ seg_off,
                int* cursor, int* chain, int* __restrict__ perm) {
    __shared__ uint32_t key[kSortChunk];      // category << 10 | row within the chunk
    __shared__ int run0[kSortChunk];          // sorted position where the element's category starts
    __shared__ int s_chunk;
    const int t = threadIdx.x;
    if (t == 0) s_chunk = atomicAdd(chain, 1);
    __syncthreads();
    const int chunk = s_chunk;
    const long long base = static_cast<long long>(chunk) * kSortChunk;
    for (int e = t; e < kSortChunk; e += 512) {
        const long long i = base + e;
        uint32_t kk = 0xFFFFFFFFu;
        if (i < n) {
            int c = cat[i];
            if (static_cast<unsigned>(c) >= static_cast<unsigned>(n_cat)) c = n_cat;
            kk = (static_cast<uint32_t>(c) << 10) | static_cast<uint32_t>(e);
        }
        key[e] = kk;
    }
    __syncthreads();
    for (int size = 2; size <= kSortChunk; size <<= 1) {      // bitonic sort, ascending
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            const int lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
            const bool up = (lo & size) == 0;
            const uint32_t x = key[lo], y = key[hi];
            if ((x > y) == up) { key[lo] = y; key[hi] = x; }
            __syncthreads();
        }
    }
    for (int e = t; e < kSortChunk; e += 512) run0[e] = (e == 0 || (key[e] >> 10) != (key[e - 1] >> 10)) ? e : 0;
    __syncthreads();
    for (int o = 1; o < kSortChunk; o <<= 1) {      // inclusive max-scan of the run heads
        const int a = t >= o ? run0[t - o] : 0, b = run0[t + 512 - o];
        __syncthreads();
        run0[t] = max(run0[t], a);
        run0[t + 512] = max(run0[t + 512], b);
        __syncthreads();
    }
    if (t == 0) {
        while (atomicAdd(chain + 1, 0) < chunk) __nanosleep(64);
        __threadfence();
    }
    __syncthreads();
    int tail_c[2] = {-1, -1}, tail_v[2] = {0, 0};
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const int e = t + 512 * j;
        const uint32_t kk = key[e];
        if (kk == 0xFFFFFFFFu) continue;
        const int c = static_cast<int>(kk >> 10);
        const int rank = __ldcg(cursor + c) + (e - run0[e]);
        perm[seg_off[c] + rank] = static_cast<int>(base + (kk & 1023u));
        if (e == kSortChunk - 1 || (key[e + 1] >> 10) != (kk >> 10)) { tail_c[j] = c; tail_v[j] = rank + 1; }
    }
    __syncthreads();          // every read of a cursor precedes its update
#pragma unroll
    for (int j = 0; j < 2; ++j)
        if (tail_c[j] >= 0) __stcg(cursor + tail_c[j], tail_v[j]);
    __threadfence();
    __syncthreads();
    if (t == 0) atomicExch(chain + 1, chunk + 1);
}

// ---------------------------------------------------------------------------------------
// Category search work list (ofx_category_search), built on the device so that the entry point never
// synchronises and can be captured in a CUDA graph:
//   cat_query_count_kernel   queries per category
//   cat_plan_kernel          per category: groups of cl query blocks, tile ranges, units (one block)
//   cat_query_pack_kernel    each query's row in its category's blocks, and its bf16 copy there
// A range holds T = max(ceil(W / CTAs), 4) tiles, W = sum over categories of groups x tiles (the whole
// tensor-core sweep), and a segment has at most kMaxCatRanges ranges: a category with a single query group
// still spreads over ~tiles / T CTAs, and there are at most CTAs + groups units.  A category's units are
// ordered range-major, so the groups that sweep the same range run side by side and share its tiles in L2.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
cat_query_count_kernel(const int* __restrict__ q_cat, int n_query, int n_cat, int* __restrict__ qcnt) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n_query) return;
    const int c = q_cat[i];
    if (static_cast<unsigned>(c) < static_cast<unsigned>(n_cat)) atomicAdd(qcnt + c, 1);
}

__global__ void __launch_bounds__(1024)
cat_plan_kernel(const long long* __restrict__ seg_off, int n_cat, const int* __restrict__ qcnt, int cl, int n_cta,
                int* __restrict__ cat_g0, int4* __restrict__ units, int* __restrict__ grp, int* __restrict__ n_units) {
    __shared__ long long sh[1024];
    const int per = (n_cat + 1023) / 1024;
    const int c0 = min(n_cat, static_cast<int>(threadIdx.x) * per), c1 = min(n_cat, c0 + per);
    auto rows = [&](int c) { return seg_off[c + 1] - seg_off[c]; };
    auto groups = [&](int c) { return rows(c) > 0 ? (qcnt[c] + kBM * cl - 1) / (kBM * cl) : 0; };
    auto tiles = [&](int c) { return static_cast<int>((rows(c) + kSearchBN - 1) / kSearchBN); };
    long long w = 0, total;
    for (int c = c0; c < c1; ++c) w += static_cast<long long>(groups(c)) * tiles(c);
    block_exscan(w, sh, &total);
    const long long tpr = max((total + n_cta - 1) / n_cta, 4ll);
    auto ranges = [&](int c, int* len) {         // -> number of ranges, *len = tiles per range
        const int t = tiles(c);
        const int r = static_cast<int>(min(static_cast<long long>(kMaxCatRanges), max(1ll, (t + tpr - 1) / tpr)));
        *len = (t + r - 1) / r;
        return (t + *len - 1) / *len;
    };
    long long gs = 0, us = 0;
    for (int c = c0; c < c1; ++c) {
        const int g = groups(c);
        int len;
        if (g) { gs += g; us += static_cast<long long>(g) * ranges(c, &len); }
    }
    long long g_tot, u_tot;
    long long gb = block_exscan(gs, sh, &g_tot);
    long long ub = block_exscan(us, sh, &u_tot);
    for (int c = c0; c < c1; ++c) {
        const int g = groups(c);
        cat_g0[c] = g ? static_cast<int>(gb) : -1;
        if (!g) continue;
        int len;
        const int r = ranges(c, &len);
        const long long s_lo = seg_off[c], s_hi = seg_off[c + 1];
        const int m_end = static_cast<int>(gb) * cl * kBM + qcnt[c];      // the category's live query rows end here
        for (int j = 0; j < r; ++j) {
            const long long n_lo = s_lo + static_cast<long long>(j) * len * kSearchBN;
            const long long n_hi = min(s_hi, n_lo + static_cast<long long>(len) * kSearchBN);
            for (int i = 0; i < g; ++i)
                units[ub + static_cast<long long>(j) * g + i] =
                    make_int4(static_cast<int>(gb + i) * cl * kBM, m_end, static_cast<int>(n_lo), static_cast<int>(n_hi));
        }
        for (int i = 0; i < g; ++i) {
            grp[3 * (gb + i)] = static_cast<int>(ub + i);
            grp[3 * (gb + i) + 1] = g;
            grp[3 * (gb + i) + 2] = r;
        }
        gb += g;
        ub += static_cast<long long>(g) * r;
    }
    if (threadIdx.x == 0) *n_units = static_cast<int>(u_tot);
}

// one warp per query: its row in the category's blocks (-1: no row of its category here, or an id out of range)
// and the bf16 copy with the bias selector columns (as to_bf16_kernel)
__global__ void __launch_bounds__(256)
cat_query_pack_kernel(const float* __restrict__ queries, const int* __restrict__ q_cat, int n_query, int dim, int n_cat,
                      float aug, const int* __restrict__ cat_g0, int cl, int* __restrict__ qfill, int* __restrict__ qpos,
                      __nv_bfloat16* __restrict__ out) {
    const int q = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (q >= n_query) return;
    int pos = -1;
    if (lane == 0) {
        const int c = q_cat[q];
        if (static_cast<unsigned>(c) < static_cast<unsigned>(n_cat) && cat_g0[c] >= 0)
            pos = cat_g0[c] * cl * kBM + atomicAdd(qfill + c, 1);
        qpos[q] = pos;
    }
    pos = __shfl_sync(0xffffffffu, pos, 0);
    if (pos < 0) return;
    const int pitch = dim + kAugCols;
    for (int col = lane * 4; col < pitch; col += 128) {
        float4 v;
        if (col < dim) v = *reinterpret_cast<const float4*>(queries + static_cast<long long>(q) * dim + col);
        else v = col == dim ? make_float4(aug, aug, 0.f, 0.f) : make_float4(0.f, 0.f, 0.f, 0.f);
        __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
        uint2 u;
        u.x = *reinterpret_cast<uint32_t*>(&a);
        u.y = *reinterpret_cast<uint32_t*>(&b);
        *reinterpret_cast<uint2*>(out + static_cast<long long>(pos) * pitch + col) = u;
    }
}

// ---------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------
struct PackedGallery {
    size_t rows_bytes, stats, total;
};
static PackedGallery gallery_layout(long long n_rows, int dim) {
    PackedGallery g{};
    g.rows_bytes = align_up(static_cast<size_t>(n_rows) * (dim + kAugCols) * 2, 256);
    g.stats = g.rows_bytes + align_up(static_cast<size_t>(n_rows) * 4, 256);
    g.total = g.stats + 256;      // [0] max over the shard of 0.5|g|^2 (fp32), for the exactness certificate
    return g;
}

struct SearchWs {
    size_t q_bf16, thr, cand_n, cand_s, cand_i, prog, bm, hq, hist, total;
    int kcap;
    SearchPlan plan;
};
// List capacity of pass 1.  The certificate needs the k-th best EXACT score to clear the kcap-th best bf16 score by
// the worst-case bf16 error (~0.13 sigma of the score distribution at dim 1024); in the far tail of 10 M rows that
// takes kcap >= ~2 k, hence the generous steps.  k <= 12 keeps the 32-entry lists of the headline top-10 search.
static int kcap_for(int k) { return k <= 12 ? 32 : (k <= 25 ? 64 : 128); }
constexpr int kMaxK = 64;

static SearchWs search_ws(long long n_rows, int dim, int n_query, int k) {
    SearchWs w{};
    w.kcap = kcap_for(k);
    w.plan = make_plan(n_rows, n_query, sm_count());
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o = align_up(o + bytes, 256); return at; };
    const size_t slots = static_cast<size_t>(w.plan.n_units) * w.plan.cl * 128;
    w.q_bf16 = take(static_cast<size_t>(n_query) * (dim + kAugCols) * 2);
    w.thr = take(static_cast<size_t>(w.plan.n_qgroups) * w.plan.cl * 128 * 4);
    w.cand_n = take(slots * 4);
    w.cand_s = take(slots * w.kcap * 4);
    w.cand_i = take(slots * w.kcap * 4);
    w.prog = take(static_cast<size_t>(w.plan.n_units) * 4);
    const size_t q_pad = static_cast<size_t>(w.plan.n_qgroups) * w.plan.cl * 128;
    w.bm = take(q_pad * kSeedSegments * 2 * w.kcap * 4);     // pooled block maxima of the seeding sweep
    w.hq = take(q_pad * 16);
    w.hist = take(q_pad * kHistBuckets * 4);
    w.total = o;
    return w;
}

template <class Epi, int STAGES, int CL>
static int launch_search(const void* q_bf16, int n_query, const void* gallery, long long n_rows,
                         const SearchPlan& pl, const typename Epi::Params& ep, int dim,
                         cudaStream_t stream) {
    CUtensorMap tm_q, tm_g;
    const int kdim = dim + kAugCols;   // contraction length including the bias k-block
    OFX_TRY(make_tmap_bf16(&tm_q, q_bf16, static_cast<uint64_t>(n_query), kdim, kdim, kBM));
    OFX_TRY(make_tmap_bf16(&tm_g, gallery, static_cast<uint64_t>(n_rows), kdim, kdim, kSearchBN / CL));
    auto kern = tc_kernel<kSearchBN, STAGES, CL, SchedSearch, Epi>;   // CL = 2: CTA pair
    constexpr int smem = tc_smem_bytes<kSearchBN, STAGES, Epi, CL>();
    static_assert(smem <= 232448, "search kernel shared memory");
    static DeviceOnce configured;
    if (configured.need()) {
        OFX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    }
    if (ep.progress) OFX_CUDA(cudaMemsetAsync(ep.progress, 0xFF, static_cast<size_t>(pl.n_units) * 4, stream));
    SchedSearch::Params sp{pl.n_qgroups, pl.n_tiles, pl.seg_tiles, pl.n_units, CL, ep.progress};
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(pl.grid);
    cfg.blockDim = dim3(tc_threads<Epi>());
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    count_launch();
#ifdef OFX_DEBUG   // instrumented builds only (allocates + synchronises; see gemm.cu)
    static int prof_on = -1;
    static long long* prof_dev = nullptr;
    if (prof_on < 0) { const char* e = getenv("OFX_TC_PROF"); prof_on = (e && e[0] == '1') ? 1 : 0; }
    if (prof_on) {   // debug only: synchronous dump of per-CTA wait counters (tc_pipeline.cuh)
        if (!prof_dev) OFX_CUDA(cudaMalloc(&prof_dev, 8 * 8 * 256));
        OFX_CUDA(cudaMemsetAsync(prof_dev, 0, 8 * 8 * 256, stream));   // 2048 counters: 8 per CTA, timeline from 1199
        OFX_CUDA(cudaMemcpyToSymbolAsync(g_tc_prof, &prof_dev, sizeof(prof_dev), 0, cudaMemcpyHostToDevice, stream));
    }
#else
    constexpr int prof_on = 0;
    long long* const prof_dev = nullptr;
#endif
    OFX_CUDA(cudaLaunchKernelEx(&cfg, kern, tm_q, tm_g, sp, ep, kdim / kBK));
    if (prof_on) {
        long long h[8 * 256];
        OFX_CUDA(cudaStreamSynchronize(stream));
        OFX_CUDA(cudaMemcpy(h, prof_dev, sizeof(h), cudaMemcpyDeviceToHost));
        fprintf(stderr, "search prof nq=%d rows=%lld grid=%d cl=%d seg_tiles=%d: cta0 mma total %lld wait_full %lld wait_tmem_empty %lld | epi total %lld wait_tmem_full %lld ; cta100 mma %lld %lld %lld | epi %lld %lld\n",
                n_query, n_rows, pl.grid, CL, pl.seg_tiles, h[0], h[1], h[2], h[4], h[5], h[800], h[801], h[802], h[804], h[805]);
        // per-unit timeline of CTA 0's first epilogue warp: wall cycles, of which inside Epi::tile (busy includes the
        // wait share measured separately = waiting for the accumulator)
        for (int u = 0; u < h[1199] && u < 40; ++u)
            fprintf(stderr, "  unit %2d: %9lld cycles, epilogue tile() %9lld, waiting for tmem_full %9lld\n", u, h[1200 + 3 * u], h[1201 + 3 * u], h[1202 + 3 * u]);
    }
    return OFX_OK;
}

template <class Epi, int STAGES, int kPairStages>
static int launch_search_cl(const void* q_bf16, int n_query, const void* gallery, long long n_rows,
                            const SearchPlan& pl, const typename Epi::Params& ep, int dim,
                            cudaStream_t stream) {
    // CTA pairs (cta_group::2, M = 256: each CTA parks only half of the gallery tile, 32 KB stages, 6-deep ring)
    // beat a multicast cluster (both CTAs park the whole tile) once the pacing window removed the HBM traffic:
    // 133.4 vs 137.6 ms at 10 M rows, 20.4 vs 21.1 ms at 1.25 M.  (Before it the multicast cluster was ahead,
    // 1004 vs 940 TFLOP/s.)  What is left is L2 -> SM throughput: 1.39 TB per sweep = ~11 TB/s.
    if (pl.cl == 2) return launch_search<Epi, kPairStages, 2>(q_bf16, n_query, gallery, n_rows, pl, ep, dim, stream);
    return launch_search<Epi, STAGES, 1>(q_bf16, n_query, gallery, n_rows, pl, ep, dim, stream);
}

// ---------------------------------------------------------------------------------------
// category search, host side
// ---------------------------------------------------------------------------------------
// packed category gallery: bf16 rows in category order, then the scratch of the counting sort
struct CatGalleryLayout {
    size_t rows_bytes, cnt, cursor, chain, total;
};
static CatGalleryLayout cat_gallery_layout(long long n_rows, int dim, int n_cat) {
    CatGalleryLayout g{};
    g.rows_bytes = align_up(static_cast<size_t>(n_rows) * (dim + kAugCols) * 2, 256);
    g.cnt = g.rows_bytes;                                              // [n_cat + 1] rows per bin
    g.cursor = g.cnt + align_up(static_cast<size_t>(n_cat + 1) * 4, 256);   // [n_cat + 1] rows placed per bin
    g.chain = g.cursor + align_up(static_cast<size_t>(n_cat + 1) * 4, 256); // chunk ticket, chunks done
    g.total = g.chain + 256;
    return g;
}

// Workspace of ofx_category_search, sized for the worst case over the categories of the queries: a category
// with q queries takes ceil(q / (128 cl)) groups of cl query blocks <= q / 128 + 1, so there are at most
// ceil(n_query / 128) + min(n_query, n_cat) groups, and at most CTAs + groups units (cat_plan_kernel).
struct CatWs {
    size_t q_bf16, thr, cand_n, cand_s, cand_i, qcnt, cat_g0, qpos, units, grp, n_units, total;
    int kcap, cl, n_cta, max_units;
    long long q_rows;
};
static CatWs cat_ws(int dim, int n_cat, int n_query, int k) {
    CatWs w{};
    w.kcap = kcap_for(k);
    w.cl = 2;   // CTA pairs
    w.n_cta = sm_count() / w.cl;
    const long long groups = (n_query + kBM - 1) / kBM + (n_query < n_cat ? n_query : n_cat);
    w.q_rows = groups * w.cl * kBM;
    w.max_units = w.n_cta + static_cast<int>(groups);
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o = align_up(o + bytes, 256); return at; };
    const size_t slots = static_cast<size_t>(w.max_units) * w.cl * 128;
    w.q_bf16 = take(static_cast<size_t>(w.q_rows) * (dim + kAugCols) * 2);
    w.thr = take(static_cast<size_t>(w.q_rows) * 4);
    w.cand_n = take(slots * 4);
    w.cand_s = take(slots * w.kcap * 4);
    w.cand_i = take(slots * w.kcap * 4);
    w.qcnt = take(static_cast<size_t>(n_cat) * 8);      // queries per category, then queries placed per category
    w.cat_g0 = take(static_cast<size_t>(n_cat) * 4);
    w.qpos = take(static_cast<size_t>(n_query) * 4);
    w.units = take(static_cast<size_t>(w.max_units) * 16);
    w.grp = take(static_cast<size_t>(groups) * 12);
    w.n_units = take(4);
    w.total = o;
    return w;
}

// pass 1 of the category search: the same tcgen05 kernel as the flat search on the category schedule (CTA pairs);
// CTAs past the last unit leave at once
template <int KCAP, int STAGES, int CL>
static int launch_cat(const void* q_bf16, long long q_rows, const void* gallery, long long n_rows,
                      const SchedCat::Params& sp, int grid, const typename EpiTopK<KCAP, SchedCat>::Params& ep, int dim,
                      cudaStream_t stream) {
    using Epi = EpiTopK<KCAP, SchedCat>;
    CUtensorMap tm_q, tm_g;
    const int kdim = dim + kAugCols;
    OFX_TRY(make_tmap_bf16(&tm_q, q_bf16, static_cast<uint64_t>(q_rows), kdim, kdim, kBM));
    OFX_TRY(make_tmap_bf16(&tm_g, gallery, static_cast<uint64_t>(n_rows), kdim, kdim, kSearchBN / CL));
    auto kern = tc_kernel<kSearchBN, STAGES, CL, SchedCat, Epi>;
    constexpr int smem = tc_smem_bytes<kSearchBN, STAGES, Epi, CL>();
    static_assert(smem <= 232448, "search kernel shared memory");
    static DeviceOnce configured;
    if (configured.need()) OFX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(tc_threads<Epi>());
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    count_launch();
    OFX_CUDA(cudaLaunchKernelEx(&cfg, kern, tm_q, tm_g, sp, ep, kdim / kBK));
    return OFX_OK;
}

template <int KCAP, int STAGES, int kPairStages>
static int launch_cat_cl(int cl, const void* q_bf16, long long q_rows, const void* gallery, long long n_rows,
                         const SchedCat::Params& sp, int grid, const typename EpiTopK<KCAP, SchedCat>::Params& ep,
                         int dim, cudaStream_t stream) {
    if (cl == 2) return launch_cat<KCAP, kPairStages, 2>(q_bf16, q_rows, gallery, n_rows, sp, grid, ep, dim, stream);
    return launch_cat<KCAP, STAGES, 1>(q_bf16, q_rows, gallery, n_rows, sp, grid, ep, dim, stream);
}

}  // namespace ofx

using namespace ofx;

extern "C" {

size_t ofx_gallery_packed_bytes(int64_t n_rows, int32_t dim) {
    if (n_rows < 0 || dim <= 0) return 0;
    return gallery_layout(n_rows, dim).total;
}

int ofx_gallery_pack(const float* gallery, int64_t n_rows, int32_t dim, void* packed, void* stream) {
    if (n_rows < 0 || n_rows >= (1ll << 31)) return fail(OFX_E_SHAPE, "ofx_gallery_pack: n_rows %lld", (long long)n_rows);
    if (dim <= 0 || dim % 128) return fail(OFX_E_SHAPE, "ofx_gallery_pack: dim %d must be a multiple of 128", dim);
    if (n_rows == 0) return OFX_OK;
    if (!gallery || !packed) return fail(OFX_E_ARG, "ofx_gallery_pack: null argument");
    if (reinterpret_cast<uintptr_t>(gallery) % 16 || reinterpret_cast<uintptr_t>(packed) % 256)
        return fail(OFX_E_ARG, "ofx_gallery_pack: misaligned pointer (gallery 16 B, packed 256 B)");
    OFX_TRY(require_sm100());
    const PackedGallery L = gallery_layout(n_rows, dim);
    uint8_t* base = static_cast<uint8_t*>(packed);
    OFX_CUDA(cudaMemsetAsync(base + L.stats, 0, 256, static_cast<cudaStream_t>(stream)));
    gallery_pack_kernel<false><<<static_cast<unsigned>((n_rows + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        gallery, n_rows, dim, reinterpret_cast<__nv_bfloat16*>(base), reinterpret_cast<float*>(base + L.rows_bytes),
        reinterpret_cast<unsigned int*>(base + L.stats));
    OFX_LAUNCH_CHECK();
    return OFX_OK;
}

size_t ofx_search_workspace_bytes(int64_t n_rows, int32_t dim, int32_t n_query, int32_t k) {
    if (n_rows < 0 || dim <= 0 || n_query < 0 || k < 1 || k > kMaxK) return 0;
    return search_ws(n_rows, dim, n_query, k).total;
}

int ofx_topk_search(const void* packed, const float* gallery_f32, int64_t n_rows, int32_t dim,
                    int64_t id_offset, const float* queries, int32_t n_query, int32_t k, int32_t metric,
                    double* out_score, int64_t* out_idx, uint8_t* out_certified, void* workspace,
                    size_t workspace_bytes, void* stream) {
    if (k < 1 || k > kMaxK) return fail(OFX_E_SHAPE, "ofx_topk_search: k %d not in [1,%d]", k, kMaxK);
    if (dim <= 0 || dim % 128) return fail(OFX_E_SHAPE, "ofx_topk_search: dim %d must be a multiple of 128", dim);
    if (n_rows < 0 || n_rows >= (1ll << 31) - 256) return fail(OFX_E_SHAPE, "ofx_topk_search: n_rows %lld", (long long)n_rows);
    if (n_query < 0) return fail(OFX_E_SHAPE, "ofx_topk_search: n_query %d", n_query);
    if (metric != OFX_METRIC_DOT && metric != OFX_METRIC_L2) return fail(OFX_E_ARG, "ofx_topk_search: metric %d", metric);
    if (n_query == 0) return OFX_OK;
    if (!queries || !out_score || !out_idx) return fail(OFX_E_ARG, "ofx_topk_search: null argument");
    if (n_rows > 0 && !packed) return fail(OFX_E_ARG, "ofx_topk_search: packed gallery is null");
    if (reinterpret_cast<uintptr_t>(queries) % 16 || reinterpret_cast<uintptr_t>(packed) % 256 ||
        reinterpret_cast<uintptr_t>(workspace) % 256 || reinterpret_cast<uintptr_t>(gallery_f32) % 16)
        return fail(OFX_E_ARG, "ofx_topk_search: misaligned pointer");
    OFX_TRY(require_sm100());
    const SearchWs W = search_ws(n_rows, dim, n_query, k);
    if (!workspace || workspace_bytes < W.total)
        return fail(OFX_E_WORKSPACE, "workspace %zu B < required %zu B", workspace_bytes, W.total);
    if (W.plan.n_seg * W.kcap > 8192) return fail(OFX_E_SHAPE, "ofx_topk_search: candidate fan-in too large");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    const uint8_t* pk = static_cast<const uint8_t*>(packed);
    const PackedGallery L = gallery_layout(n_rows, dim);
    __nv_bfloat16* q_bf16 = reinterpret_cast<__nv_bfloat16*>(ws + W.q_bf16);
    uint32_t* thr = reinterpret_cast<uint32_t*>(ws + W.thr);
    int* cand_n = reinterpret_cast<int*>(ws + W.cand_n);
    float* cand_s = reinterpret_cast<float*>(ws + W.cand_s);
    int* cand_i = reinterpret_cast<int*>(ws + W.cand_i);
    int* prog = reinterpret_cast<int*>(ws + W.prog);

    if (n_rows > 0) {
        const long long nq_el = static_cast<long long>(n_query) * (dim + kAugCols);
        to_bf16_kernel<<<static_cast<unsigned>((nq_el / 4 + 255) / 256), 256, 0, st>>>(
            queries, n_query, dim, metric == OFX_METRIC_L2 ? 1.f : 0.f, q_bf16);
        OFX_LAUNCH_CHECK();
        OFX_CUDA(cudaMemsetAsync(thr, 0, static_cast<size_t>(W.plan.n_qgroups) * W.plan.cl * 128 * 4, st));
        // Threshold seeding (EpiBlockMax): the kcap-th largest of 2 kcap block maxima over the first rows is a
        // valid lower bound of every query's final kcap-th best, so the main sweep starts near the 0.5 %
        // quantile instead of cold and most of the divergent list insertions never happen.  A sample segment is
        // 2 kcap blocks of 128 rows; shards of fewer than 16 such segments are not seeded.
        const long long warm_rows = 8192LL * (W.kcap / 32);
        float* bm = reinterpret_cast<float*>(ws + W.bm);
        float4* hq = nullptr;
        uint32_t* hist = nullptr;
        if (n_rows >= 16 * warm_rows) {
            // same query blocks / cluster shape; one sample segment of warm_rows rows per idle CTA pair of a
            // query group (all units run in one wave), at most kSeedSegments and 1/16 of the shard
            SearchPlan wp = W.plan;
            const int n_cl = sm_count() / wp.cl;
            int n_seg = n_cl / (wp.n_qgroups > 0 ? wp.n_qgroups : 1);
            n_seg = n_seg < 1 ? 1 : (n_seg > kSeedSegments ? kSeedSegments : n_seg);
            while (n_seg > 1 && n_rows < 16 * warm_rows * n_seg) --n_seg;
            const long long sample_rows = warm_rows * n_seg;
            wp.seg_tiles = static_cast<int>(warm_rows / kSearchBN);
            wp.n_seg = n_seg;
            wp.n_tiles = wp.seg_tiles * n_seg;
            wp.n_units = wp.n_qgroups * n_seg;
            wp.grid = (wp.n_units < n_cl ? wp.n_units : n_cl) * wp.cl;
            const int nb_seg = static_cast<int>(warm_rows / 128), nb_total = nb_seg * n_seg;
            if (W.kcap == 32) {
                EpiBlockMax<64>::Params ep{sample_rows, n_query, prog, bm, nb_seg, nb_total};
                OFX_TRY((launch_search_cl<EpiBlockMax<64>, 4, 6>(q_bf16, n_query, pk, sample_rows, wp, ep, dim, st)));
            } else if (W.kcap == 64) {
                EpiBlockMax<128>::Params ep{sample_rows, n_query, prog, bm, nb_seg, nb_total};
                OFX_TRY((launch_search_cl<EpiBlockMax<128>, 3, 5>(q_bf16, n_query, pk, sample_rows, wp, ep, dim, st)));
            } else {
                EpiBlockMax<256>::Params ep{sample_rows, n_query, prog, bm, nb_seg, nb_total};
                OFX_TRY((launch_search_cl<EpiBlockMax<256>, 2, 3>(q_bf16, n_query, pk, sample_rows, wp, ep, dim, st)));
            }
            // every query gets a seeded bound and a sample maximum: the counting bound can run
            hq = reinterpret_cast<float4*>(ws + W.hq);
            hist = reinterpret_cast<uint32_t*>(ws + W.hist);
            seed_finish_kernel<<<(n_query + 7) / 8, 256, 0, st>>>(queries, n_query, dim, metric, bm, nb_total, W.kcap, thr,
                reinterpret_cast<const float*>(pk + L.stats), hq, hist);
            OFX_LAUNCH_CHECK();
        }
        if (W.kcap == 32) {
            EpiTopK<32>::Params ep{n_rows, n_query, thr, cand_s, cand_i, cand_n, prog, hist, hq, k};
            OFX_TRY((launch_search_cl<EpiTopK<32>, 4, 6>(q_bf16, n_query, pk, n_rows, W.plan, ep, dim, st)));
        } else if (W.kcap == 64) {
            EpiTopK<64>::Params ep{n_rows, n_query, thr, cand_s, cand_i, cand_n, prog, hist, hq, k};
            OFX_TRY((launch_search_cl<EpiTopK<64>, 3, 5>(q_bf16, n_query, pk, n_rows, W.plan, ep, dim, st)));
        } else {
            EpiTopK<128>::Params ep{n_rows, n_query, thr, cand_s, cand_i, cand_n, prog, hist, hq, k};
            OFX_TRY((launch_search_cl<EpiTopK<128>, 2, 3>(q_bf16, n_query, pk, n_rows, W.plan, ep, dim, st)));
        }
    }
    MergeArgs ma{};
    ma.cand_s = cand_s; ma.cand_i = cand_i; ma.cand_n = cand_n;
    ma.kcap = W.kcap; ma.n_seg = W.plan.n_seg; ma.n_qgroups = W.plan.n_qgroups; ma.cl = W.plan.cl;
    int n_pad = 2;
    while (n_pad < W.plan.n_seg * W.kcap) n_pad <<= 1;
    ma.n_pad = n_pad;
    ma.queries = queries; ma.gallery_f32 = gallery_f32; ma.dim = dim; ma.metric = metric; ma.k = k;
    ma.id_offset = id_offset; ma.out_score = out_score; ma.out_idx = reinterpret_cast<long long*>(out_idx);
    ma.thr_enc = n_rows > 0 ? thr : nullptr;
    ma.max_half_sqnorm = reinterpret_cast<const float*>(pk + L.stats);
    ma.certified = out_certified;
#ifdef OFX_DEBUG   // instrumented builds only (allocates + synchronises)
    static int merge_prof = -1;
    static unsigned long long* merge_prof_dev = nullptr;
    if (merge_prof < 0) { const char* e = getenv("OFX_MERGE_PROF"); merge_prof = (e && e[0] == '1') ? 1 : 0; }
    if (merge_prof) {
        if (!merge_prof_dev) OFX_CUDA(cudaMalloc(&merge_prof_dev, 64));
        OFX_CUDA(cudaMemsetAsync(merge_prof_dev, 0, 64, st));
    }
#else
    constexpr int merge_prof = 0;
    unsigned long long* const merge_prof_dev = nullptr;
#endif
    ma.prof = merge_prof ? merge_prof_dev : nullptr;
    const size_t smem = static_cast<size_t>(n_pad + kMergeSmall) * 8;
    static DeviceOnce configured;
    if (configured.need()) {
        OFX_CUDA(cudaFuncSetAttribute(merge_rerank_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (8192 + kMergeSmall) * 8));
    }
    merge_rerank_kernel<false><<<n_query, kMergeThreads, smem, st>>>(ma);
    OFX_LAUNCH_CHECK();
    if (merge_prof) {     // debug only: synchronous dump
        unsigned long long h[8];
        OFX_CUDA(cudaStreamSynchronize(st));
        OFX_CUDA(cudaMemcpy(h, merge_prof_dev, 64, cudaMemcpyDeviceToHost));
        fprintf(stderr, "merge prof (avg cycles per query CTA): gather %llu  sort %llu  re-score %llu ; full sorts %llu of %d ; n_pad %d n_seg %d\n",
                h[0] / n_query, h[1] / n_query, h[2] / n_query, h[4], n_query, n_pad, W.plan.n_seg);
    }
    return OFX_OK;
}

static int exact_chunks(long long n_rows, int k) {
    long long c = (n_rows + 2047) / 2048;             // at least 2048 rows per chunk
    const long long cap = 2048 / k < 128 ? 2048 / k : 128;     // topk_merge_kernel takes n_lists * k <= 2048
    if (c > cap) c = cap;
    return c < 1 ? 1 : static_cast<int>(c);
}

size_t ofx_exact_search_workspace_bytes(int64_t n_rows, int32_t n_sel, int32_t k) {
    if (n_rows < 0 || n_sel < 0 || k < 1 || k > kMaxK) return 0;
    return align_up(static_cast<size_t>(exact_chunks(n_rows, k)) * n_sel * k * 16, 256) + 256;
}

// The exhaustive fp64 fallback of both searches.  cat: xc describes the category layout, every selected query
// scans only its category's segment (one query per CTA row) and ids map through xc.perm.
static int exact_search(const char* who, bool cat, const ExactCat& xc, const float* gallery_f32, int64_t n_rows,
                        int32_t dim, int64_t id_offset, const float* queries, const int32_t* sel, int32_t n_sel,
                        int32_t k, int32_t metric, double* out_score, int64_t* out_idx, uint8_t* out_certified,
                        void* workspace, size_t workspace_bytes, void* stream) {
    if (k < 1 || k > kMaxK) return fail(OFX_E_SHAPE, "%s: k %d not in [1,%d]", who, k, kMaxK);
    if (dim <= 0 || dim % 4 || dim > 4096) return fail(OFX_E_SHAPE, "%s: dim %d (multiple of 4, <= 4096)", who, dim);
    if (n_rows < 0 || n_sel < 0) return fail(OFX_E_SHAPE, "%s: n_rows %lld, n_sel %d", who, (long long)n_rows, n_sel);
    if (metric != OFX_METRIC_DOT && metric != OFX_METRIC_L2) return fail(OFX_E_ARG, "%s: metric %d", who, metric);
    if (n_sel == 0) return OFX_OK;
    if (!queries || !sel || !out_score || !out_idx || (n_rows > 0 && !gallery_f32)) return fail(OFX_E_ARG, "%s: null argument", who);
    if (reinterpret_cast<uintptr_t>(gallery_f32) % 16 || reinterpret_cast<uintptr_t>(queries) % 16 || reinterpret_cast<uintptr_t>(workspace) % 256)
        return fail(OFX_E_ARG, "%s: misaligned pointer", who);
    const size_t need = ofx_exact_search_workspace_bytes(n_rows, n_sel, k);
    if (!workspace || workspace_bytes < need) return fail(OFX_E_WORKSPACE, "workspace %zu B < required %zu B", workspace_bytes, need);
    OFX_TRY(require_sm100());
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int chunks = exact_chunks(n_rows, k);
    const size_t n_part = static_cast<size_t>(chunks) * n_sel * k;
    double* part_s = static_cast<double*>(workspace);
    long long* part_i = reinterpret_cast<long long*>(part_s + n_part);
    // padding: idx -1 (0xFF..), score bits 0xFF.. = NaN, never read for idx < 0
    OFX_CUDA(cudaMemsetAsync(workspace, 0xFF, n_part * 16, st));
    const long long rows_per_chunk = (n_rows + chunks - 1) / chunks;
    const size_t smem = sizeof(float) * kExactQ * dim + static_cast<size_t>(kExactWarps) * kExactQ * k * 16;
    const int smem_max = static_cast<int>(sizeof(float) * kExactQ * 4096 + kExactWarps * kExactQ * kMaxK * 16);
    static DeviceOnce configured;
    if (configured.need()) {
        OFX_CUDA(cudaFuncSetAttribute(exact_scan_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
        OFX_CUDA(cudaFuncSetAttribute(exact_scan_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
    }
    if (n_rows > 0) {
        if (cat)
            exact_scan_kernel<true><<<dim3(n_sel, chunks), kExactWarps * 32, smem, st>>>(
                gallery_f32, n_rows, dim, metric, queries, sel, n_sel, k, 1, part_s, part_i, xc);
        else
            exact_scan_kernel<false><<<dim3(chunks, (n_sel + kExactQ - 1) / kExactQ), kExactWarps * 32, smem, st>>>(
                gallery_f32, n_rows, dim, metric, queries, sel, n_sel, k, rows_per_chunk > 0 ? rows_per_chunk : 1, part_s, part_i, xc);
        OFX_LAUNCH_CHECK();
    }
    topk_merge_kernel<<<n_sel, 128, static_cast<size_t>(chunks) * k * 16, st>>>(
        part_s, part_i, chunks, n_sel, k, out_score, reinterpret_cast<long long*>(out_idx), sel);
    OFX_LAUNCH_CHECK();
    if (cat)
        add_offset_kernel<true><<<(n_sel * k + 255) / 256, 256, 0, st>>>(reinterpret_cast<long long*>(out_idx), sel, n_sel, k, id_offset, out_certified, xc.perm);
    else
        add_offset_kernel<false><<<(n_sel * k + 255) / 256, 256, 0, st>>>(reinterpret_cast<long long*>(out_idx), sel, n_sel, k, id_offset, out_certified, nullptr);
    OFX_LAUNCH_CHECK();
    return OFX_OK;
}

int ofx_exact_search(const float* gallery_f32, int64_t n_rows, int32_t dim, int64_t id_offset,
                     const float* queries, const int32_t* sel, int32_t n_sel, int32_t k, int32_t metric,
                     double* out_score, int64_t* out_idx, uint8_t* out_certified, void* workspace,
                     size_t workspace_bytes, void* stream) {
    return exact_search("ofx_exact_search", false, ExactCat{}, gallery_f32, n_rows, dim, id_offset, queries, sel, n_sel,
                        k, metric, out_score, out_idx, out_certified, workspace, workspace_bytes, stream);
}

int ofx_category_exact_search(const float* gallery_f32, const int32_t* perm, const int64_t* seg_off,
                              int32_t n_categories, int64_t n_rows, int32_t dim, int64_t id_offset,
                              const float* queries, const int32_t* query_category, const int32_t* sel, int32_t n_sel,
                              int32_t k, int32_t metric, double* out_score, int64_t* out_idx, uint8_t* out_certified,
                              void* workspace, size_t workspace_bytes, void* stream) {
    if (n_categories < 1 || n_categories > kMaxCategories)
        return fail(OFX_E_SHAPE, "ofx_category_exact_search: n_categories %d not in [1,%d]", n_categories, kMaxCategories);
    if (n_sel > 0 && (!seg_off || !query_category || (n_rows > 0 && !perm)))
        return fail(OFX_E_ARG, "ofx_category_exact_search: null argument");
    const ExactCat xc{perm, reinterpret_cast<const long long*>(seg_off), query_category, n_categories};
    return exact_search("ofx_category_exact_search", true, xc, gallery_f32, n_rows, dim, id_offset, queries, sel, n_sel,
                        k, metric, out_score, out_idx, out_certified, workspace, workspace_bytes, stream);
}

int ofx_topk_merge(const double* scores, const int64_t* idx, int32_t n_lists, int32_t n_query, int32_t k,
                   double* out_score, int64_t* out_idx, void* stream) {
    if (n_lists < 1 || k < 1 || n_query < 0 || static_cast<long long>(n_lists) * k > 2048)
        return fail(OFX_E_SHAPE, "ofx_topk_merge: n_lists %d, k %d", n_lists, k);
    if (n_query == 0) return OFX_OK;
    if (!scores || !idx || !out_score || !out_idx) return fail(OFX_E_ARG, "ofx_topk_merge: null argument");
    OFX_TRY(require_sm100());
    const size_t smem = static_cast<size_t>(n_lists) * k * 16;
    topk_merge_kernel<<<n_query, 128, smem, static_cast<cudaStream_t>(stream)>>>(
        scores, reinterpret_cast<const long long*>(idx), n_lists, n_query, k, out_score,
        reinterpret_cast<long long*>(out_idx));
    OFX_LAUNCH_CHECK();
    return OFX_OK;
}

size_t ofx_category_gallery_packed_bytes(int64_t n_rows, int32_t dim, int32_t n_categories) {
    if (n_rows < 0 || dim <= 0 || n_categories < 1 || n_categories > kMaxCategories) return 0;
    return cat_gallery_layout(n_rows, dim, n_categories).total;
}

int ofx_category_gallery_pack(const float* gallery, const int32_t* categories, int64_t n_rows, int32_t dim,
                              int32_t n_categories, void* packed, int32_t* perm, int64_t* seg_off,
                              float* cat_max_half_sqnorm, void* stream) {
    if (n_rows < 0 || n_rows >= (1ll << 31) - 256)
        return fail(OFX_E_SHAPE, "ofx_category_gallery_pack: n_rows %lld", (long long)n_rows);
    if (dim <= 0 || dim % 128) return fail(OFX_E_SHAPE, "ofx_category_gallery_pack: dim %d must be a multiple of 128", dim);
    if (n_categories < 1 || n_categories > kMaxCategories)
        return fail(OFX_E_SHAPE, "ofx_category_gallery_pack: n_categories %d not in [1,%d]", n_categories, kMaxCategories);
    if (!packed || !seg_off || !cat_max_half_sqnorm || (n_rows > 0 && (!gallery || !categories || !perm)))
        return fail(OFX_E_ARG, "ofx_category_gallery_pack: null argument");
    if (reinterpret_cast<uintptr_t>(gallery) % 16 || reinterpret_cast<uintptr_t>(packed) % 256)
        return fail(OFX_E_ARG, "ofx_category_gallery_pack: misaligned pointer (gallery 16 B, packed 256 B)");
    OFX_TRY(require_sm100());
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const CatGalleryLayout L = cat_gallery_layout(n_rows, dim, n_categories);
    uint8_t* base = static_cast<uint8_t*>(packed);
    int* cnt = reinterpret_cast<int*>(base + L.cnt);
    OFX_CUDA(cudaMemsetAsync(base + L.cnt, 0, L.total - L.cnt, st));
    OFX_CUDA(cudaMemsetAsync(cat_max_half_sqnorm, 0, static_cast<size_t>(n_categories) * 4, st));
    if (n_rows > 0) {
        cat_count_kernel<<<static_cast<unsigned>((n_rows + 255) / 256), 256, 0, st>>>(categories, n_rows, n_categories, cnt);
        OFX_LAUNCH_CHECK();
    }
    cat_scan_kernel<<<1, 1024, 0, st>>>(cnt, n_categories + 1, reinterpret_cast<long long*>(seg_off));
    OFX_LAUNCH_CHECK();
    if (n_rows == 0) return OFX_OK;
    cat_sort_kernel<<<static_cast<unsigned>((n_rows + kSortChunk - 1) / kSortChunk), 512, 0, st>>>(
        categories, n_rows, n_categories, reinterpret_cast<const long long*>(seg_off), reinterpret_cast<int*>(base + L.cursor),
        reinterpret_cast<int*>(base + L.chain), perm);
    OFX_LAUNCH_CHECK();
    gallery_pack_kernel<true><<<static_cast<unsigned>((n_rows + 7) / 8), 256, 0, st>>>(
        gallery, n_rows, dim, reinterpret_cast<__nv_bfloat16*>(base), nullptr,
        reinterpret_cast<unsigned int*>(cat_max_half_sqnorm), perm, categories, n_categories);
    OFX_LAUNCH_CHECK();
    return OFX_OK;
}

size_t ofx_category_search_workspace_bytes(int32_t dim, int32_t n_categories, int32_t n_query, int32_t k) {
    if (dim <= 0 || n_query < 0 || k < 1 || k > kMaxK || n_categories < 1 || n_categories > kMaxCategories) return 0;
    const CatWs W = cat_ws(dim, n_categories, n_query, k);
    return W.q_rows >= (1ll << 31) ? 0 : W.total;
}

int ofx_category_search(const void* packed, const int32_t* perm, const int64_t* seg_off, const float* cat_max_half_sqnorm,
                        int32_t n_categories, const float* gallery_f32, int64_t n_rows, int32_t dim, int64_t id_offset,
                        const float* queries, const int32_t* query_category, int32_t n_query, int32_t k, int32_t metric,
                        double* out_score, int64_t* out_idx, uint8_t* out_certified, void* workspace,
                        size_t workspace_bytes, void* stream) {
    if (k < 1 || k > kMaxK) return fail(OFX_E_SHAPE, "ofx_category_search: k %d not in [1,%d]", k, kMaxK);
    if (dim <= 0 || dim % 128) return fail(OFX_E_SHAPE, "ofx_category_search: dim %d must be a multiple of 128", dim);
    if (n_rows < 0 || n_rows >= (1ll << 31) - 256) return fail(OFX_E_SHAPE, "ofx_category_search: n_rows %lld", (long long)n_rows);
    if (n_query < 0) return fail(OFX_E_SHAPE, "ofx_category_search: n_query %d", n_query);
    if (n_categories < 1 || n_categories > kMaxCategories)
        return fail(OFX_E_SHAPE, "ofx_category_search: n_categories %d not in [1,%d]", n_categories, kMaxCategories);
    if (metric != OFX_METRIC_DOT && metric != OFX_METRIC_L2) return fail(OFX_E_ARG, "ofx_category_search: metric %d", metric);
    if (n_query == 0) return OFX_OK;
    if (!queries || !query_category || !out_score || !out_idx || !seg_off || !cat_max_half_sqnorm ||
        (n_rows > 0 && (!packed || !perm)))
        return fail(OFX_E_ARG, "ofx_category_search: null argument");
    if (reinterpret_cast<uintptr_t>(queries) % 16 || reinterpret_cast<uintptr_t>(packed) % 256 ||
        reinterpret_cast<uintptr_t>(workspace) % 256 || reinterpret_cast<uintptr_t>(gallery_f32) % 16)
        return fail(OFX_E_ARG, "ofx_category_search: misaligned pointer");
    OFX_TRY(require_sm100());
    const CatWs W = cat_ws(dim, n_categories, n_query, k);
    if (W.q_rows >= (1ll << 31)) return fail(OFX_E_SHAPE, "ofx_category_search: n_query %d too large", n_query);
    if (!workspace || workspace_bytes < W.total)
        return fail(OFX_E_WORKSPACE, "workspace %zu B < required %zu B", workspace_bytes, W.total);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint8_t* ws = static_cast<uint8_t*>(workspace);
    __nv_bfloat16* q_bf16 = reinterpret_cast<__nv_bfloat16*>(ws + W.q_bf16);
    uint32_t* thr = reinterpret_cast<uint32_t*>(ws + W.thr);
    int* cand_n = reinterpret_cast<int*>(ws + W.cand_n);
    float* cand_s = reinterpret_cast<float*>(ws + W.cand_s);
    int* cand_i = reinterpret_cast<int*>(ws + W.cand_i);
    int* qcnt = reinterpret_cast<int*>(ws + W.qcnt);
    int* cat_g0 = reinterpret_cast<int*>(ws + W.cat_g0);
    int* qpos = reinterpret_cast<int*>(ws + W.qpos);
    int4* units = reinterpret_cast<int4*>(ws + W.units);
    int* grp = reinterpret_cast<int*>(ws + W.grp);
    int* n_units = reinterpret_cast<int*>(ws + W.n_units);
    const long long* seg = reinterpret_cast<const long long*>(seg_off);

    OFX_CUDA(cudaMemsetAsync(qcnt, 0, static_cast<size_t>(n_categories) * 8, st));
    OFX_CUDA(cudaMemsetAsync(thr, 0, static_cast<size_t>(W.q_rows) * 4, st));
    cat_query_count_kernel<<<(n_query + 255) / 256, 256, 0, st>>>(query_category, n_query, n_categories, qcnt);
    OFX_LAUNCH_CHECK();
    cat_plan_kernel<<<1, 1024, 0, st>>>(seg, n_categories, qcnt, W.cl, W.n_cta, cat_g0, units, grp, n_units);
    OFX_LAUNCH_CHECK();
    cat_query_pack_kernel<<<(n_query + 7) / 8, 256, 0, st>>>(queries, query_category, n_query, dim, n_categories,
        metric == OFX_METRIC_L2 ? 1.f : 0.f, cat_g0, W.cl, qcnt + n_categories, qpos, q_bf16);
    OFX_LAUNCH_CHECK();
    if (n_rows > 0) {
        const SchedCat::Params sp{units, n_units, W.cl};
        const int grid = W.n_cta * W.cl;
        if (W.kcap == 32) {
            EpiTopK<32, SchedCat>::Params ep{n_rows, n_query, thr, cand_s, cand_i, cand_n, nullptr, nullptr, nullptr, k};
            OFX_TRY((launch_cat_cl<32, 4, 6>(W.cl, q_bf16, W.q_rows, packed, n_rows, sp, grid, ep, dim, st)));
        } else if (W.kcap == 64) {
            EpiTopK<64, SchedCat>::Params ep{n_rows, n_query, thr, cand_s, cand_i, cand_n, nullptr, nullptr, nullptr, k};
            OFX_TRY((launch_cat_cl<64, 3, 5>(W.cl, q_bf16, W.q_rows, packed, n_rows, sp, grid, ep, dim, st)));
        } else {
            EpiTopK<128, SchedCat>::Params ep{n_rows, n_query, thr, cand_s, cand_i, cand_n, nullptr, nullptr, nullptr, k};
            OFX_TRY((launch_cat_cl<128, 2, 3>(W.cl, q_bf16, W.q_rows, packed, n_rows, sp, grid, ep, dim, st)));
        }
    }
    MergeArgs ma{};
    ma.cand_s = cand_s; ma.cand_i = cand_i; ma.cand_n = cand_n;
    ma.kcap = W.kcap; ma.cl = W.cl;
    int n_pad = 2;
    while (n_pad < kMaxCatRanges * W.kcap) n_pad <<= 1;
    ma.n_pad = n_pad;
    ma.queries = queries; ma.gallery_f32 = gallery_f32; ma.dim = dim; ma.metric = metric; ma.k = k;
    ma.id_offset = id_offset; ma.out_score = out_score; ma.out_idx = reinterpret_cast<long long*>(out_idx);
    ma.thr_enc = n_rows > 0 ? thr : nullptr;
    ma.max_half_sqnorm = cat_max_half_sqnorm;
    ma.certified = out_certified;
    ma.qpos = qpos; ma.grp = grp; ma.perm = perm; ma.q_cat = query_category;
    static DeviceOnce configured;
    if (configured.need())
        OFX_CUDA(cudaFuncSetAttribute(merge_rerank_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (8192 + kMergeSmall) * 8));
    merge_rerank_kernel<true><<<n_query, kMergeThreads, static_cast<size_t>(n_pad + kMergeSmall) * 8, st>>>(ma);
    OFX_LAUNCH_CHECK();
    return OFX_OK;
}
}
