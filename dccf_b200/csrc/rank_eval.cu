// rank_eval.cu — kernel (d) of the DCCF hot path: per-user top-k over the candidate list (positives +
// test_neg_n sampled negatives) and the ranking metrics at every requested k, in ONE launch.
//
// Replaces the ranking branch of BaseModel.evaluate_method (src/models/BaseModel.py:82-126:
// global pandas sort by score, groupby uid, one Python loop per user PER METRIC) and the helpers it
// calls, src/utils/rank_metrics.py:61-87 (precision_at_k) and :130-201 (dcg_at_k / ndcg_at_k, method=1).
//
// k_rank_stream (k <= 16): one warp per user, ONE streaming pass over the user's candidates: lane l reads
// candidates l, l+32, ... (coalesced, eight loads in flight), stages the scores in shared memory and keeps only its
// maximum.  The k-th largest of the 32 lane maxima is a threshold no member of the top k can be below; a second
// pass over shared memory compacts the survivors (typically k .. 3k of 1001) with ballots, and only those get
// their item ids loaded and are ordered exactly (score desc, item id asc, row asc) by k shuffle tournaments.
// About six instructions per candidate.  (Two earlier designs, kept out: k selection rounds over global memory —
// 2k+1 passes, 110-145 us per 1 024 users; per-lane sorted top-k lists in registers — one pass, but ~1 700
// instructions per candidate-iteration of divergent insertion code, 52 us.)  Users with more candidates than the
// staging buffer, or with more than 128 candidates tied at the threshold, take the general selection rounds.
// Labels are read once: total relevance, number of positives (ideal DCG of 0/1 labels is a count; graded labels
// take selection rounds over the labels), and the labels of the k winners.  Every metric (ndcg, hit, precision,
// recall, f1) at every requested k (up to 4 values of k per launch) comes out of that one pass; per-user values are
// optional, the per-metric SUMS over users are accumulated in a fixed order (warp -> CTA -> last CTA), so a metric
// list such as "ndcg@5,recall@5,precision@5" costs one launch and one 120-byte read-back.
// Order: score descending, then item id ascending, then row ascending — a total order, so the result is
// deterministic (the reference's quicksort leaves ties unordered).  NaN scores rank last, as pandas does.
// k_rank_select (any k <= 1024): the k-rounds selection kernel, kept for k > 16.
// k_topk_metrics: the same metrics for full-catalogue top-k lists (dccf_full_scores with known-item exclusion) against
// each user's held-out positives, summed over users in the same fixed order.
#include <math.h>

#include "common.cuh"

namespace dccf {

struct RankKey {
    float s;
    int64_t iid;
    int32_t row;
    float label;
};

// true when a ranks strictly before b
__device__ __forceinline__ bool key_before(const RankKey& a, const RankKey& b) {
    if (a.s != b.s) return a.s > b.s;
    if (a.iid != b.iid) return a.iid < b.iid;
    return a.row < b.row;
}

__device__ __forceinline__ RankKey shfl_key(const RankKey& k, int src_xor) {
    RankKey o;
    o.s = __shfl_xor_sync(0xffffffffu, k.s, src_xor);
    o.iid = __shfl_xor_sync(0xffffffffu, k.iid, src_xor);
    o.row = __shfl_xor_sync(0xffffffffu, k.row, src_xor);
    o.label = __shfl_xor_sync(0xffffffffu, k.label, src_xor);
    return o;
}

__device__ __forceinline__ float order_score(float s) { return (s != s) ? -INFINITY : s; }

constexpr int RANK_WARPS = 4;
constexpr int RANK_MAX_NK = 4;       // values of k per launch
constexpr int RANK_NCOL = 5;         // ndcg, hit, precision, recall, f1
constexpr int RANK_STREAM_MAX_K = 16;

struct RankKs {
    int32_t k[RANK_MAX_NK];
    int32_t n_k, kmax;
};

// log2(t + 2) for the first RANK_STREAM_MAX_K rank positions, as float64 (filled by the host: std::log2 of the exact
// integers, the values np.log2 gives): a table instead of a software FP64 log2 per position and user
__constant__ double c_log2_pos[16];
__constant__ double c_inv_log2_pos[16];      // 1 / log2(t + 2), correctly rounded (host division)

constexpr int RANK_CHUNK = 2048;     // candidates of one user staged in shared memory (8 KB per warp); more: fallback
constexpr int RANK_SURV = 128;       // survivors of the threshold test kept per user; more (massive ties): fallback

__device__ __forceinline__ RankKey key_sentinel() {
    RankKey k;
    k.s = -INFINITY; k.iid = INT64_MAX; k.row = INT32_MAX; k.label = 0.f;      // after every real candidate
    return k;
}

// warp-wide best of one key per lane (lanes without a candidate carry the sentinel)
__device__ __forceinline__ RankKey warp_best(RankKey best) {
#pragma unroll 1
    for (int o = 16; o > 0; o >>= 1) {
        const RankKey other = shfl_key(best, o);
        if (key_before(other, best)) best = other;
    }
    return best;
}

// The general selection: kk rounds of "best key strictly after the previous winner" over the user's candidates in
// global memory (L1 / L2 after the streaming pass).  Used when a user has more candidates than the staging buffer or
// when the threshold test leaves too many survivors (massive score ties).  Lane t returns winner t.
__device__ __forceinline__ RankKey select_rounds(const float* __restrict__ scores, const int64_t* __restrict__ iids,
                                                 const int32_t* __restrict__ cand_rows, int64_t lo, int64_t hi, int kk,
                                                 int lane) {
    RankKey mine = key_sentinel(), last;
    last.s = INFINITY; last.iid = -1; last.row = -1; last.label = 0.f;
#pragma unroll 1
    for (int t = 0; t < kk; ++t) {
        RankKey best = key_sentinel();
#pragma unroll 1
        for (int64_t c = lo + lane; c < hi; c += 32) {
            RankKey cur;
            cur.row = cand_rows != nullptr ? __ldg(cand_rows + c) : (int32_t)c;
            cur.s = order_score(__ldg(scores + cur.row));
            cur.label = 0.f;
            if (cur.s > last.s || cur.s < best.s) continue;          // not after the last winner / cannot beat the best
            cur.iid = __ldg(iids + cur.row);
            if ((t == 0 || key_before(last, cur)) && key_before(cur, best)) best = cur;
        }
        best = warp_best(best);
        if (lane == t) mine = best;
        last = best;
    }
    return mine;
}

__global__ void __launch_bounds__(RANK_WARPS * 32) k_rank_stream(
    const float* __restrict__ scores, const float* __restrict__ labels, const int64_t* __restrict__ iids,
    const int32_t* __restrict__ cand_rows, const int64_t* __restrict__ user_off, int64_t n_users, const RankKs ks,
    int64_t* __restrict__ out_topk_iid, int32_t* __restrict__ out_topk_row, double* __restrict__ out_metrics,
    double* __restrict__ part_sums, int32_t* __restrict__ cta_counter, double* __restrict__ out_sums) {
    __shared__ double acc_s[RANK_WARPS][RANK_MAX_NK * RANK_NCOL];
    __shared__ float sc_s[RANK_WARPS][RANK_CHUNK];
    __shared__ int32_t surv_s[RANK_WARPS][RANK_SURV];
    __shared__ int s_last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ncol = ks.n_k * RANK_NCOL;
    if (lane < RANK_MAX_NK * RANK_NCOL) acc_s[warp][lane] = 0.0;
    __syncwarp();
    const int kmax = ks.kmax;
    const int64_t n_warps = (int64_t)gridDim.x * RANK_WARPS;
    float* my_s = sc_s[warp];
    int32_t* my_surv = surv_s[warp];
    const uint32_t lt_mask = (1u << lane) - 1u;

    for (int64_t g = (int64_t)blockIdx.x * RANK_WARPS + warp; g < n_users; g += n_warps) {   // warp-uniform
        const int64_t lo = user_off[g], hi = user_off[g + 1];
        const int64_t n = hi - lo;
        const int kk = (int)min((int64_t)kmax, n);
        const bool fits = n <= RANK_CHUNK;
        double label_sum = 0.0;
        int n_pos = 0;
        bool nonbinary = false;
        float lane_max = -INFINITY;

        // ---- phase 1, the streaming pass: scores -> shared memory, the lane's maximum, label statistics.  All of a
        // 1001-candidate user's loads are in flight at once (32 scores + 32 labels per lane): ONE memory round trip per
        // user instead of four — with one warp per user the pass is bound by that latency, not by bandwidth.
        constexpr int NF = 32;
        for (int64_t c0 = lo + lane; c0 < hi; c0 += 32 * NF) {
            int32_t row[NF];
            float s[NF], l[NF];
#pragma unroll
            for (int j = 0; j < NF; ++j) {
                const int64_t c = c0 + 32 * j;
                row[j] = (c < hi) ? (cand_rows != nullptr ? __ldg(cand_rows + c) : (int32_t)c) : -1;
            }
#pragma unroll
            for (int j = 0; j < NF; ++j) {
                if (row[j] >= 0) {
                    s[j] = __ldg(scores + row[j]);
                    l[j] = __ldg(labels + row[j]);
                }
            }
#pragma unroll
            for (int j = 0; j < NF; ++j) {
                if (row[j] >= 0) {
                    const float os = order_score(s[j]);
                    if (fits) my_s[c0 - lo + 32 * j] = os;
                    lane_max = fmaxf(lane_max, os);
                    label_sum += (double)l[j];
                    n_pos += (l[j] == 1.f) ? 1 : 0;
                    nonbinary |= (l[j] != 0.f && l[j] != 1.f);
                }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            label_sum += __shfl_xor_sync(0xffffffffu, label_sum, o);
            n_pos += __shfl_xor_sync(0xffffffffu, n_pos, o);
        }
        nonbinary = __any_sync(0xffffffffu, nonbinary);
        __syncwarp();

        RankKey mine = key_sentinel();     // lane t: the candidate at rank t
        bool have = false;                 // warp-uniform
        if (fits) {
            // ---- phase 2, a threshold nothing in the top kk can be below: the kk-th largest of the 32 lane maxima
            // (kk distinct candidates are >= it) ----
            float lm = lane_max, thr = -INFINITY;
#pragma unroll 1
            for (int t = 0; t < kk; ++t) {
                thr = warp_max(lm);
                if (thr == -INFINITY) break;
                const uint32_t b = __ballot_sync(0xffffffffu, lm == thr);
                if (lane == __ffs(b) - 1) lm = -INFINITY;
            }
            // ---- phase 3, the survivors (score >= threshold: typically kk .. 3 kk of the 1001), compacted in candidate
            // order by ballots ----
            int n_s = 0;
#pragma unroll 1
            for (int c = lane; c < (int)((n + 31) & ~(int64_t)31); c += 32) {
                const bool pred = c < n && my_s[c] >= thr;
                const uint32_t m = __ballot_sync(0xffffffffu, pred);
                if (pred) {
                    const int pos = n_s + __popc(m & lt_mask);
                    if (pos < RANK_SURV) my_surv[pos] = c;
                }
                n_s += __popc(m);
            }
            __syncwarp();
            if (n_s <= RANK_SURV) {
                // ---- phase 4, exact order of the survivors (score desc, item id asc, row asc): each lane holds up to
                // four of them, kk tournaments, the winning lane retires its entry ----
                RankKey key[RANK_SURV / 32];
#pragma unroll
                for (int q = 0; q < RANK_SURV / 32; ++q) {
                    key[q] = key_sentinel();
                    const int j = lane + 32 * q;
                    if (j < n_s) {
                        const int c = my_surv[j];
                        key[q].row = cand_rows != nullptr ? __ldg(cand_rows + lo + c) : (int32_t)(lo + c);
                        key[q].s = my_s[c];
                        key[q].iid = __ldg(iids + key[q].row);
                    }
                }
#pragma unroll 1
                for (int t = 0; t < kk; ++t) {
                    RankKey best = key[0];
#pragma unroll
                    for (int q = 1; q < RANK_SURV / 32; ++q)
                        if (key_before(key[q], best)) best = key[q];
                    best = warp_best(best);
#pragma unroll
                    for (int q = 0; q < RANK_SURV / 32; ++q)
                        if (key[q].row == best.row) key[q] = key_sentinel();      // rows are unique: one entry retires
                    if (lane == t) mine = best;
                }
                have = true;
            }
        }
        if (!have) mine = select_rounds(scores, iids, cand_rows, lo, hi, kk, lane);
        const float my_label = (lane < kk) ? __ldg(labels + mine.row) : 0.f;
        if (out_topk_iid != nullptr && lane < kmax) out_topk_iid[g * kmax + lane] = (lane < kk) ? mine.iid : -1;
        if (out_topk_row != nullptr && lane < kmax) out_topk_row[g * kmax + lane] = (lane < kk) ? mine.row : -1;

        // ---- ideal ordering of the labels: 0/1 labels -> the first n_pos positions are 1; otherwise the kmax
        // largest labels by a second pass (values only) --------------------------------------------------------
        float ideal = (lane < min(kk, n_pos)) ? 1.f : 0.f;    // lane t: label at ideal position t
        if (nonbinary) {                                       // warp-uniform
            // graded labels: kk rounds of "largest label after the previous one" over (label desc, position asc)
            ideal = 0.f;
            float last_l = INFINITY;
            int64_t last_c = -1;
#pragma unroll 1
            for (int t = 0; t < kk; ++t) {
                float best_l = -INFINITY;
                int64_t best_c = -1;
#pragma unroll 1
                for (int64_t c = lo + lane; c < hi; c += 32) {
                    const float l = __ldg(labels + (cand_rows != nullptr ? __ldg(cand_rows + c) : (int32_t)c));
                    const bool below = (t == 0) || (l < last_l) || (l == last_l && c > last_c);
                    if (below && (best_c < 0 || l > best_l || (l == best_l && c < best_c))) {
                        best_l = l;
                        best_c = c;
                    }
                }
#pragma unroll 1
                for (int o = 16; o > 0; o >>= 1) {
                    const float ol = __shfl_xor_sync(0xffffffffu, best_l, o);
                    const int64_t oc = __shfl_xor_sync(0xffffffffu, best_c, o);
                    if (oc >= 0 && (best_c < 0 || ol > best_l || (ol == best_l && oc < best_c))) {
                        best_l = ol;
                        best_c = oc;
                    }
                }
                if (lane == t) ideal = best_l;
                last_l = best_l;
                last_c = best_c;
            }
        }

        // ---- metrics at every requested k: sequential float64 sums over positions 0 .. k-1 ---------------
        double dcg = 0.0, idcg = 0.0, hit_sum = 0.0;
        int nonzero = 0, next_k = 0;
#pragma unroll 1
        for (int t = 0; t < kmax; ++t) {
            const float lab = __shfl_sync(0xffffffffu, my_label, t);
            const float idl = __shfl_sync(0xffffffffu, ideal, t);
            if (t < kk) {
                // rel / log2(position + 1), rank_metrics.py:160.  0/1 labels (the ranking path's labels) take the tabulated
                // reciprocal — 1 / x is the correctly rounded quotient either way, so the bits are those of the division;
                // graded labels divide.  (The software FP64 division was half of the kernel's instructions.)
                const double disc = c_log2_pos[t], inv = c_inv_log2_pos[t];
                dcg += (lab == 0.f) ? 0.0 : (lab == 1.f ? inv : (double)lab / disc);
                idcg += (idl == 0.f) ? 0.0 : (idl == 1.f ? inv : (double)idl / disc);
                hit_sum += (double)lab;
                nonzero += (lab != 0.f) ? 1 : 0;
            }
            while (next_k < ks.n_k && ks.k[next_k] == t + 1) {     // ks ascending
                if (lane == 0) {
                    const double k = (double)(t + 1);
                    double m[RANK_NCOL];
                    m[0] = (idcg != 0.0) ? dcg / idcg : 0.0;                    // ndcg@k   (rank_metrics.py:198-201)
                    m[1] = (hit_sum > 0.0) ? 1.0 : 0.0;                         // hit@k    (BaseModel.py:98-102)
                    m[2] = (double)nonzero / k;                                 // precision@k (rank_metrics.py:83-87)
                    m[3] = hit_sum / label_sum;                                 // recall@k (BaseModel.py:108-112)
                    m[4] = 2.0 * hit_sum / (k + label_sum);                     // f1@k     (BaseModel.py:121-126)
#pragma unroll
                    for (int q = 0; q < RANK_NCOL; ++q) {
                        if (out_metrics != nullptr) out_metrics[(g * ks.n_k + next_k) * RANK_NCOL + q] = m[q];
                        acc_s[warp][next_k * RANK_NCOL + q] += m[q];
                    }
                }
                ++next_k;
            }
        }
        __syncwarp();
    }

    // ---- sums over users in a fixed order: warps of the CTA, then (last CTA) the CTAs in index order ------
    if (out_sums == nullptr) return;
    __syncthreads();
    if ((int)threadIdx.x < ncol) {
        double v = 0.0;
        for (int w = 0; w < RANK_WARPS; ++w) v += acc_s[w][threadIdx.x];
        part_sums[(size_t)blockIdx.x * (RANK_MAX_NK * RANK_NCOL) + threadIdx.x] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const int32_t prev = atomicAdd(cta_counter, 1);
        s_last = (prev == (int32_t)gridDim.x - 1) ? 1 : 0;
        if (s_last) {
            __threadfence();
            *cta_counter = 0;
        }
    }
    __syncthreads();
    if (!s_last) return;
    // warp w sums columns w, w + RANK_WARPS, ...: lane-strided over the CTAs (ascending), then a shuffle tree
    for (int col = warp; col < ncol; col += RANK_WARPS) {
        double v = 0.0;
        for (int b = lane; b < (int)gridDim.x; b += 32) v += __ldcg(part_sums + (size_t)b * (RANK_MAX_NK * RANK_NCOL) + col);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) out_sums[col] = v;
    }
}

// The k-rounds selection kernel (k > 16): each round finds the best key strictly below the previous winner.
__global__ void __launch_bounds__(RANK_WARPS * 32) k_rank_select(
    const float* __restrict__ scores, const float* __restrict__ labels, const int64_t* __restrict__ iids,
    const int32_t* __restrict__ cand_rows, const int64_t* __restrict__ user_off, int64_t n_users, int32_t k,
    int64_t* __restrict__ out_topk_iid, int32_t* __restrict__ out_topk_row, double* __restrict__ out_metrics) {
    const int lane = threadIdx.x & 31;
    const int64_t g = (int64_t)blockIdx.x * RANK_WARPS + (threadIdx.x >> 5);
    if (g >= n_users) return;  // warp-uniform
    const int64_t lo = user_off[g], hi = user_off[g + 1];
    const int64_t n = hi - lo;
    auto row_of = [&](int64_t c) { return cand_rows != nullptr ? cand_rows[c] : (int32_t)c; };

    double label_sum = 0.0;
    for (int64_t c = lo + lane; c < hi; c += 32) label_sum += (double)__ldg(labels + row_of(c));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) label_sum += __shfl_xor_sync(0xffffffffu, label_sum, o);

    const int kk = (int)min((int64_t)k, n);
    double idcg = 0.0;
    {
        float last_l = INFINITY;
        int64_t last_c = -1;
        for (int t = 0; t < kk; ++t) {
            float best_l = -INFINITY;
            int64_t best_c = -1;
            for (int64_t c = lo + lane; c < hi; c += 32) {
                const float l = __ldg(labels + row_of(c));
                const bool below = (t == 0) || (l < last_l) || (l == last_l && c > last_c);
                if (below && (best_c < 0 || l > best_l || (l == best_l && c < best_c))) {
                    best_l = l;
                    best_c = c;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ol = __shfl_xor_sync(0xffffffffu, best_l, o);
                const int64_t oc = __shfl_xor_sync(0xffffffffu, best_c, o);
                if (oc >= 0 && (best_c < 0 || ol > best_l || (ol == best_l && oc < best_c))) {
                    best_l = ol;
                    best_c = oc;
                }
            }
            idcg += (double)best_l / log2((double)(t + 2));
            last_l = best_l;
            last_c = best_c;
        }
    }

    double dcg = 0.0, hit_sum = 0.0;
    int nonzero = 0;
    RankKey last;
    last.s = INFINITY; last.iid = -1; last.row = -1; last.label = 0.f;
    for (int t = 0; t < k; ++t) {
        RankKey best;
        best.s = -INFINITY; best.iid = INT64_MAX; best.row = INT32_MAX; best.label = 0.f;
        bool have = false;
        if (t < kk) {
            for (int64_t c = lo + lane; c < hi; c += 32) {
                RankKey cur;
                cur.row = row_of(c);
                cur.s = order_score(__ldg(scores + cur.row));
                cur.iid = __ldg(iids + cur.row);
                const bool below = (t == 0) || key_before(last, cur);
                if (below && (!have || key_before(cur, best))) {
                    best = cur;
                    have = true;
                }
            }
            if (!have) { best.s = -INFINITY; best.iid = INT64_MAX; best.row = INT32_MAX; }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const RankKey other = shfl_key(best, o);
                if (other.row != INT32_MAX && (best.row == INT32_MAX || key_before(other, best))) best = other;
            }
            best.label = __ldg(labels + best.row);
            dcg += (double)best.label / log2((double)(t + 2));
            hit_sum += (double)best.label;
            nonzero += (best.label != 0.f) ? 1 : 0;
            last = best;
        }
        if (lane == 0) {
            if (out_topk_iid) out_topk_iid[g * k + t] = (t < kk) ? best.iid : -1;
            if (out_topk_row) out_topk_row[g * k + t] = (t < kk) ? best.row : -1;
        }
    }

    if (lane == 0) {
        double* o = out_metrics + g * RANK_NCOL;
        o[0] = (idcg != 0.0) ? dcg / idcg : 0.0;
        o[1] = (hit_sum > 0.0) ? 1.0 : 0.0;
        o[2] = (double)nonzero / (double)k;
        o[3] = hit_sum / label_sum;
        o[4] = 2.0 * hit_sum / ((double)k + label_sum);
    }
}

// Metrics of ranked full-catalogue lists: one warp per user, lane t looks up the item at rank t in the user's sorted
// positives (binary search; the list has at most 16 entries, the positives are few).  The label at rank t is 1 for a hit;
// the ideal list puts the n_pos positives first.  Per-user values, per-warp accumulation and the sums over users follow
// k_rank_stream exactly (its code is repeated here, not shared, so that the ranker's instructions stay what they are).
__global__ void __launch_bounds__(RANK_WARPS * 32) k_topk_metrics(
    const int64_t* __restrict__ topk_id, int64_t n_users, int32_t k_list, const int64_t* __restrict__ pos_off,
    const int32_t* __restrict__ pos_items, const RankKs ks, double* __restrict__ out_metrics,
    double* __restrict__ part_sums, int32_t* __restrict__ cta_counter, double* __restrict__ out_sums,
    unsigned long long* __restrict__ out_count) {
    __shared__ double acc_s[RANK_WARPS][RANK_MAX_NK * RANK_NCOL];
    __shared__ int s_last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ncol = ks.n_k * RANK_NCOL;
    if (lane < RANK_MAX_NK * RANK_NCOL) acc_s[warp][lane] = 0.0;
    __syncwarp();
    const int kmax = ks.kmax;
    const int64_t n_warps = (int64_t)gridDim.x * RANK_WARPS;
    unsigned long long counted = 0;

    for (int64_t g = (int64_t)blockIdx.x * RANK_WARPS + warp; g < n_users; g += n_warps) {   // warp-uniform
        const int64_t lo = pos_off[g], hi = pos_off[g + 1];
        const int64_t n_pos = hi - lo;
        if (n_pos <= 0) {
            if (out_metrics != nullptr && lane < ncol) out_metrics[g * ncol + lane] = __longlong_as_double(0x7ff8000000000000LL);
            continue;
        }
        float my_label = 0.f;
        if (lane < k_list) {
            const int64_t id = __ldg(topk_id + g * k_list + lane);
            if (id >= 0) {
                int64_t a = lo, b = hi;
                while (a < b) {
                    const int64_t mid = (a + b) >> 1;
                    if ((int64_t)__ldg(pos_items + mid) < id) a = mid + 1; else b = mid;
                }
                my_label = (a < hi && (int64_t)__ldg(pos_items + a) == id) ? 1.f : 0.f;
            }
        }
        double dcg = 0.0, idcg = 0.0, hit_sum = 0.0;
        int next_k = 0;
#pragma unroll 1
        for (int t = 0; t < kmax; ++t) {
            const float lab = __shfl_sync(0xffffffffu, my_label, t);
            const double inv = c_inv_log2_pos[t];
            dcg += (lab == 0.f) ? 0.0 : inv;
            idcg += (t < n_pos) ? inv : 0.0;
            hit_sum += (double)lab;
            while (next_k < ks.n_k && ks.k[next_k] == t + 1) {     // ks ascending
                if (lane == 0) {
                    const double k = (double)(t + 1), np = (double)n_pos;
                    double m[RANK_NCOL];
                    m[0] = dcg / idcg;                  // idcg > 0: n_pos >= 1
                    m[1] = (hit_sum > 0.0) ? 1.0 : 0.0;
                    m[2] = hit_sum / k;
                    m[3] = hit_sum / np;
                    m[4] = 2.0 * hit_sum / (k + np);
#pragma unroll
                    for (int q = 0; q < RANK_NCOL; ++q) {
                        if (out_metrics != nullptr) out_metrics[(g * ks.n_k + next_k) * RANK_NCOL + q] = m[q];
                        acc_s[warp][next_k * RANK_NCOL + q] += m[q];
                    }
                }
                ++next_k;
            }
        }
        ++counted;
        __syncwarp();
    }
    if (out_count != nullptr && lane == 0 && counted > 0) atomicAdd(out_count, counted);    // integer: order-free

    // ---- sums over users in a fixed order: warps of the CTA, then (last CTA) the CTAs in index order ------
    if (out_sums == nullptr) return;
    __syncthreads();
    if ((int)threadIdx.x < ncol) {
        double v = 0.0;
        for (int w = 0; w < RANK_WARPS; ++w) v += acc_s[w][threadIdx.x];
        part_sums[(size_t)blockIdx.x * (RANK_MAX_NK * RANK_NCOL) + threadIdx.x] = v;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const int32_t prev = atomicAdd(cta_counter, 1);
        s_last = (prev == (int32_t)gridDim.x - 1) ? 1 : 0;
        if (s_last) {
            __threadfence();
            *cta_counter = 0;
        }
    }
    __syncthreads();
    if (!s_last) return;
    for (int col = warp; col < ncol; col += RANK_WARPS) {
        double v = 0.0;
        for (int b = lane; b < (int)gridDim.x; b += 32) v += __ldcg(part_sums + (size_t)b * (RANK_MAX_NK * RANK_NCOL) + col);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) out_sums[col] = v;
    }
}

}  // namespace dccf

using namespace dccf;

// the c_log2_pos / c_inv_log2_pos tables, once per device
static int install_log2_tables(const char* who) {
    static PerDeviceOnce table_once;
    if (!table_once.need()) return DCCF_OK;
    double h[16], hi[16];
    for (int t = 0; t < 16; ++t) {
        h[t] = log2((double)(t + 2));
        hi[t] = 1.0 / h[t];
    }
    cudaError_t e = cudaMemcpyToSymbol(c_log2_pos, h, sizeof(h));
    if (e == cudaSuccess) e = cudaMemcpyToSymbol(c_inv_log2_pos, hi, sizeof(hi));
    if (e != cudaSuccess) {
        set_error("%s: cannot install the log2 table: %s", who, cudaGetErrorString(e));
        return DCCF_ERR_CUDA;
    }
    table_once.mark();
    return DCCF_OK;
}

extern "C" int64_t dccf_rank_eval_ws_bytes(int64_t n_users) {
    (void)n_users;
    // partial sums of at most 148 * 4 CTAs + the CTA counter
    return (int64_t)(148 * 4) * RANK_MAX_NK * RANK_NCOL * (int64_t)sizeof(double) + 16;
}

extern "C" int dccf_rank_eval_multi(const float* scores, const float* labels, const int64_t* iids, const int32_t* cand_rows,
                                    const int64_t* user_off, int64_t n_users, const int32_t* ks_host, int32_t n_k,
                                    int64_t* out_topk_iid, int32_t* out_topk_row, double* out_metrics, void* ws,
                                    double* out_sums, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    DCCF_CHECK_ARG(scores && labels && iids && user_off, "dccf_rank_eval_multi: null buffer");
    DCCF_CHECK_ARG(ks_host && n_k >= 1 && n_k <= RANK_MAX_NK, "dccf_rank_eval_multi: 1 to %d values of k per call", RANK_MAX_NK);
    DCCF_CHECK_ARG(out_metrics || out_sums, "dccf_rank_eval_multi: no output requested");
    DCCF_CHECK_ARG(out_sums == nullptr || ws != nullptr, "dccf_rank_eval_multi: the sums need the workspace (dccf_rank_eval_ws_bytes)");
    RankKs ks;
    ks.n_k = n_k;
    for (int i = 0; i < RANK_MAX_NK; ++i) ks.k[i] = 0;
    for (int i = 0; i < n_k; ++i) {
        DCCF_CHECK_ARG(ks_host[i] >= 1 && ks_host[i] <= RANK_STREAM_MAX_K, "dccf_rank_eval_multi: k=%d outside [1,%d]", ks_host[i], RANK_STREAM_MAX_K);
        DCCF_CHECK_ARG(i == 0 || ks_host[i] > ks_host[i - 1], "dccf_rank_eval_multi: the values of k must be strictly ascending");
        ks.k[i] = ks_host[i];
    }
    ks.kmax = ks.k[n_k - 1];
    if (n_users <= 0) {
        if (out_sums) cudaMemsetAsync(out_sums, 0, sizeof(double) * n_k * RANK_NCOL, stream);
        return DCCF_OK;
    }
    const int rc = install_log2_tables("dccf_rank_eval_multi");
    if (rc != DCCF_OK) return rc;
    int64_t ctas = (n_users + RANK_WARPS - 1) / RANK_WARPS;
    if (ctas > 148 * 4) ctas = 148 * 4;
    double* part = reinterpret_cast<double*>(ws);
    int32_t* counter = ws ? reinterpret_cast<int32_t*>(reinterpret_cast<uint8_t*>(ws) + (size_t)(148 * 4) * RANK_MAX_NK * RANK_NCOL * sizeof(double)) : nullptr;
    k_rank_stream<<<(unsigned)ctas, RANK_WARPS * 32, 0, stream>>>(scores, labels, iids, cand_rows, user_off, n_users, ks,
                                                                  out_topk_iid, out_topk_row, out_metrics, part, counter,
                                                                  out_sums);
    DCCF_CHECK_LAUNCH("k_rank_stream");
    return DCCF_OK;
}

extern "C" int dccf_rank_eval(const float* scores, const float* labels, const int64_t* iids, const int32_t* cand_rows,
                              const int64_t* user_off, int64_t n_users, int32_t k, int64_t* out_topk_iid,
                              int32_t* out_topk_row, double* out_metrics, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    DCCF_CHECK_ARG(scores && labels && iids && user_off && out_metrics, "dccf_rank_eval: null buffer");
    DCCF_CHECK_ARG(k >= 1 && k <= 1024, "dccf_rank_eval: k=%d outside [1,1024]", k);
    if (n_users <= 0) return DCCF_OK;
    if (k <= RANK_STREAM_MAX_K)
        return dccf_rank_eval_multi(scores, labels, iids, cand_rows, user_off, n_users, &k, 1, out_topk_iid, out_topk_row,
                                    out_metrics, nullptr, nullptr, stream_);
    k_rank_select<<<(unsigned)((n_users + RANK_WARPS - 1) / RANK_WARPS), RANK_WARPS * 32, 0, stream>>>(
        scores, labels, iids, cand_rows, user_off, n_users, k, out_topk_iid, out_topk_row, out_metrics);
    DCCF_CHECK_LAUNCH("k_rank_select");
    return DCCF_OK;
}

extern "C" int dccf_topk_metrics(const int64_t* topk_id, int64_t n_users, int32_t k_list, const int64_t* pos_off,
                                 const int32_t* pos_items, const int32_t* ks_host, int32_t n_k, double* out_metrics, void* ws,
                                 double* out_sums, int64_t* out_count, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    DCCF_CHECK_ARG(topk_id && pos_off, "dccf_topk_metrics: null buffer");
    DCCF_CHECK_ARG(k_list >= 1 && k_list <= RANK_STREAM_MAX_K, "dccf_topk_metrics: list length %d outside [1,%d]", k_list, RANK_STREAM_MAX_K);
    DCCF_CHECK_ARG(ks_host && n_k >= 1 && n_k <= RANK_MAX_NK, "dccf_topk_metrics: 1 to %d values of k per call", RANK_MAX_NK);
    DCCF_CHECK_ARG(out_metrics || out_sums || out_count, "dccf_topk_metrics: no output requested");
    DCCF_CHECK_ARG(out_sums == nullptr || ws != nullptr, "dccf_topk_metrics: the sums need the workspace (dccf_rank_eval_ws_bytes)");
    RankKs ks;
    ks.n_k = n_k;
    for (int i = 0; i < RANK_MAX_NK; ++i) ks.k[i] = 0;
    for (int i = 0; i < n_k; ++i) {
        DCCF_CHECK_ARG(ks_host[i] >= 1 && ks_host[i] <= k_list, "dccf_topk_metrics: k=%d outside [1,%d] (the list length)", ks_host[i], k_list);
        DCCF_CHECK_ARG(i == 0 || ks_host[i] > ks_host[i - 1], "dccf_topk_metrics: the values of k must be strictly ascending");
        ks.k[i] = ks_host[i];
    }
    ks.kmax = ks.k[n_k - 1];
    if (out_count) {
        const cudaError_t e = cudaMemsetAsync(out_count, 0, sizeof(int64_t), stream);
        if (e != cudaSuccess) {
            set_error("dccf_topk_metrics: cannot clear the user count: %s", cudaGetErrorString(e));
            return DCCF_ERR_CUDA;
        }
    }
    if (n_users <= 0) {
        if (out_sums) cudaMemsetAsync(out_sums, 0, sizeof(double) * n_k * RANK_NCOL, stream);
        return DCCF_OK;
    }
    const int rc = install_log2_tables("dccf_topk_metrics");
    if (rc != DCCF_OK) return rc;
    int64_t ctas = (n_users + RANK_WARPS - 1) / RANK_WARPS;
    if (ctas > 148 * 4) ctas = 148 * 4;
    double* part = reinterpret_cast<double*>(ws);
    int32_t* counter = ws ? reinterpret_cast<int32_t*>(reinterpret_cast<uint8_t*>(ws) + (size_t)(148 * 4) * RANK_MAX_NK * RANK_NCOL * sizeof(double)) : nullptr;
    k_topk_metrics<<<(unsigned)ctas, RANK_WARPS * 32, 0, stream>>>(topk_id, n_users, k_list, pos_off, pos_items, ks, out_metrics,
                                                                   part, counter, out_sums,
                                                                   reinterpret_cast<unsigned long long*>(out_count));
    DCCF_CHECK_LAUNCH("k_topk_metrics");
    return DCCF_OK;
}
