// adam.cu — kernel (c) part 2 of the DCCF hot path: l2 + clip + Adam, dense over every parameter.
//
// Replaces, per training step of the reference:
//   loss += l2 * model.l2()              src/runners/BaseRunner.py:181, src/models/BaseModel.py:179-187
//   clip_grad_value_(params, 50)          src/runners/BaseRunner.py:185
//   Adam(lr, weight_decay=l2).step()      src/runners/BaseRunner.py:100,187  (torch 2.11 optim/adam.py,
//                                         _multi_tensor_adam, non-capturable branch)
//   or SGD / Adagrad(lr, weight_decay=l2)  src/runners/BaseRunner.py:83-98 (rule_elem below)
// which together put a non-zero gradient on EVERY row of both embedding tables each step, so the
// update is a full streaming sweep (Adam 24 B/param: read p,m,v, write p,m,v; Adagrad 16; GD 8).  The sparse part of the
// gradient arrives as records (row id + 64 floats) linked per row through head/next; records of one
// row are summed in ascending record order so the result does not depend on atomics timing.
#include "common.cuh"
#include "backdoor.cuh"
#include "dp_sync.cuh"

namespace dccf {

struct AdamScalars {
    float w1;          // 1 - beta1 (lerp weight)
    float beta2;       // beta2
    float omb2;        // 1 - beta2
    float step_size;   // -(lr / (1 - beta1^t))
    float bc2_sqrt;    // sqrt(1 - beta2^t)
    float inv_bc2_sqrt;
    float eps;
    float two_l2;      // 2 * l2
    float wd;          // weight decay
    float clip;        // <= 0: off
};

struct AdamHost {
    double lr, beta1, beta2;
    float eps, l2, wd, clip;
    int32_t step;
    const int32_t* step_dev;
};

__device__ __forceinline__ AdamScalars resolve_adam(const AdamHost& h) {
    const int32_t t = (h.step_dev != nullptr) ? __ldg(h.step_dev) : h.step;
    AdamScalars s;
    s.w1 = (float)(1.0 - h.beta1);
    s.beta2 = (float)h.beta2;
    s.omb2 = (float)(1.0 - h.beta2);
    const double bc1 = 1.0 - pow(h.beta1, (double)t);
    const double bc2 = 1.0 - pow(h.beta2, (double)t);
    s.step_size = (float)(-(h.lr / bc1));
    s.bc2_sqrt = (float)sqrt(bc2);
    s.inv_bc2_sqrt = (float)(1.0 / sqrt(bc2));
    s.eps = h.eps;
    s.two_l2 = 2.0f * h.l2;
    s.wd = h.wd;
    s.clip = h.clip;
    return s;
}

// clip_grad_value_: clamp to [-clip, clip], NaN stays NaN as in torch.clamp (fmaxf / fminf would turn it into -clip, and
// a diverged step would go on with finite parameters).  The .NaN forms of max / min cost what fmaxf / fminf cost; finite
// values and +-inf clip as before.
__device__ __forceinline__ float clip_value(float g, float clip) {
    float r;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(g), "f"(-clip));
    asm("min.NaN.f32 %0, %0, %1;" : "+f"(r) : "f"(clip));
    return r;
}

// one element of the update; g_sparse is the data-dependent part of the gradient
__device__ __forceinline__ void adam_elem(float& p, float& m, float& v, float g_sparse, const AdamScalars& s) {
    float g = __fadd_rn(g_sparse, __fmul_rn(s.two_l2, p));       // + d/dp (l2 * sum p^2)
    if (s.clip > 0.f) g = clip_value(g, s.clip);                 // clip_grad_value_
    g = fmaf(s.wd, p, g);                                        // Adam weight_decay: g + wd * p
    m = fmaf(s.w1, __fsub_rn(g, m), m);                          // exp_avg.lerp_(g, 1 - beta1)
    v = __fmul_rn(v, s.beta2);                                   // exp_avg_sq.mul_(beta2)
    v = fmaf(__fmul_rn(s.omb2, g), g, v);                        //   .addcmul_(g, g, value = 1 - beta2)
    // denom = sqrt(v)/sqrt(bc2) + eps ; p += step_size * m / denom.  The sweep is HBM-bound only if the
    // arithmetic stays short: sqrt and the division use the hardware approximations (MUFU.SQRT, MUFU.RCP;
    // <= 2 ulp each) and the per-step constant divides by multiplication.  The update term is <= lr relative
    // to the step size, so this perturbs p by ~1e-7 * lr — four orders below the 1e-5 parity bound; exp_avg
    // and exp_avg_sq above follow torch's IEEE arithmetic exactly.
    float sq;
    asm("sqrt.approx.f32 %0, %1;" : "=f"(sq) : "f"(v));
    const float denom = fmaf(sq, s.inv_bc2_sqrt, s.eps);
    p = fmaf(s.step_size, __fdividef(m, denom), p);              // param.addcdiv_(exp_avg, denom, value = step_size)
}

// The optimizer rule (dccf_adam.rule) is a compile-time parameter of the step kernels below.  A rule streams only the
// state it has: Adam exp_avg (m) and exp_avg_sq (v), Adagrad state_sum (in m), GD none.
enum : int { RULE_ADAM = 0, RULE_GD = 1, RULE_ADAGRAD = 2 };
template <int R> constexpr bool rule_has_m = R != RULE_GD;
template <int R> constexpr bool rule_has_v = R == RULE_ADAM;

// GD and Adagrad need no per-step constant beyond lr (lr_decay = 0): step_size = -lr
template <int R> __device__ __forceinline__ AdamScalars resolve_rule(const AdamHost& h) {
    if constexpr (R == RULE_ADAM) {
        return resolve_adam(h);
    } else {
        AdamScalars s = {};
        s.step_size = (float)(-h.lr);
        s.eps = h.eps;
        s.two_l2 = 2.0f * h.l2;
        s.wd = h.wd;
        s.clip = h.clip;
        return s;
    }
}

template <int R> __device__ __forceinline__ void rule_elem(float& p, float& m, float& v, float g_sparse, const AdamScalars& s) {
    if constexpr (R == RULE_ADAM) {
        adam_elem(p, m, v, g_sparse, s);
    } else {
        float g = __fadd_rn(g_sparse, __fmul_rn(s.two_l2, p));   // same preamble as adam_elem
        if (s.clip > 0.f) g = clip_value(g, s.clip);
        g = fmaf(s.wd, p, g);                                    // weight_decay: g + wd * p
        if constexpr (R == RULE_GD) {
            p = fmaf(s.step_size, g, p);                         // SGD: param.add_(g, alpha = -lr)
        } else {
            m = fmaf(g, g, m);                                   // Adagrad: state_sum.addcmul_(g, g, value = 1)
            // std = sqrt(state_sum) + eps ; p += -lr * g / std.  Since state_sum >= g^2, |g| / std <= 1 and the step is
            // at most lr; MUFU.SQRT and MUFU.RCP (<= 2 ulp each) perturb it by ~4e-7 relative, i.e. by ~4e-7 * lr in p —
            // far below the 1e-5 parity bound.  state_sum itself is exact IEEE arithmetic.
            float sq;
            asm("sqrt.approx.f32 %0, %1;" : "=f"(sq) : "f"(m));
            p = fmaf(s.step_size, __fdividef(g, __fadd_rn(sq, s.eps)), p);
        }
    }
}

template <int R> __device__ __forceinline__ void rule_elem4(float4& p, float4& m, float4& v, const float4& g,
                                                            const AdamScalars& s) {
    rule_elem<R>(p.x, m.x, v.x, g.x, s); rule_elem<R>(p.y, m.y, v.y, g.y, s);
    rule_elem<R>(p.z, m.z, v.z, g.z, s); rule_elem<R>(p.w, m.w, v.w, g.w, s);
}

// loads / stores of one state tensor that are compiled away for a rule without it
template <bool On> __device__ __forceinline__ float4 ld4_if(const float* p) {
    if constexpr (On) return ld4(p); else return make_float4(0.f, 0.f, 0.f, 0.f);
}
template <bool On> __device__ __forceinline__ void st4_if(float* p, const float4& v) {
    if constexpr (On) st4(p, v);
}

// Records may arrive in n_seg segments of seg_len records each (one segment per data-parallel rank after the
// all-gather): record r lives in segment r / seg_len at local index r % seg_len.
struct RecLayout {
    int64_t seg_len;
    int64_t key_seg_stride;   // int32 elements between the key arrays of consecutive segments
    int64_t grad_seg_stride;  // floats between the gradient arrays of consecutive segments
};
__device__ __forceinline__ size_t rec_key_index(const RecLayout& L, int64_t r) {
    const int64_t seg = r / L.seg_len;
    return (size_t)(seg * L.key_seg_stride + (r - seg * L.seg_len));
}
__device__ __forceinline__ size_t rec_grad_index(const RecLayout& L, int64_t r) {
    const int64_t seg = r / L.seg_len;
    return (size_t)(seg * L.grad_seg_stride + (r - seg * L.seg_len) * D);
}

__global__ void k_link_records(const int32_t* __restrict__ keys, int64_t n_rec, int64_t n_rows, RecLayout L,
                               int32_t* __restrict__ head, int32_t* __restrict__ next) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    const int32_t k = keys[rec_key_index(L, r)];
    if (k < 0 || k >= n_rows) {
        next[r] = -1;
        return;
    }
    next[r] = atomicExch(&head[k], (int32_t)r);
}

// 16 lanes per table row (one float4 each); a warp covers two consecutive rows = 512 contiguous bytes.
__global__ void __launch_bounds__(256) k_adam_sweep(float* __restrict__ table, float* __restrict__ m_,
                                                    float* __restrict__ v_, int64_t n_rows,
                                                    const float* __restrict__ rec_grads, RecLayout L,
                                                    int32_t* __restrict__ head, const int32_t* __restrict__ next,
                                                    const AdamHost hp) {
    const AdamScalars s = resolve_adam(hp);
    const int sub = threadIdx.x & 15;
    const int half = (threadIdx.x >> 4) & 1;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    // warp-uniform trip count: a warp owns rows 2*w and 2*w+1
    for (int64_t w = warp; 2 * w < n_rows; w += n_warps) {
        const int64_t row = 2 * w + half;
        const bool valid = row < n_rows;
        const size_t off = (size_t)(valid ? row : 2 * w) * D + sub * 4;
        float4 p = ld4(table + off);
        float4 m = ld4(m_ + off);
        float4 v = ld4(v_ + off);
        float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
        const int32_t h = valid ? head[row] : -1;
        __syncwarp();  // every lane holds its list head before any lane resets it
        if (h >= 0) {
            // ascending-index traversal of this row's (unordered) record list
            int32_t last = -1;
            while (true) {
                int32_t best = 0x7fffffff;
                for (int32_t r = h; r >= 0; r = __ldg(next + r))
                    if (r > last && r < best) best = r;
                if (best == 0x7fffffff) break;
                const float4 rg = ldg4(rec_grads + rec_grad_index(L, best) + sub * 4);
                g.x += rg.x; g.y += rg.y; g.z += rg.z; g.w += rg.w;
                last = best;
            }
            if (sub == 0) head[row] = -1;
        }
        if (valid) {
            adam_elem(p.x, m.x, v.x, g.x, s);
            adam_elem(p.y, m.y, v.y, g.y, s);
            adam_elem(p.z, m.z, v.z, g.z, s);
            adam_elem(p.w, m.w, v.w, g.w, s);
            st4(table + off, p);
            st4(m_ + off, m);
            st4(v_ + off, v);
        }
    }
}

__global__ void __launch_bounds__(256) k_adam_dense(float* __restrict__ p_, float* __restrict__ m_,
                                                    float* __restrict__ v_, int64_t n,
                                                    const float* __restrict__ g_parts, int32_t n_parts,
                                                    int64_t part_stride, const AdamHost hp) {
    const AdamScalars s = resolve_adam(hp);
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        float g = 0.f;
        for (int32_t k = 0; k < n_parts; ++k) g += __ldg(g_parts + (size_t)k * part_stride + i);
        float p = p_[i], m = m_[i], v = v_[i];
        adam_elem(p, m, v, g, s);
        p_[i] = p; m_[i] = m; v_[i] = v;
    }
}

// out[i] = sum_k parts[k * stride + i], ascending k (fixed order)
__global__ void __launch_bounds__(256) k_sum_parts(const float* __restrict__ parts, int32_t n_parts, int64_t stride,
                                                   int64_t n, float* __restrict__ out) {
    const int64_t step = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += step) {
        float g = 0.f;
        for (int32_t k = 0; k < n_parts; ++k) g += __ldg(parts + (size_t)k * stride + i);
        out[i] = g;
    }
}

// ---------------------------------------------------------------------------------------------
// One launch for the whole optimizer step: every embedding table and every dense tensor.  The grid is
// partitioned by block ranges; each range grid-strides over its own tensor.
// ---------------------------------------------------------------------------------------------
constexpr int ADAM_MAX_T = 4;

struct AdamTableArgs {
    float *table, *m, *v;
    int64_t n_rows;
    const int32_t* keys;
    const float* grads;
    int64_t n_rec;
    RecLayout L;
    int32_t* head;
    int32_t* next;
    int32_t* rec_row;             // CSR mode (all four non-null), see dccf_adam_table
    int32_t* csr_off;
    int32_t* csr;
    int32_t* csr_pool;
    int32_t block_lo, block_n;    // block range of the sweep kernel
    int32_t link_lo, link_n;      // block range of the link kernel
};
struct AdamDenseArgs {
    float *p, *m, *v;
    int64_t n;
    const float* g_parts;
    int32_t n_parts;
    int64_t part_stride;
    int32_t block_lo, block_n;
};
struct AdamAllArgs {
    AdamTableArgs t[ADAM_MAX_T];
    AdamDenseArgs d[ADAM_MAX_T];
    int32_t n_tables, n_dense;
    AdamHost hp;
};

__global__ void k_link_all(const AdamAllArgs a) {
    for (int i = 0; i < a.n_tables; ++i) {
        const AdamTableArgs& t = a.t[i];
        const int b = (int)blockIdx.x - t.link_lo;
        if (b < 0 || b >= t.link_n) continue;
        const int64_t r = (int64_t)b * blockDim.x + threadIdx.x;
        if (r >= t.n_rec) return;
        const int32_t k = t.keys[rec_key_index(t.L, r)];
        t.next[r] = (k < 0 || k >= t.n_rows) ? -1 : atomicExch(&t.head[k], (int32_t)r);
        return;
    }
}

// gradient of one table row from its record list, summed in ascending record index (deterministic whatever
// order the atomics linked the list in).  Executed by the 16 lanes of a half-warp together (lane = 4 columns):
// the list is walked once into shared memory, ranked by counting (L^2/16 cheap compares), then the records
// are added in rank order — O(L) dependent loads instead of the O(L^2) of selecting the next-larger index
// by repeated walks, which made the hottest item row (tens of records per step under data parallelism and
// Zipf popularity) the critical path of the whole sweep.  Lists longer than ADAM_LIST_CAP fall back to the
// repeated walk.
constexpr int ADAM_LIST_CAP = 96;

__device__ __forceinline__ float4 gather_row_grad(const AdamTableArgs& t, int32_t h, int sub, uint32_t half_mask,
                                                  int32_t* idx_s, int32_t* ord_s) {
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
    const int32_t second = __ldg(t.next + h);
    if (second < 0) {                                   // the common case: one record
        const float4 rg = ldg4(t.grads + rec_grad_index(t.L, h) + sub * 4);
        return rg;
    }
    int n = 0;
    int32_t r = h;
    for (; r >= 0 && n < ADAM_LIST_CAP; r = __ldg(t.next + r)) {
        if (sub == 0) idx_s[n] = r;
        ++n;
    }
    if (r >= 0) {
        // longer than the buffer: repeated walks, still ascending
        int32_t last = -1;
        while (true) {
            int32_t best = 0x7fffffff;
            for (int32_t q = h; q >= 0; q = __ldg(t.next + q))
                if (q > last && q < best) best = q;
            if (best == 0x7fffffff) break;
            const float4 rg = ldg4(t.grads + rec_grad_index(t.L, best) + sub * 4);
            g.x += rg.x; g.y += rg.y; g.z += rg.z; g.w += rg.w;
            last = best;
        }
        return g;
    }
    __syncwarp(half_mask);
    for (int e = sub; e < n; e += 16) {
        const int32_t mine = idx_s[e];
        int rank = 0;
        for (int j = 0; j < n; ++j) rank += (idx_s[j] < mine) ? 1 : 0;
        ord_s[rank] = mine;
    }
    __syncwarp(half_mask);
    // records added in ascending index, four loads in flight at a time (a hot item row has tens of records under
    // data parallelism: one load per add would expose the L2 latency once per record)
    int q = 0;
    for (; q + 4 <= n; q += 4) {
        float4 rg[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) rg[j] = ldg4(t.grads + rec_grad_index(t.L, ord_s[q + j]) + sub * 4);
#pragma unroll
        for (int j = 0; j < 4; ++j) { g.x += rg[j].x; g.y += rg[j].y; g.z += rg[j].z; g.w += rg[j].w; }
    }
    for (; q < n; ++q) {
        const float4 rg = ldg4(t.grads + rec_grad_index(t.L, ord_s[q]) + sub * 4);
        g.x += rg.x; g.y += rg.y; g.z += rg.z; g.w += rg.w;
    }
    __syncwarp(half_mask);
    return g;
}

// The same sum from a CSR list: the row's record ids sit at csr[o .. o + n) in arrival order (no walk: sixteen lanes
// load them at once), are ranked in shared memory and added in ascending index, four loads in flight.
__device__ __forceinline__ float4 gather_row_grad_csr(const AdamTableArgs& t, int32_t first, int32_t o, int32_t n, int sub,
                                                      uint32_t half_mask, int32_t* idx_s, int32_t* ord_s) {
    if (n == 1) return ldg4(t.grads + rec_grad_index(t.L, first) + sub * 4);
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
    if (n > ADAM_LIST_CAP) {
        // longer than the buffer: n rounds of "smallest id above the last one", each a strided scan by the half-warp
        int32_t last = -1;
        for (int k = 0; k < n; ++k) {
            int32_t best = 0x7fffffff;
            for (int e = sub; e < n; e += 16) {
                const int32_t q = __ldg(t.csr + o + e);
                if (q > last && q < best) best = q;
            }
#pragma unroll
            for (int w = 8; w > 0; w >>= 1) best = min(best, __shfl_xor_sync(half_mask, best, w));
            const float4 rg = ldg4(t.grads + rec_grad_index(t.L, best) + sub * 4);
            g.x += rg.x; g.y += rg.y; g.z += rg.z; g.w += rg.w;
            last = best;
        }
        return g;
    }
    for (int e = sub; e < n; e += 16) idx_s[e] = __ldg(t.csr + o + e);
    __syncwarp(half_mask);
    for (int e = sub; e < n; e += 16) {
        const int32_t mine = idx_s[e];
        int rank = 0;
        for (int j = 0; j < n; ++j) rank += (idx_s[j] < mine) ? 1 : 0;
        ord_s[rank] = mine;
    }
    __syncwarp(half_mask);
    int q = 0;
    for (; q + 4 <= n; q += 4) {
        float4 rg[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) rg[j] = ldg4(t.grads + rec_grad_index(t.L, ord_s[q + j]) + sub * 4);
#pragma unroll
        for (int j = 0; j < 4; ++j) { g.x += rg[j].x; g.y += rg[j].y; g.z += rg[j].z; g.w += rg[j].w; }
    }
    for (; q < n; ++q) {
        const float4 rg = ldg4(t.grads + rec_grad_index(t.L, ord_s[q]) + sub * 4);
        g.x += rg.x; g.y += rg.y; g.z += rg.z; g.w += rg.w;
    }
    __syncwarp(half_mask);
    return g;
}

// CSR build after the counting link: phase 0 — the first record of every row reserves the row's range in the pool;
// phase 1 — every record drops its id at (range start + its arrival position).
__global__ void k_csr_build(const AdamAllArgs a, int phase) {
    tl_begin(13);
    tl_end(13);
    for (int i = 0; i < a.n_tables; ++i) {
        const AdamTableArgs& t = a.t[i];
        // the tables' record ranges are laid out in blocks of 256 records, one 256-thread CTA each
        const int b = (int)blockIdx.x - t.link_lo;
        if (b < 0 || b >= t.link_n) continue;
        if (t.csr == nullptr) return;
        const int64_t r = (int64_t)b * 256 + threadIdx.x;
        if (r >= t.n_rec) return;
        const int32_t pos = t.next[r];
        if (pos < 0) return;                                   // (a record no link touched)
        const int32_t row = t.rec_row[r];
        if (phase == 0) {
            if (pos == 0) {
                t.csr_off[row] = atomicAdd(t.csr_pool, t.head[row] + 1);
                // compact list of the step's touched rows (second half of the csr buffer, count in csr_pool[1]): the
                // touched-row sweep walks THIS list — one half-warp per row, no pass over the records that own nothing
                t.csr[t.n_rec + atomicAdd(t.csr_pool + 1, 1)] = row;
            }
        } else {
            t.csr[t.csr_off[row] + pos] = (int32_t)r;
        }
        return;
    }
}

template <int R> __device__ __forceinline__ void step_all(const AdamAllArgs& a) {
    constexpr bool HM = rule_has_m<R>, HV = rule_has_v<R>;
    __shared__ int32_t list_s[16][2][ADAM_LIST_CAP];   // per half-warp: record indices as linked / in ascending order
    const AdamScalars s = resolve_rule<R>(a.hp);
    const int bid = (int)blockIdx.x;
    for (int i = 0; i < a.n_tables; ++i) {
        const AdamTableArgs& t = a.t[i];
        const int b = bid - t.block_lo;
        if (b < 0 || b >= t.block_n) continue;
        const int sub = threadIdx.x & 15;
        const int half = (threadIdx.x >> 4) & 1;
        const int64_t warp = ((int64_t)b * blockDim.x + threadIdx.x) >> 5;
        const int64_t n_warps = ((int64_t)t.block_n * blockDim.x) >> 5;
        // a warp owns rows 4w .. 4w+3 per trip (two per half-warp): six 16-byte loads in flight per lane
        for (int64_t w = warp; 4 * w < t.n_rows; w += n_warps) {
            const int64_t r0 = 4 * w + half, r1 = r0 + 2;
            const bool v0 = r0 < t.n_rows, v1 = r1 < t.n_rows;
            const size_t o0 = (size_t)(v0 ? r0 : 0) * D + sub * 4, o1 = (size_t)(v1 ? r1 : 0) * D + sub * 4;
            float4 p0 = ld4(t.table + o0), m0 = ld4_if<HM>(t.m + o0), q0 = ld4_if<HV>(t.v + o0);
            float4 p1 = ld4(t.table + o1), m1 = ld4_if<HM>(t.m + o1), q1 = ld4_if<HV>(t.v + o1);
            const int32_t h0 = v0 ? t.head[r0] : -1;
            const int32_t h1 = v1 ? t.head[r1] : -1;
            __syncwarp();  // every lane holds its list heads before any lane resets them
            float4 g0 = make_float4(0.f, 0.f, 0.f, 0.f), g1 = g0;
            const uint32_t half_mask = half ? 0xffff0000u : 0x0000ffffu;
            int32_t* idx_s = list_s[threadIdx.x >> 4][0];
            int32_t* ord_s = list_s[threadIdx.x >> 4][1];
            if (h0 >= 0) {
                g0 = gather_row_grad(t, h0, sub, half_mask, idx_s, ord_s);
                if (sub == 0) t.head[r0] = -1;
            }
            if (h1 >= 0) {
                g1 = gather_row_grad(t, h1, sub, half_mask, idx_s, ord_s);
                if (sub == 0) t.head[r1] = -1;
            }
            if (v0) {
                rule_elem4<R>(p0, m0, q0, g0, s);
                st4(t.table + o0, p0); st4_if<HM>(t.m + o0, m0); st4_if<HV>(t.v + o0, q0);
            }
            if (v1) {
                rule_elem4<R>(p1, m1, q1, g1, s);
                st4(t.table + o1, p1); st4_if<HM>(t.m + o1, m1); st4_if<HV>(t.v + o1, q1);
            }
        }
        return;
    }
    for (int i = 0; i < a.n_dense; ++i) {
        const AdamDenseArgs& d = a.d[i];
        const int b = bid - d.block_lo;
        if (b < 0 || b >= d.block_n) continue;
        const int64_t stride = (int64_t)d.block_n * blockDim.x;
        for (int64_t e = (int64_t)b * blockDim.x + threadIdx.x; e < d.n; e += stride) {
            float g = 0.f;
            for (int32_t k = 0; k < d.n_parts; ++k) g += __ldg(d.g_parts + (size_t)k * d.part_stride + e);
            float p = d.p[e], m = HM ? d.m[e] : 0.f, v = HV ? d.v[e] : 0.f;
            rule_elem<R>(p, m, v, g, s);
            d.p[e] = p;
            if constexpr (HM) d.m[e] = m;
            if constexpr (HV) d.v[e] = v;
        }
        return;
    }
}

__global__ void __launch_bounds__(256, 4) k_adam_all(const AdamAllArgs a) { step_all<RULE_ADAM>(a); }
__global__ void __launch_bounds__(256, 4) k_gd_all(const AdamAllArgs a) { step_all<RULE_GD>(a); }
__global__ void __launch_bounds__(256, 4) k_adagrad_all(const AdamAllArgs a) { step_all<RULE_ADAGRAD>(a); }

// ---------------------------------------------------------------------------------------------
// The same step split around the backward pass, so that the HBM-bound sweep of the rows a step does NOT touch
// (99 % of both tables) runs concurrently with the FMA/tensor-bound forward and backward on another stream:
//   k_link_ids       the record lists of the step built from the ids alone (record p = user row of pair p, record
//                    p*Z + z = item row of slot z), before any gradient exists: head[row] >= 0 marks a touched row
//   k_adam_untouched rows with head == -1: gradient = l2 / weight-decay terms only
//   k_adam_touched   after the backward: the record that ended up as the HEAD of its row's list processes the row
//                    (records summed in ascending index as always); + W, b; the last CTA advances the step counters
// Every row is updated exactly once per step and with the same arithmetic as k_adam_all.
// ---------------------------------------------------------------------------------------------
struct LinkIdsArgs {
    const int64_t* X;            // segment 0; segment s at + s * seg_stride (int64 elements)
    const int64_t* sample_item;
    const int64_t* X_local;      // this rank's own batch (exposure softmax)
    const int64_t* si_local;
    int64_t n_pairs;             // per segment
    int64_t seg_stride;
    int32_t n_seg, user_seg;     // user_seg >= 0: only that segment carries user records (row-sharded user table)
    int32_t S, A, user_base, n_users, n_items;
    int32_t* head_u;
    int32_t* next_u;
    int32_t* head_i;
    int32_t* next_i;
    int32_t link_blocks;     // blocks [0, link_blocks) link; the rest evaluate the exposure softmax (warp per pair)
    int32_t expo_blocks;     // then expo_blocks blocks of exposure softmax, then the dense-range prefetch blocks
    dccf_expo ex;
    float* expo_e;           // [P, Z]
    float* expo_den;         // [P]
    dccf_link_extra extra;   // staging + L2 prefetch + counting mode (all-null: none)
    int32_t feat_dim;
    DpSync sync;             // data-parallel global link: wait for the ids, hand the buffer back (n_wait = n_done = 0: none)
};

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// one 256-byte table row of each of up to three tensors (parameter + its two Adam moments)
__device__ __forceinline__ void prefetch_rows(const float* const (&t)[3], int32_t row) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        if (t[k] != nullptr) {
            const char* p = reinterpret_cast<const char*>(t[k] + (size_t)row * D);
            prefetch_l2(p);
            prefetch_l2(p + 128);
        }
    }
}

__global__ void __launch_bounds__(256) k_link_ids(const LinkIdsArgs a) {
    tl_begin(0);
    // the next kernel on the stream may have been launched as a programmatic dependent (the partial-product kernel of the
    // step reads nothing this launch writes): it may start now
    asm volatile("griddepcontrol.launch_dependents;");
    __shared__ int64_t s_batch;
    // epoch_ptrs_dev given: X_out given -> this launch STAGES batch *cursor of the rank's own epoch; X_out null ->
    // data-parallel link of the global step from the epoch-wide gather of every rank's ids (slots 2..5: base addresses of
    // X_all [world, n, P, 2] / si_all [world, n, P, S] and their per-rank strides).  Nobody moves the cursor before the
    // end of the step (dccf_adam_touched, advance_cursor_dev): the forward reads the same batch beside this launch.
    const bool staged = a.extra.epoch_ptrs_dev != nullptr && a.extra.X_out != nullptr;
    const bool epoch_global = a.extra.epoch_ptrs_dev != nullptr && a.extra.X_out == nullptr;
    const int64_t *X = a.X, *si = a.sample_item, *X_local = a.X_local, *si_local = a.si_local;
    int64_t seg_stride_x = a.seg_stride, seg_stride_s = a.seg_stride;
    if (staged || epoch_global) {
        if (threadIdx.x == 0) s_batch = *a.extra.cursor_dev;
        __syncthreads();
        const int base = epoch_global ? 2 : 0;
        X = reinterpret_cast<const int64_t*>(a.extra.epoch_ptrs_dev[base]) + s_batch * a.n_pairs * 2;
        si = reinterpret_cast<const int64_t*>(a.extra.epoch_ptrs_dev[base + 1]) + s_batch * a.n_pairs * a.S;
        if (epoch_global) {
            seg_stride_x = (int64_t)a.extra.epoch_ptrs_dev[4];
            seg_stride_s = (int64_t)a.extra.epoch_ptrs_dev[5];
        } else {
            X_local = X;
            si_local = si;
        }
    }
    dp_wait_inline(a.sync);      // (data parallel) the peers' ids have arrived
    const int bid = (int)blockIdx.x;
    if (bid >= a.link_blocks + a.expo_blocks) {
        // dense ranges (W, its moments, its operand images) into L2, one 128-byte line per thread and trip
        const int64_t t0 = (int64_t)(bid - a.link_blocks - a.expo_blocks) * blockDim.x + threadIdx.x;
        const int64_t nt = (int64_t)(gridDim.x - a.link_blocks - a.expo_blocks) * blockDim.x;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const char* base = reinterpret_cast<const char*>(a.extra.pf_dense[k]);
            if (base == nullptr) continue;
            for (int64_t off = t0 * 128; off < a.extra.pf_dense_bytes[k]; off += nt * 128) prefetch_l2(base + off);
        }
    } else if (bid >= a.link_blocks) {
        // exposure softmax of every local pair: depends on the ids only, so it is taken off the critical path here
        const int64_t p = (int64_t)(bid - a.link_blocks) * (blockDim.x >> 5) + (threadIdx.x >> 5);
        if (p < a.n_pairs)   // warp-uniform
            backdoor_weights(a.ex, X_local, si_local, p, threadIdx.x & 31, a.n_users, a.user_base, a.n_items, a.S, a.A,
                             a.expo_e + p * (a.S + 1), a.expo_den + p, nullptr);
    } else {
        // record index (the one the gradient records will have): segment-major, as the Adam tables number them
        const int Z = a.S + 1;
        const int64_t per_seg = a.n_pairs * (Z + 1);
        const int64_t i = (int64_t)bid * blockDim.x + threadIdx.x;
        // (a staging launch with n_seg == 0 — the local launch of a data-parallel step — copies the ids, links nothing)
        if (i < per_seg * max(a.n_seg, staged ? 1 : 0)) {
            const int seg = (int)(i / per_seg);
            const bool do_link = seg < a.n_seg;
            const int64_t il = i - (int64_t)seg * per_seg;
            const int64_t p = il / (Z + 1);
            const int slot = (int)(il - p * (Z + 1));   // 0 = the user record of pair p, 1 + z = its item record of slot z
            const int64_t* Xs = X + (int64_t)seg * seg_stride_x;
            const int64_t* sis = si + (int64_t)seg * seg_stride_s;
            if (slot == 0) {
                const int64_t uid = Xs[2 * p];
                if (staged) {
                    a.extra.X_out[2 * p] = uid;
                    // rating prediction: the pair's label, from the label epoch in slot 6
                    if (a.extra.Y_out != nullptr)
                        a.extra.Y_out[p] = reinterpret_cast<const float*>(a.extra.epoch_ptrs_dev[6])[s_batch * a.n_pairs + p];
                }
                if (do_link && !(a.user_seg >= 0 && seg != a.user_seg)) {
                    const int32_t u = checked_id(uid - a.user_base, a.n_users, nullptr);
                    const int32_t r = (int32_t)((a.user_seg >= 0 ? 0 : (int64_t)seg * a.n_pairs) + p);
                    if (a.extra.rec_row_user != nullptr) {       // counting mode: arrival position + the row itself
                        a.next_u[r] = atomicAdd(&a.head_u[u], 1) + 1;
                        a.extra.rec_row_user[r] = u;
                    } else {
                        a.next_u[r] = atomicExch(&a.head_u[u], r);
                    }
                    prefetch_rows(a.extra.pf_user, u);
                }
            } else {
                const int z = slot - 1;
                const int64_t id = slot_item(Xs, sis, p, z, a.S);
                if (staged) {
                    if (z == 0) a.extra.X_out[2 * p + 1] = id;
                    else a.extra.sample_item_out[p * a.S + (z - 1)] = id;
                }
                if (do_link) {
                    const int32_t it = checked_id(id, a.n_items, nullptr);
                    const int32_t r = (int32_t)(((int64_t)seg * a.n_pairs + p) * Z + z);
                    if (a.extra.rec_row_item != nullptr) {
                        a.next_i[r] = atomicAdd(&a.head_i[it], 1) + 1;
                        a.extra.rec_row_item[r] = it;
                    } else {
                        a.next_i[r] = atomicExch(&a.head_i[it], r);
                    }
                    prefetch_rows(a.extra.pf_item, it);
                }
            }
            if (a.extra.pf_feat != nullptr && (a.n_seg == 1 || (staged && a.n_seg == 0))) {
                // the true item's feature row (feat_dim * 4 bytes), its 128-byte lines shared out over the pair's Z + 1
                // threads (one GPU only: under data parallelism the other ranks' pairs are not multiplied here)
                const int32_t fi = checked_id(Xs[2 * p + 1], a.n_items, nullptr);
                const char* row = reinterpret_cast<const char*>(a.extra.pf_feat + (size_t)fi * a.feat_dim);
                for (int off = slot * 128; off < a.feat_dim * 4; off += (Z + 1) * 128) prefetch_l2(row + off);
            }
        }
    }
    if (a.sync.n_done > 0) {
        // the last CTA to finish hands the id buffer back to the peers
        __shared__ int s_last;
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            s_last = (atomicAdd(a.extra.stage_counter, 1) == (int32_t)gridDim.x - 1) ? 1 : 0;
            if (s_last) *a.extra.stage_counter = 0;
        }
        __syncthreads();
        if (s_last) dp_done_inline(a.sync);
    }
    tl_end(0);
}

constexpr int ADAM_SIDE_SMEM = 120 * 1024;     // occupancy limiter of the side-stream sweep, see dccf_adam_untouched

// L2-only loads / stores: the sweep streams 100 MB past SMs whose L1 holds the feature rows of the concurrent
// forward — it must not evict them
__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void stcg4(float* p, const float4& v) { __stcg(reinterpret_cast<float4*>(p), v); }

template <bool On> __device__ __forceinline__ float4 ldcg4_if(const float* p) {
    if constexpr (On) return ldcg4(p); else return make_float4(0.f, 0.f, 0.f, 0.f);
}
template <bool On> __device__ __forceinline__ void stcg4_if(float* p, const float4& v) {
    if constexpr (On) stcg4(p, v);
}

template <int R> __device__ __forceinline__ void step_untouched(const AdamAllArgs& a) {
    constexpr bool HM = rule_has_m<R>, HV = rule_has_v<R>;
    tl_begin(1);
    const AdamScalars s = resolve_rule<R>(a.hp);
    const int bid = (int)blockIdx.x;
    for (int i = 0; i < a.n_tables; ++i) {
        const AdamTableArgs& t = a.t[i];
        const int b = bid - t.block_lo;
        if (b < 0 || b >= t.block_n) continue;
        const int sub = threadIdx.x & 15;
        const int half = (threadIdx.x >> 4) & 1;
        const int64_t warp = ((int64_t)b * blockDim.x + threadIdx.x) >> 5;   // (block size: see dccf_adam_untouched)
        const int64_t n_warps = ((int64_t)t.block_n * blockDim.x) >> 5;
        // One trip = 4 rows per warp (two per half-warp).  The touched flags of the NEXT trip are loaded, and its rows
        // requested into L2, before this trip's rows are read: a trip then costs one memory round trip that mostly ends
        // in L2 instead of two that end in DRAM.
        auto row_ok = [&](int64_t r) { return r < t.n_rows && t.head[r] == -1; };
        auto request = [&](int64_t r) {
            if (r >= t.n_rows || (sub & 7) != 0) return;              // one lane per 128-byte line
            const size_t o = (size_t)r * D + sub * 4;
            prefetch_l2(t.table + o);
            if constexpr (HM) prefetch_l2(t.m + o);
            if constexpr (HV) prefetch_l2(t.v + o);
        };
        bool v0 = 4 * warp < t.n_rows && row_ok(4 * warp + half), v1 = 4 * warp < t.n_rows && row_ok(4 * warp + half + 2);
        for (int64_t w = warp; 4 * w < t.n_rows; w += n_warps) {
            const int64_t r0 = 4 * w + half, r1 = r0 + 2;
            const int64_t n0 = r0 + 4 * n_warps, n1 = n0 + 2;
            request(n0);
            request(n1);
            const bool nv0 = row_ok(n0), nv1 = row_ok(n1);
            const size_t o0 = (size_t)(v0 ? r0 : 0) * D + sub * 4, o1 = (size_t)(v1 ? r1 : 0) * D + sub * 4;
            float4 p0, m0, q0, p1, m1, q1;
            if (v0) { p0 = ldcg4(t.table + o0); m0 = ldcg4_if<HM>(t.m + o0); q0 = ldcg4_if<HV>(t.v + o0); }
            if (v1) { p1 = ldcg4(t.table + o1); m1 = ldcg4_if<HM>(t.m + o1); q1 = ldcg4_if<HV>(t.v + o1); }
            const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
            if (v0) {
                rule_elem4<R>(p0, m0, q0, zero, s);
                stcg4(t.table + o0, p0); stcg4_if<HM>(t.m + o0, m0); stcg4_if<HV>(t.v + o0, q0);
            }
            if (v1) {
                rule_elem4<R>(p1, m1, q1, zero, s);
                stcg4(t.table + o1, p1); stcg4_if<HM>(t.m + o1, m1); stcg4_if<HV>(t.v + o1, q1);
            }
            v0 = nv0; v1 = nv1;
        }
        __syncthreads();
        tl_end(1);
        return;
    }
}

__global__ void __maxnreg__(64) k_adam_untouched(const AdamAllArgs a) { step_untouched<RULE_ADAM>(a); }
__global__ void __maxnreg__(64) k_gd_untouched(const AdamAllArgs a) { step_untouched<RULE_GD>(a); }
__global__ void __maxnreg__(64) k_adagrad_untouched(const AdamAllArgs a) { step_untouched<RULE_ADAGRAD>(a); }

struct WImageArgs {
    float* img;          // operand images of W for the tensor-core forward of the NEXT step (tc_train.cu), or null
    int32_t tensor;      // index of W among the dense tensors
    int32_t K;           // row length of W
    // optional: the last CTA to finish advances the graph's device counters (replaces dccf_state_advance)
    int32_t* cta_counter;    // zero on entry, zero again on exit
    int32_t* step_dev;
    uint64_t* offset_dev;
    int64_t* cursor_dev;     // batch cursor of a device-resident epoch (dccf_link_extra / dccf_batch_ref): += 1
};

__device__ __forceinline__ void touched_cta_done(const AdamAllArgs& a, const WImageArgs& wi, const DpSync& sync) {
    __shared__ int s_last;
    __syncthreads();
    tl_end(5);
    // (launched as a programmatic dependent of the dW / db push: this grid must not complete before that one has — a
    // no-op in a plain launch)
    asm volatile("griddepcontrol.wait;" ::: "memory");
    if (wi.cta_counter == nullptr) return;                       // every thread of this CTA has read the counters it needs and stored its rows
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = (atomicAdd(wi.cta_counter, 1) == (int32_t)gridDim.x - 1) ? 1 : 0;
        if (s_last) {
            if (wi.step_dev) wi.step_dev[0] += 1;
            if (wi.offset_dev) wi.offset_dev[0] += 1;
            if (wi.cursor_dev) wi.cursor_dev[0] += 1;
            for (int i = 0; i < a.n_tables; ++i)
                if (a.t[i].csr_pool != nullptr) { a.t[i].csr_pool[0] = 0; a.t[i].csr_pool[1] = 0; }   // ranges and row list released
            *wi.cta_counter = 0;
        }
    }
    if (sync.n_done > 0 || sync.loss_out != nullptr) {           // (kernel-uniform)
        __syncthreads();
        if (s_last) dp_done_inline(sync);
    }
}

template <int R> __device__ __forceinline__ void step_touched(const AdamAllArgs& a, const WImageArgs& wi, const DpSync& sync) {
    constexpr bool HM = rule_has_m<R>, HV = rule_has_v<R>;
    __shared__ int32_t list_s[16][2][ADAM_LIST_CAP];
    tl_begin(5);
    const int bid = (int)blockIdx.x;
    {
        // (data parallel) every rank's gradient records and dW / db / loss have arrived.  DCCF_DP_SYNC_OVERLAP_PUSH: the
        // CTAs that sweep table rows need the records only (wait[0]) and start while this rank's dW / db push — the kernel
        // before this one on the stream, of which this launch is then a programmatic dependent — is still running; the
        // CTAs of the dense tensors wait for wait[1..].
        uint32_t mask = 7u;
        if ((sync.flags & DCCF_DP_SYNC_OVERLAP_PUSH) && sync.n_wait >= 2) {
            bool table_cta = false;
            for (int i = 0; i < a.n_tables; ++i) table_cta = table_cta || (bid >= a.t[i].block_lo && bid < a.t[i].block_lo + a.t[i].block_n);
            mask = table_cta ? 1u : 6u;
        }
        dp_wait_inline(sync, mask);
        if (sync.n_wait > 0 && (mask & 2u)) { tl_begin(12); tl_end(12); }
    }
    const AdamScalars s = resolve_rule<R>(a.hp);
    for (int i = 0; i < a.n_tables; ++i) {
        const AdamTableArgs& t = a.t[i];
        const int b = bid - t.block_lo;
        if (b < 0 || b >= t.block_n) continue;
        // half-warp per record (grid-stride: under data parallelism a step has tens of thousands of records, and one
        // CTA per 16 of them would queue in several waves); the record that is the head of its row's list owns the row
        const int sub = threadIdx.x & 15;
        const uint32_t half_mask = (threadIdx.x & 16) ? 0xffff0000u : 0x0000ffffu;
        const int64_t hw_stride = ((int64_t)t.block_n * blockDim.x) >> 4;
        const bool csr = t.csr != nullptr;
        // CSR mode: one half-warp per TOUCHED ROW (compact list built by k_csr_build); list mode: per record, the head
        // record of a row's list owns the row
        const int64_t n_work = csr ? (int64_t)__ldcg(t.csr_pool + 1) : t.n_rec;
        if (csr) {
            // TWO rows per half-warp and trip: their independent chains (row id -> count / range -> parameters, moments,
            // record ids -> gradients) are in flight together — the sweep is bound by the latency of these dependent
            // loads, not by their bytes
            int32_t* idx_s = list_s[threadIdx.x >> 4][0];
            int32_t* ord_s = list_s[threadIdx.x >> 4][1];
            for (int64_t r = ((int64_t)b * blockDim.x + threadIdx.x) >> 4; r < n_work; r += 2 * hw_stride) {
                const bool two = r + hw_stride < n_work;
                const int32_t rowA = __ldcg(t.csr + t.n_rec + r);
                const int32_t rowB = two ? __ldcg(t.csr + t.n_rec + r + hw_stride) : rowA;
                const int32_t nA = t.head[rowA] + 1, nB = t.head[rowB] + 1;
                const int32_t offA = t.csr_off[rowA], offB = t.csr_off[rowB];
                __syncwarp(half_mask);      // every lane of the half-warp has read the heads before lane 0 resets them
                const size_t oA = (size_t)rowA * D + sub * 4, oB = (size_t)rowB * D + sub * 4;
                float4 pA = ld4(t.table + oA), mA = ld4_if<HM>(t.m + oA), qA = ld4_if<HV>(t.v + oA);
                float4 pB = ld4(t.table + oB), mB = ld4_if<HM>(t.m + oB), qB = ld4_if<HV>(t.v + oB);
                const int32_t fA = __ldcg(t.csr + offA), fB = __ldcg(t.csr + offB);
                float4 gA, gB;
                if (nA == 1 && nB == 1) {   // the common case: both single records, both loads in flight
                    gA = ldg4(t.grads + rec_grad_index(t.L, fA) + sub * 4);
                    gB = ldg4(t.grads + rec_grad_index(t.L, fB) + sub * 4);
                } else {
                    gA = gather_row_grad_csr(t, fA, offA, nA, sub, half_mask, idx_s, ord_s);
                    gB = gather_row_grad_csr(t, fB, offB, nB, sub, half_mask, idx_s, ord_s);
                }
                if (sub == 0) {
                    t.head[rowA] = -1;
                    if (two) t.head[rowB] = -1;
                }
                rule_elem4<R>(pA, mA, qA, gA, s);
                st4(t.table + oA, pA); st4_if<HM>(t.m + oA, mA); st4_if<HV>(t.v + oA, qA);
                if (two) {
                    rule_elem4<R>(pB, mB, qB, gB, s);
                    st4(t.table + oB, pB); st4_if<HM>(t.m + oB, mB); st4_if<HV>(t.v + oB, qB);
                }
            }
            touched_cta_done(a, wi, sync);
            return;
        }
        for (int64_t r = ((int64_t)b * blockDim.x + threadIdx.x) >> 4; r < n_work; r += hw_stride) {
            int32_t row, n_list = 0, off = 0, first = (int32_t)r;
            if (csr) {
                row = __ldcg(t.csr + t.n_rec + r);
                n_list = t.head[row] + 1;
                off = t.csr_off[row];
            } else {
                row = t.keys[rec_key_index(t.L, r)];
                if (row < 0 || row >= t.n_rows || t.head[row] != (int32_t)r) row = -1;
            }
            if (row < 0) continue;          // (uniform over the half-warp: all 16 lanes read the same key and head)
            __syncwarp(half_mask);          // every lane of the half-warp has read the head before lane 0 resets it
            const size_t o = (size_t)row * D + sub * 4;
            float4 p = ld4(t.table + o), m = ld4_if<HM>(t.m + o), q = ld4_if<HV>(t.v + o);
            if (csr && n_list == 1) first = __ldcg(t.csr + off);
            const float4 g = csr ? gather_row_grad_csr(t, first, off, n_list, sub, half_mask,
                                                       list_s[threadIdx.x >> 4][0], list_s[threadIdx.x >> 4][1])
                                 : gather_row_grad(t, (int32_t)r, sub, half_mask, list_s[threadIdx.x >> 4][0], list_s[threadIdx.x >> 4][1]);
            if (sub == 0) t.head[row] = -1;
            rule_elem4<R>(p, m, q, g, s);
            st4(t.table + o, p); st4_if<HM>(t.m + o, m); st4_if<HV>(t.v + o, q);
        }
        touched_cta_done(a, wi, sync);
        return;
    }
    for (int i = 0; i < a.n_dense; ++i) {
        const AdamDenseArgs& d = a.d[i];
        const int b = bid - d.block_lo;
        if (b < 0 || b >= d.block_n) continue;
        const int64_t stride = (int64_t)d.block_n * blockDim.x;
        const bool image = wi.img != nullptr && wi.tensor == i;
        for (int64_t e = (int64_t)b * blockDim.x + threadIdx.x; e < d.n; e += stride) {
            float p = d.p[e], m = HM ? d.m[e] : 0.f, v = HV ? d.v[e] : 0.f;
            // partials added in ascending order, up to sixteen loads in flight at a time (the dW kernel of the reference
            // shape leaves 20: a rolled tail loop waited for the last four one L2 round trip after the other)
            float g = 0.f;
            for (int32_t k = 0; k < d.n_parts; k += 16) {
                float t16[16];
#pragma unroll
                for (int q = 0; q < 16; ++q)
                    if (k + q < d.n_parts) t16[q] = __ldg(d.g_parts + (size_t)(k + q) * d.part_stride + e);
#pragma unroll
                for (int q = 0; q < 16; ++q)
                    if (k + q < d.n_parts) g += t16[q];
            }
            rule_elem<R>(p, m, v, g, s);
            d.p[e] = p;
            if constexpr (HM) d.m[e] = m;
            if constexpr (HV) d.v[e] = v;
            if (image) {
                // same layout as k_prep_w_image (tc_train.cu): 32-wide K chunks of [hi 8 KB | lo 8 KB], 8x4 core matrices
                const int n = (int)(e / wi.K), k = (int)(e - (int64_t)n * wi.K);
                const int c = k >> 5, kk = k & 31;
                const float hi = __uint_as_float(__float_as_uint(p) & 0xFFFFE000u);
                float* base = wi.img + (size_t)c * 4096;
                const int off = (n >> 3) * 256 + (kk >> 2) * 32 + (n & 7) * 4 + (kk & 3);
                base[off] = hi;
                base[2048 + off] = __fsub_rn(p, hi);
            }
        }
        touched_cta_done(a, wi, sync);
        return;
    }
}

__global__ void __launch_bounds__(256) k_adam_touched(const AdamAllArgs a, const WImageArgs wi, const DpSync sync) {
    step_touched<RULE_ADAM>(a, wi, sync);
}
__global__ void __launch_bounds__(256) k_gd_touched(const AdamAllArgs a, const WImageArgs wi, const DpSync sync) {
    step_touched<RULE_GD>(a, wi, sync);
}
__global__ void __launch_bounds__(256) k_adagrad_touched(const AdamAllArgs a, const WImageArgs wi, const DpSync sync) {
    step_touched<RULE_ADAGRAD>(a, wi, sync);
}

__global__ void k_state_advance(int32_t* step_dev, uint64_t* offset_dev, uint64_t inc) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        if (step_dev) step_dev[0] += 1;
        if (offset_dev) offset_dev[0] += inc;
    }
}

// Copy batch number *cursor of a device-resident epoch ([n_batches, P, 2] ids and [n_batches, P, S] confounder
// draws, with Y_out also [n_batches, P] labels; base addresses read from device memory) into the step graph's static
// input buffers, then advance the cursor: a replayed graph walks through the epoch without any host-side copy.
__global__ void __launch_bounds__(1024) k_stage_batch(const uint64_t* __restrict__ epoch_ptrs, int64_t* cursor,
                                                      int64_t n_x, int64_t n_s, int64_t* __restrict__ X_out,
                                                      int64_t* __restrict__ si_out, float* __restrict__ Y_out) {
    tl_begin(6);
    tl_end(6);
    const int64_t b = *cursor;
    const int64_t* X_src = reinterpret_cast<const int64_t*>(epoch_ptrs[0]) + b * n_x;
    const int64_t* s_src = reinterpret_cast<const int64_t*>(epoch_ptrs[1]) + b * n_s;
    // 16-byte copies when the batch slices are 16-byte aligned (they are: n_x and n_s are even), all loads of a
    // thread issued before its first store
    const int64_t n2x = n_x >> 1, n2s = n_s >> 1;
    const longlong2* X2 = reinterpret_cast<const longlong2*>(X_src);
    const longlong2* S2 = reinterpret_cast<const longlong2*>(s_src);
    if (((n_x | n_s) & 1) == 0 && (reinterpret_cast<uintptr_t>(X_src) & 15) == 0 && (reinterpret_cast<uintptr_t>(s_src) & 15) == 0 &&
        (reinterpret_cast<uintptr_t>(X_out) & 15) == 0 && (reinterpret_cast<uintptr_t>(si_out) & 15) == 0) {
        for (int64_t i0 = 0; i0 < n2x + n2s; i0 += 4 * blockDim.x) {
            longlong2 v[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int64_t i = i0 + q * blockDim.x + threadIdx.x;
                if (i < n2x) v[q] = X2[i];
                else if (i < n2x + n2s) v[q] = S2[i - n2x];
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int64_t i = i0 + q * blockDim.x + threadIdx.x;
                if (i < n2x) reinterpret_cast<longlong2*>(X_out)[i] = v[q];
                else if (i < n2x + n2s) reinterpret_cast<longlong2*>(si_out)[i - n2x] = v[q];
            }
        }
    } else {
        for (int64_t i = threadIdx.x; i < n_x; i += blockDim.x) X_out[i] = X_src[i];
        for (int64_t i = threadIdx.x; i < n_s; i += blockDim.x) si_out[i] = s_src[i];
    }
    if (Y_out != nullptr) {
        const float* y_src = reinterpret_cast<const float*>(epoch_ptrs[6]) + b * (n_x >> 1);
        for (int64_t i = threadIdx.x; i < (n_x >> 1); i += blockDim.x) Y_out[i] = y_src[i];
    }
    __syncthreads();
    if (threadIdx.x == 0) *cursor = b + 1;
}

static int marshal_sync(const char* who, const dccf_dp_sync* in, DpSync* out) {
    out->world = 1; out->rank = 0; out->n_wait = 0; out->n_done = 0;
    out->loss_parts = nullptr; out->loss_stride = 0; out->n_loss = 0; out->loss_out = nullptr;
    out->flags = 0;
    if (in == nullptr) return DCCF_OK;
    out->flags = in->flags;
    DCCF_CHECK_ARG(in->world >= 1 && in->world <= DP_MAX_WORLD && in->rank >= 0 && in->rank < in->world,
                   "%s: sync: world %d / rank %d outside [1,%d]", who, in->world, in->rank, DP_MAX_WORLD);
    DCCF_CHECK_ARG(in->n_wait >= 0 && in->n_wait <= 3 && in->n_done >= 0 && in->n_done <= 3, "%s: sync: at most 3 channels", who);
    DCCF_CHECK_ARG(in->loss_out == nullptr || (in->loss_parts != nullptr && in->n_loss >= 1), "%s: sync: loss_out needs loss_parts", who);
    out->world = in->world; out->rank = in->rank; out->n_wait = in->n_wait; out->n_done = in->n_done;
    for (int k = 0; k < 3; ++k) {
        const dccf_dp_channel* src[2] = {&in->wait[k], &in->done[k]};
        DpChannel* dst[2] = {&out->wait[k], &out->done[k]};
        const int used[2] = {k < in->n_wait, k < in->n_done};
        for (int w = 0; w < 2; ++w) {
            for (int p = 0; p < DP_MAX_WORLD; ++p) dst[w]->base[p] = (used[w] && p < in->world) ? reinterpret_cast<float*>(src[w]->peer_bases[p]) : nullptr;
            dst[w]->flag_off = used[w] ? src[w]->flag_off : 0;
            dst[w]->epoch_dev = used[w] ? src[w]->epoch_dev : nullptr;
            dst[w]->n_ctas = used[w] ? dp_push_ctas(src[w]->seg_floats) : 0;
            if (used[w]) {
                DCCF_CHECK_ARG(src[w]->epoch_dev != nullptr, "%s: sync: channel %d has no epoch counter", who, k);
                for (int p = 0; p < in->world; ++p) DCCF_CHECK_ARG(src[w]->peer_bases[p] != 0, "%s: sync: channel %d peer %d is null", who, k, p);
            }
        }
    }
    out->loss_parts = in->loss_parts; out->loss_stride = in->loss_stride; out->n_loss = in->n_loss; out->loss_out = in->loss_out;
    return DCCF_OK;
}

static int check_hp(const dccf_adam* hp, AdamHost* out, const char* who) {
    DCCF_CHECK_ARG(hp != nullptr, "%s: null hyper-parameter struct", who);
    DCCF_CHECK_ARG(hp->step_dev != nullptr || hp->step >= 1, "%s: step must be >= 1 (got %d)", who, hp->step);
    DCCF_CHECK_ARG(hp->beta1 >= 0.0 && hp->beta1 < 1.0 && hp->beta2 >= 0.0 && hp->beta2 < 1.0, "%s: betas out of range", who);
    DCCF_CHECK_ARG(hp->rule == RULE_ADAM || hp->rule == RULE_GD || hp->rule == RULE_ADAGRAD,
                   "%s: unknown optimizer rule %d (0 Adam, 1 GD, 2 Adagrad)", who, hp->rule);
    out->lr = hp->lr; out->beta1 = hp->beta1; out->beta2 = hp->beta2;
    out->eps = (float)hp->eps; out->l2 = (float)hp->l2; out->wd = (float)hp->weight_decay; out->clip = (float)hp->clip;
    out->step = hp->step; out->step_dev = hp->step_dev;
    return DCCF_OK;
}

// the per-tensor entry points implement Adam only
static int check_hp_adam(const dccf_adam* hp, AdamHost* out, const char* who) {
    int rc = check_hp(hp, out, who);
    if (rc != DCCF_OK) return rc;
    DCCF_CHECK_ARG(hp->rule == RULE_ADAM, "%s: Adam only (rule %d); use dccf_adam_step for GD / Adagrad", who, hp->rule);
    return DCCF_OK;
}

// kernel of each rule, indexed by dccf_adam.rule
typedef void (*StepKernel)(AdamAllArgs);
typedef void (*TouchedKernel)(AdamAllArgs, WImageArgs, DpSync);
static const StepKernel k_all_of[3] = {k_adam_all, k_gd_all, k_adagrad_all};
static const StepKernel k_untouched_of[3] = {k_adam_untouched, k_gd_untouched, k_adagrad_untouched};
static const TouchedKernel k_touched_of[3] = {k_adam_touched, k_gd_touched, k_adagrad_touched};
static const char* const all_name[3] = {"k_adam_all", "k_gd_all", "k_adagrad_all"};
static const char* const untouched_name[3] = {"k_adam_untouched", "k_gd_untouched", "k_adagrad_untouched"};
static const char* const touched_name[3] = {"k_adam_touched", "k_gd_touched", "k_adagrad_touched"};

}  // namespace dccf

using namespace dccf;

extern "C" int dccf_adam_sweep_seg(float* table, float* m, float* v, int64_t n_table_rows, const int32_t* rec_keys,
                                   const float* rec_grads, int32_t n_seg, int64_t seg_len, int64_t key_seg_stride,
                                   int64_t grad_seg_stride, int32_t* head, int32_t* next, const dccf_adam* hp,
                                   void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AdamHost h;
    int rc = check_hp_adam(hp, &h, "dccf_adam_sweep");
    if (rc != DCCF_OK) return rc;
    DCCF_CHECK_ARG(table && m && v && head, "dccf_adam_sweep: null buffer");
    DCCF_CHECK_ARG(n_seg >= 0 && seg_len >= 0, "dccf_adam_sweep: negative record layout");
    const int64_t n_rec = (int64_t)n_seg * seg_len;
    DCCF_CHECK_ARG(n_rec == 0 || (rec_keys && rec_grads && next), "dccf_adam_sweep: %lld records but a null record buffer", (long long)n_rec);
    DCCF_CHECK_ARG(n_rec < ((int64_t)1 << 31) && n_table_rows < ((int64_t)1 << 31), "dccf_adam_sweep: sizes exceed int32 indexing");
    DCCF_CHECK_ARG(n_seg <= 1 || (key_seg_stride >= seg_len && grad_seg_stride >= seg_len * D), "dccf_adam_sweep: segment strides overlap");
    if (n_table_rows <= 0) return DCCF_OK;
    RecLayout L;
    L.seg_len = seg_len > 0 ? seg_len : 1;
    L.key_seg_stride = key_seg_stride;
    L.grad_seg_stride = grad_seg_stride;
    if (n_rec > 0) {
        k_link_records<<<(unsigned)((n_rec + 255) / 256), 256, 0, stream>>>(rec_keys, n_rec, n_table_rows, L, head, next);
        DCCF_CHECK_LAUNCH("k_link_records");
    }
    // 16 rows per 256-thread CTA per pass; cap the grid at 8 CTAs per SM and grid-stride beyond
    int64_t ctas = (n_table_rows + 15) / 16;
    const int64_t cap = 148 * 8;
    if (ctas > cap) ctas = cap;
    k_adam_sweep<<<(unsigned)ctas, 256, 0, stream>>>(table, m, v, n_table_rows, rec_grads, L, head, next, h);
    DCCF_CHECK_LAUNCH("k_adam_sweep");
    return DCCF_OK;
}

extern "C" int dccf_adam_sweep(float* table, float* m, float* v, int64_t n_table_rows, const int32_t* rec_keys,
                               const float* rec_grads, int64_t n_rec, int32_t* head, int32_t* next,
                               const dccf_adam* hp, void* stream_) {
    DCCF_CHECK_ARG(n_rec >= 0, "dccf_adam_sweep: negative record count");
    return dccf_adam_sweep_seg(table, m, v, n_table_rows, rec_keys, rec_grads, 1, n_rec, n_rec, n_rec * D, head, next,
                               hp, stream_);
}

extern "C" int dccf_sum_parts(const float* parts, int32_t n_parts, int64_t part_stride, int64_t n, float* out,
                              void* stream_) {
    DCCF_CHECK_ARG(out && (n_parts == 0 || parts), "dccf_sum_parts: null buffer");
    DCCF_CHECK_ARG(n_parts >= 0 && part_stride >= 0, "dccf_sum_parts: bad layout");
    if (n <= 0) return DCCF_OK;
    int64_t ctas = (n + 255) / 256;
    if (ctas > 148 * 8) ctas = 148 * 8;
    k_sum_parts<<<(unsigned)ctas, 256, 0, (cudaStream_t)stream_>>>(parts, n_parts, part_stride, n, out);
    DCCF_CHECK_LAUNCH("k_sum_parts");
    return DCCF_OK;
}

extern "C" int dccf_adam_dense(float* p, float* m, float* v, int64_t n, const float* g_parts, int32_t n_parts,
                               int64_t part_stride, const dccf_adam* hp, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AdamHost h;
    int rc = check_hp_adam(hp, &h, "dccf_adam_dense");
    if (rc != DCCF_OK) return rc;
    DCCF_CHECK_ARG(p && m && v, "dccf_adam_dense: null buffer");
    DCCF_CHECK_ARG(n_parts == 0 || g_parts, "dccf_adam_dense: null gradient buffer");
    DCCF_CHECK_ARG(n_parts >= 0 && part_stride >= 0, "dccf_adam_dense: bad partial layout");
    if (n <= 0) return DCCF_OK;
    int64_t ctas = (n + 255) / 256;
    if (ctas > 148 * 8) ctas = 148 * 8;
    k_adam_dense<<<(unsigned)ctas, 256, 0, stream>>>(p, m, v, n, g_parts, n_parts, part_stride, h);
    DCCF_CHECK_LAUNCH("k_adam_dense");
    return DCCF_OK;
}

extern "C" int dccf_state_advance(int32_t* step_dev, uint64_t* offset_dev, uint64_t offset_inc, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!step_dev && !offset_dev) return DCCF_OK;
    k_state_advance<<<1, 32, 0, stream>>>(step_dev, offset_dev, offset_inc);
    DCCF_CHECK_LAUNCH("k_state_advance");
    return DCCF_OK;
}

// CTAs of one table's range in a launch of `mode` (see marshal_adam).  total_rows / n_rec_all: over every table of the
// launch.
static int64_t table_blocks(int mode, int64_t n_rows, int64_t total_rows, int64_t n_rec, int64_t n_rec_all) {
    int64_t want;
    if (mode == 2) {
        // 16 records (half-warps) per 256-thread CTA per trip; ALL tables and dense tensors of the launch together stay
        // within one wave (three 256-thread CTAs of this kernel fit an SM: 444, of which the dense tensors take up to
        // 149) — a second wave started only when first-wave CTAs retired (data-parallel steps: 533 CTAs)
        const int64_t table_budget = 148 * 3 - 150;
        want = (n_rec + 15) / 16;
        const int64_t share = n_rec_all > 0 ? (table_budget * n_rec + n_rec_all - 1) / n_rec_all : 0;
        if (want > share) want = share;
        if (want < 1 && n_rec > 0) want = 1;
    } else {
        // CTAs for the table sweeps, shared in proportion to the row counts (mode 3: the wide untouched-row sweep)
        const int64_t budget = (mode == 1) ? 148 : 148 * 8;
        want = (n_rows + 31) / 32;                           // 32 rows per 256-thread CTA per trip
        const int64_t share = total_rows > 0 ? (budget * n_rows + total_rows - 1) / total_rows : 0;
        if (want > share) want = share;
        if (want < 1 && n_rows > 0) want = 1;
    }
    return want;
}

// CTAs of one dense tensor's range (every mode)
static int64_t dense_blocks(int64_t n) {
    const int64_t want = (n + 255) / 256;
    return want > 148 ? 148 : want;
}

// Validate and marshal the table / tensor descriptors.  mode 0: k_adam_all (sweep blocks over all rows);
// 1: k_adam_untouched (sweep blocks, at most one 256-thread CTA per SM so that a tensor-core CTA of the forward /
// backward fits beside it); 2: k_adam_touched (one half-warp per record); 3: the wide k_adam_untouched.
static int marshal_adam(const char* who, const dccf_adam_table* tables, int32_t n_tables, const dccf_adam_tensor* dense,
                        int32_t n_dense, const dccf_adam* hp, int mode, AdamAllArgs& a, int32_t* blocks_out,
                        int32_t* link_blocks_out) {
    int rc = check_hp(hp, &a.hp, who);
    if (rc != DCCF_OK) return rc;
    // state tensors the rule reads and writes: Adam m and v, Adagrad m (state_sum), GD none
    const bool need_m = hp->rule != RULE_GD, need_v = hp->rule == RULE_ADAM;
    DCCF_CHECK_ARG(n_tables >= 0 && n_tables <= ADAM_MAX_T && n_dense >= 0 && n_dense <= ADAM_MAX_T,
                   "%s: at most %d tables and %d dense tensors per call", who, ADAM_MAX_T, ADAM_MAX_T);
    DCCF_CHECK_ARG((n_tables == 0 || tables) && (n_dense == 0 || dense), "%s: null descriptor array", who);
    a.n_tables = n_tables;
    a.n_dense = n_dense;
    int64_t total_rows = 0, n_rec_all = 0;
    for (int i = 0; i < n_tables; ++i) {
        total_rows += tables[i].n_rows > 0 ? tables[i].n_rows : 0;
        n_rec_all += (int64_t)tables[i].n_seg * tables[i].seg_len;
    }
    int32_t blocks = 0, link_blocks = 0;
    for (int i = 0; i < n_tables; ++i) {
        const dccf_adam_table& t = tables[i];
        DCCF_CHECK_ARG(t.table && t.head && (t.m || !need_m) && (t.v || !need_v), "%s: table %d has a null buffer (rule %d)", who, i, hp->rule);
        const int64_t n_rec = (int64_t)t.n_seg * t.seg_len;
        DCCF_CHECK_ARG(t.n_seg >= 0 && t.seg_len >= 0, "%s: table %d has a negative record layout", who, i);
        DCCF_CHECK_ARG(n_rec == 0 || (t.rec_keys && t.rec_grads && t.next), "%s: table %d has records but a null record buffer", who, i);
        DCCF_CHECK_ARG(n_rec < ((int64_t)1 << 31) && t.n_rows < ((int64_t)1 << 31), "%s: table %d exceeds int32 indexing", who, i);
        DCCF_CHECK_ARG(t.n_seg <= 1 || (t.key_seg_stride >= t.seg_len && t.grad_seg_stride >= t.seg_len * D), "%s: table %d segment strides overlap", who, i);
        AdamTableArgs& o = a.t[i];
        o.table = t.table; o.m = t.m; o.v = t.v; o.n_rows = t.n_rows > 0 ? t.n_rows : 0;
        o.keys = t.rec_keys; o.grads = t.rec_grads; o.n_rec = n_rec;
        o.L.seg_len = t.seg_len > 0 ? t.seg_len : 1; o.L.key_seg_stride = t.key_seg_stride; o.L.grad_seg_stride = t.grad_seg_stride;
        o.head = t.head; o.next = t.next;
        const int n_csr = (t.rec_row != nullptr) + (t.csr_off != nullptr) + (t.csr != nullptr) + (t.csr_pool != nullptr);
        DCCF_CHECK_ARG(n_csr == 0 || n_csr == 4, "%s: table %d: the CSR buffers (rec_row, csr_off, csr, csr_pool) go together", who, i);
        o.rec_row = t.rec_row; o.csr_off = t.csr_off; o.csr = t.csr; o.csr_pool = t.csr_pool;
        const int64_t want = table_blocks(mode, o.n_rows, total_rows, n_rec, n_rec_all);
        o.block_lo = blocks; o.block_n = (int32_t)want; blocks += (int32_t)want;
        o.link_lo = link_blocks; o.link_n = (int32_t)((n_rec + 255) / 256); link_blocks += o.link_n;
    }
    for (int i = 0; i < n_dense; ++i) {
        const dccf_adam_tensor& d = dense[i];
        DCCF_CHECK_ARG(d.p && (d.m || !need_m) && (d.v || !need_v), "%s: dense tensor %d has a null buffer (rule %d)", who, i, hp->rule);
        DCCF_CHECK_ARG(d.n_parts == 0 || d.g_parts, "%s: dense tensor %d has a null gradient", who, i);
        AdamDenseArgs& o = a.d[i];
        o.p = d.p; o.m = d.m; o.v = d.v; o.n = d.n > 0 ? d.n : 0; o.g_parts = d.g_parts; o.n_parts = d.n_parts;
        o.part_stride = d.part_stride;
        const int64_t want = dense_blocks(o.n);
        o.block_lo = blocks; o.block_n = (int32_t)want; blocks += (int32_t)want;
    }
    *blocks_out = blocks;
    *link_blocks_out = link_blocks;
    return DCCF_OK;
}

extern "C" int32_t dccf_adam_blocks(int32_t mode, const int64_t* n_rows, const int64_t* n_rec, int32_t n_tables,
                                    const int64_t* n_dense_elems, int32_t n_dense, int32_t* block_lo, int32_t* block_n) {
    if (mode < 0 || mode > 3 || n_tables < 0 || n_tables > ADAM_MAX_T || n_dense < 0 || n_dense > ADAM_MAX_T ||
        (n_tables > 0 && (n_rows == nullptr || n_rec == nullptr)) || (n_dense > 0 && n_dense_elems == nullptr) ||
        (n_tables + n_dense > 0 && (block_lo == nullptr || block_n == nullptr)))
        return -1;
    int64_t total_rows = 0, n_rec_all = 0;
    for (int i = 0; i < n_tables; ++i) {
        if (n_rows[i] < 0 || n_rec[i] < 0) return -1;
        total_rows += n_rows[i];
        n_rec_all += n_rec[i];
    }
    for (int i = 0; i < n_dense; ++i)
        if (n_dense_elems[i] < 0) return -1;
    int32_t blocks = 0;
    for (int i = 0; i < n_tables + n_dense; ++i) {
        const int64_t want = i < n_tables ? table_blocks(mode, n_rows[i], total_rows, n_rec[i], n_rec_all)
                                          : dense_blocks(n_dense_elems[i - n_tables]);
        block_lo[i] = blocks; block_n[i] = (int32_t)want; blocks += (int32_t)want;
    }
    return blocks;
}

extern "C" int dccf_adam_step(const dccf_adam_table* tables, int32_t n_tables, const dccf_adam_tensor* dense,
                              int32_t n_dense, const dccf_adam* hp, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AdamAllArgs a;
    int32_t blocks = 0, link_blocks = 0;
    int rc = marshal_adam("dccf_adam_step", tables, n_tables, dense, n_dense, hp, 0, a, &blocks, &link_blocks);
    if (rc != DCCF_OK) return rc;
    if (link_blocks > 0) {
        k_link_all<<<(unsigned)link_blocks, 256, 0, stream>>>(a);
        DCCF_CHECK_LAUNCH("k_link_all");
    }
    if (blocks > 0) {
        k_all_of[hp->rule]<<<(unsigned)blocks, 256, 0, stream>>>(a);
        DCCF_CHECK_LAUNCH(all_name[hp->rule]);
    }
    return DCCF_OK;
}

extern "C" int dccf_debug_timeline_adam(unsigned long long* slots) {
    cudaError_t e = cudaMemcpyToSymbol(g_timeline, &slots, sizeof(slots));
    if (e != cudaSuccess) {
        set_error("dccf_debug_timeline: %s", cudaGetErrorString(e));
        return DCCF_ERR_CUDA;
    }
    return DCCF_OK;
}

extern "C" int dccf_adam_link_ids(const dccf_dims* dims, const int64_t* X, const int64_t* sample_item, int64_t n_pairs,
                                  int32_t n_seg, int64_t seg_stride, int32_t user_seg, int32_t* head_user,
                                  int32_t* next_user, int32_t* head_item, int32_t* next_item, const dccf_expo* expo,
                                  const int64_t* X_local, const int64_t* sample_item_local, float* expo_e,
                                  float* expo_den, const dccf_link_extra* extra, void* stream_) {
    const bool staged = extra != nullptr && extra->epoch_ptrs_dev != nullptr;
    DCCF_CHECK_ARG(dims && (X || staged) && head_user && next_user && head_item && next_item, "dccf_adam_link_ids: null argument");
    DCCF_CHECK_ARG(dims->n_samples == 0 || sample_item || staged, "dccf_adam_link_ids: sample_item is null");
    const bool epoch_link = staged && extra->X_out == nullptr;      // segments come from the epoch-wide gather (strides in device memory)
    DCCF_CHECK_ARG(n_seg >= 0 && (n_seg <= 1 || seg_stride > 0 || epoch_link) && (n_seg == 0 || user_seg < n_seg), "dccf_adam_link_ids: bad segment layout");
    DCCF_CHECK_ARG(n_seg > 0 || expo != nullptr || staged, "dccf_adam_link_ids: nothing to do (n_seg == 0 and no exposure source)");
    DCCF_CHECK_ARG(n_pairs * n_seg * (dims->n_samples + 1) < ((int64_t)1 << 31), "dccf_adam_link_ids: too many records");
    DCCF_CHECK_ARG(expo == nullptr || (expo_e && expo_den), "dccf_adam_link_ids: expo needs expo_e and expo_den");
    const bool epoch_global = staged && extra->X_out == nullptr;
    DCCF_CHECK_ARG(!staged || epoch_global || (n_seg <= 1 && extra->cursor_dev && (dims->n_samples == 0 || extra->sample_item_out)),
                   "dccf_adam_link_ids: staging needs n_seg <= 1, the cursor and the output buffers");
    DCCF_CHECK_ARG(!epoch_global || (extra->cursor_dev != nullptr && n_seg >= 1), "dccf_adam_link_ids: the epoch-wide link needs the cursor and n_seg >= 1");
    DCCF_CHECK_ARG(extra == nullptr || extra->Y_out == nullptr || (staged && !epoch_global), "dccf_adam_link_ids: Y_out needs staging (epoch_ptrs_dev and X_out)");
    if (n_pairs <= 0) return DCCF_OK;
    LinkIdsArgs a;
    a.X = X; a.sample_item = sample_item; a.n_pairs = n_pairs; a.S = dims->n_samples; a.A = dims->n_attr;
    a.X_local = X_local ? X_local : X; a.si_local = X_local ? sample_item_local : sample_item;
    a.n_seg = n_seg; a.seg_stride = seg_stride; a.user_seg = user_seg;
    a.user_base = dims->user_base; a.n_users = dims->n_users; a.n_items = dims->n_items;
    a.head_u = head_user; a.next_u = next_user; a.head_i = head_item; a.next_i = next_item;
    a.feat_dim = dims->feat_dim;
    if (extra != nullptr) {
        a.extra = *extra;
    } else {
        a.extra.epoch_ptrs_dev = nullptr; a.extra.cursor_dev = nullptr; a.extra.X_out = nullptr;
        a.extra.sample_item_out = nullptr; a.extra.Y_out = nullptr; a.extra.stage_counter = nullptr; a.extra.pf_feat = nullptr; a.extra.sync = nullptr;
        a.extra.rec_row_user = nullptr; a.extra.rec_row_item = nullptr;
        for (int k = 0; k < 3; ++k) { a.extra.pf_user[k] = nullptr; a.extra.pf_item[k] = nullptr; }
        for (int k = 0; k < 4; ++k) { a.extra.pf_dense[k] = nullptr; a.extra.pf_dense_bytes[k] = 0; }
    }
    int rc_sync = marshal_sync("dccf_adam_link_ids", extra != nullptr ? extra->sync : nullptr, &a.sync);
    if (rc_sync != DCCF_OK) return rc_sync;
    DCCF_CHECK_ARG(a.sync.n_done == 0 || a.extra.stage_counter != nullptr, "dccf_adam_link_ids: sync needs stage_counter (the CTA counter)");
    DCCF_CHECK_ARG((a.extra.rec_row_user == nullptr) == (a.extra.rec_row_item == nullptr), "dccf_adam_link_ids: counting mode needs rec_row of both tables");
    a.extra.sync = nullptr;
    const int64_t n = n_pairs * (n_seg > 0 ? n_seg : ((staged && !epoch_global) ? 1 : 0)) * (dims->n_samples + 2);
    a.link_blocks = (int32_t)((n + 255) / 256);
    int64_t blocks = a.link_blocks;
    a.expo_e = expo_e; a.expo_den = expo_den;
    a.expo_blocks = 0;
    if (expo != nullptr) {
        a.ex = *expo;
        a.expo_blocks = (int32_t)((n_pairs + 7) / 8);
        blocks += a.expo_blocks;
    } else {
        a.ex.mode = 0; a.ex.dense = nullptr;
    }
    int64_t dense_bytes = 0;
    for (int k = 0; k < 4; ++k) dense_bytes += a.extra.pf_dense[k] != nullptr ? a.extra.pf_dense_bytes[k] : 0;
    if (dense_bytes > 0) {
        int64_t pf = (dense_bytes / 128 + 255) / 256;
        blocks += pf > 16 ? 16 : (pf < 1 ? 1 : pf);
    }
    // same shared-memory carveout as the tensor-core kernels that follow it in the step: a kernel that asks for another
    // L1 / shared split makes its successor wait for the SMs to be reconfigured
    static PerDeviceOnce carve_once;
    if (carve_once.need()) {
        cudaFuncSetAttribute(k_link_ids, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        carve_once.mark();
    }
    k_link_ids<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream_>>>(a);
    DCCF_CHECK_LAUNCH("k_link_ids");
    return DCCF_OK;
}

extern "C" int dccf_adam_untouched(const dccf_adam_table* tables, int32_t n_tables, const dccf_adam* hp,
                                   int32_t threads_per_cta, void* stream_) {
    AdamAllArgs a;
    int32_t blocks = 0, link_blocks = 0;
    // record buffers are not read by this kernel: strip them so the validation does not demand them
    dccf_adam_table local[ADAM_MAX_T];
    DCCF_CHECK_ARG(n_tables >= 0 && n_tables <= ADAM_MAX_T && (n_tables == 0 || tables), "dccf_adam_untouched: bad table array");
    for (int i = 0; i < n_tables; ++i) {
        local[i] = tables[i];
        local[i].n_seg = 0; local[i].seg_len = 0;
    }
    // threads_per_cta < 0: WIDE sweep — the tables are so large (scaled configuration: 10^7 user rows) that the sweep,
    // not the forward / backward, bounds the step: full occupancy (8 CTAs of 256 threads per SM, no shared-memory
    // limiter) instead of one small CTA per SM hidden beside the tensor-core kernels.
    const bool wide = threads_per_cta < 0;
    int rc = marshal_adam("dccf_adam_untouched", local, n_tables, nullptr, 0, hp, wide ? 3 : 1, a, &blocks, &link_blocks);
    if (rc != DCCF_OK) return rc;
    const StepKernel kernel = k_untouched_of[hp->rule];
    if (blocks > 0 && wide) {
        kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream_>>>(a);
        DCCF_CHECK_LAUNCH(untouched_name[hp->rule]);
        return DCCF_OK;
    }
    if (blocks > 0) {
        // Occupancy limiter: the sweep runs beside the tensor-core kernels of the forward / backward (96 KB of shared
        // memory, ~48 K registers per CTA).  Two sweep CTAs on one SM would leave no room for such a CTA and push it
        // into a second wave, so every sweep CTA reserves (and never touches) 120 KB of dynamic shared memory:
        // at most one per SM, and 120 + 96 KB still fit the 227 KB of an SM.
        static PerDeviceOnce attr_once[3];
        if (attr_once[hp->rule].need()) {
            cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ADAM_SIDE_SMEM);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            if (e != cudaSuccess) {
                set_error("dccf_adam_untouched: cannot opt in to %d bytes of shared memory: %s", ADAM_SIDE_SMEM, cudaGetErrorString(e));
                return DCCF_ERR_CUDA;
            }
            attr_once[hp->rule].mark();
        }
        // threads_per_cta (0 = default 224).  The CTA has to stay resident beside the tensor-core kernels AND the middle
        // kernel (768 threads x 64 registers = 3/4 of the register file): 7 warps x 64 registers fit, 8 do not.  Measured (tools/step_timeline.py, electronics shape, L2 flushed): 128 threads swept
        // the tables in 46 us — the longest chain of the step once k_link_ids had left the forward's way; a launch
        // that did not fit beside the middle kernel (160 / 192 threads at 70 registers) held that kernel back until the
        // sweep had finished (+15 us).
        const int side_threads = (threads_per_cta >= 32 && threads_per_cta <= 256) ? (threads_per_cta / 32) * 32 : 224;
        kernel<<<(unsigned)blocks, side_threads, ADAM_SIDE_SMEM, (cudaStream_t)stream_>>>(a);
        DCCF_CHECK_LAUNCH(untouched_name[hp->rule]);
    }
    return DCCF_OK;
}

extern "C" int dccf_adam_csr_build(const dccf_adam_table* tables, int32_t n_tables, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AdamAllArgs a;
    int32_t blocks = 0, link_blocks = 0;
    dccf_adam hp;
    hp.lr = 0; hp.beta1 = 0.9; hp.beta2 = 0.999; hp.eps = 0; hp.l2 = 0; hp.weight_decay = 0; hp.clip = 0; hp.step = 1; hp.step_dev = nullptr;
    hp.rule = RULE_GD;      // (this launch reads no optimizer state: validated as the rule without any)
    int rc = marshal_adam("dccf_adam_csr_build", tables, n_tables, nullptr, 0, &hp, 2, a, &blocks, &link_blocks);
    if (rc != DCCF_OK) return rc;
    for (int i = 0; i < n_tables; ++i)
        DCCF_CHECK_ARG(tables[i].csr != nullptr || (int64_t)tables[i].n_seg * tables[i].seg_len == 0, "dccf_adam_csr_build: table %d has records but no CSR buffers", i);
    if (link_blocks == 0) return DCCF_OK;
    k_csr_build<<<(unsigned)link_blocks, 256, 0, stream>>>(a, 0);
    DCCF_CHECK_LAUNCH("k_csr_build");
    k_csr_build<<<(unsigned)link_blocks, 256, 0, stream>>>(a, 1);
    DCCF_CHECK_LAUNCH("k_csr_build");
    return DCCF_OK;
}

extern "C" int dccf_adam_touched(const dccf_adam_table* tables, int32_t n_tables, const dccf_adam_tensor* dense,
                                 int32_t n_dense, const dccf_adam* hp, int32_t already_linked, float* w_image,
                                 int32_t w_image_tensor, int32_t w_image_K, int32_t* cta_counter, int32_t* advance_step_dev,
                                 uint64_t* advance_offset_dev, int64_t* advance_cursor_dev, const dccf_dp_sync* sync,
                                 void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    AdamAllArgs a;
    int32_t blocks = 0, link_blocks = 0;
    int rc = marshal_adam("dccf_adam_touched", tables, n_tables, dense, n_dense, hp, 2, a, &blocks, &link_blocks);
    if (rc != DCCF_OK) return rc;
    DCCF_CHECK_ARG(w_image == nullptr || (w_image_tensor >= 0 && w_image_tensor < n_dense && w_image_K > 0 && w_image_K % 32 == 0 &&
                                          dense[w_image_tensor].n == (int64_t)D * w_image_K),
                   "dccf_adam_touched: the W image needs the index of W [D, K] among the dense tensors and K %% 32 == 0");
    WImageArgs wi;
    wi.img = w_image; wi.tensor = w_image_tensor; wi.K = w_image_K;
    wi.cta_counter = cta_counter; wi.step_dev = advance_step_dev; wi.offset_dev = advance_offset_dev;
    wi.cursor_dev = advance_cursor_dev;
    DCCF_CHECK_ARG(cta_counter != nullptr || (advance_step_dev == nullptr && advance_offset_dev == nullptr && advance_cursor_dev == nullptr),
                   "dccf_adam_touched: advancing the counters needs cta_counter");
    DpSync ds;
    rc = marshal_sync("dccf_adam_touched", sync, &ds);
    if (rc != DCCF_OK) return rc;
    DCCF_CHECK_ARG((ds.n_done == 0 && ds.loss_out == nullptr) || cta_counter != nullptr, "dccf_adam_touched: sync needs cta_counter");
    if (link_blocks > 0 && !already_linked) {
        for (int i = 0; i < n_tables; ++i)
            DCCF_CHECK_ARG(tables[i].csr == nullptr, "dccf_adam_touched: CSR tables need dccf_adam_link_ids + dccf_adam_csr_build (already_linked = 1)");
        k_link_all<<<(unsigned)link_blocks, 256, 0, stream>>>(a);
        DCCF_CHECK_LAUNCH("k_link_all");
    }
    const TouchedKernel kernel = k_touched_of[hp->rule];
    static PerDeviceOnce carve_once[3];
    if (carve_once[hp->rule].need()) {
        cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        carve_once[hp->rule].mark();
    }
    if (blocks > 0) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)blocks); cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = 0; cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = ((ds.flags & DCCF_DP_SYNC_OVERLAP_PUSH) && ds.n_wait >= 2 && already_linked) ? 1 : 0;
        cudaError_t le = cudaLaunchKernelEx(&cfg, kernel, a, wi, ds);
        if (le != cudaSuccess) {
            set_error("%s: launch failed: %s", touched_name[hp->rule], cudaGetErrorString(le));
            return DCCF_ERR_CUDA;
        }
        DCCF_CHECK_LAUNCH(touched_name[hp->rule]);
    }
    return DCCF_OK;
}

extern "C" int dccf_stage_batch(const uint64_t* epoch_ptrs_dev, int64_t* cursor_dev, int64_t n_pairs, int32_t n_samples,
                                int64_t* X_out, int64_t* sample_item_out, float* Y_out, void* stream_) {
    DCCF_CHECK_ARG(epoch_ptrs_dev && cursor_dev && X_out && (n_samples == 0 || sample_item_out), "dccf_stage_batch: null argument");
    DCCF_CHECK_ARG(n_pairs >= 0 && n_samples >= 0, "dccf_stage_batch: negative size");
    if (n_pairs == 0) return DCCF_OK;
    static PerDeviceOnce carve_once;
    if (carve_once.need()) {
        cudaFuncSetAttribute(k_stage_batch, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
        carve_once.mark();
    }
    k_stage_batch<<<1, 1024, 0, (cudaStream_t)stream_>>>(epoch_ptrs_dev, cursor_dev, n_pairs * 2, n_pairs * n_samples, X_out,
                                                         sample_item_out, Y_out);
    DCCF_CHECK_LAUNCH("k_stage_batch");
    return DCCF_OK;
}
