// MoE router: LayerNorm + Linear(E) + noise + softmax + top-K + normalised weights + aux-loss sums,
// and its backward.  Replaces core.py:480-492, 499-505, 524-529 and their autograd.
//
// Forward: one warp per token.  The row is read twice (mean, then centred second moment + the E dot
// products in the same pass; the second read hits L1), LayerNorm affine is folded into the router
// weight once per CTA (G[e,d] = ln_w[d]*Wr[e,d] in shared memory; c[e] = sum_d ln_b[d]*Wr[e,d] + br[e]).
// Lanes 0..E-1 then own one expert each for softmax / top-K.  Ties in top-K go to the lower expert id.
#include <cuda_fp16.h>

#include "common.cuh"

namespace {

constexpr int WARPS = 8;
constexpr int MAX_K = 8;

// round-trip through the autocast dtype (round to nearest even, like torch's casts)
__device__ __forceinline__ float ab_round_to(float v, int quant) {
    if (quant == AB_ROUTER_BF16) return __bfloat162float(__float2bfloat16_rn(v));
    if (quant == AB_ROUTER_FP16) return __half2float(__float2half_rn(v));
    return v;
}

template <typename T>
__device__ __forceinline__ void row_load(const T* row, int i, float* f) {   // vector i of the row
    ab_vec16<T>::unpack(__ldg(reinterpret_cast<const uint4*>(row) + i), f);
}

// four consecutive elements: one 16-byte (fp32) or 8-byte (bf16) access
template <typename T>
__device__ __forceinline__ void ld4g(const T* p, float* f) {
    if constexpr (sizeof(T) == 4) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(p));
        f[0] = q.x; f[1] = q.y; f[2] = q.z; f[3] = q.w;
    } else {
        const uint2 r = __ldg(reinterpret_cast<const uint2*>(p));
        f[0] = __uint_as_float(r.x << 16); f[1] = __uint_as_float(r.x & 0xffff0000u);
        f[2] = __uint_as_float(r.y << 16); f[3] = __uint_as_float(r.y & 0xffff0000u);
    }
}
template <typename T>
__device__ __forceinline__ void ab_st4(T* p, const float* o) {
    if constexpr (sizeof(T) == 4) {
        *reinterpret_cast<float4*>(p) = make_float4(o[0], o[1], o[2], o[3]);
    } else {
        __nv_bfloat162 lo = __floats2bfloat162_rn(o[0], o[1]), hi = __floats2bfloat162_rn(o[2], o[3]);
        *reinterpret_cast<uint2*>(p) = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
    }
}

// softmax / top-K / weights on lanes (lane e < E holds logit e).  Returns the gate in g; lane k < K ends up holding
// slot k's expert id and probability (my_idx, my_p) -- no per-thread arrays, so nothing spills to local memory.
__device__ __forceinline__ void select_topk(float logit, int lane, int E, int K, float& g, float& lse, int& my_idx, float& my_p,
                                            float& den, unsigned& sel_mask) {
    const float lv = lane < E ? logit : -INFINITY;
    const float m = ab_warp_max(lv);
    const float ex = lane < E ? expf(lv - m) : 0.f;
    const float sum = ab_warp_sum(ex);
    g = ex / sum;
    lse = m + logf(sum);
    float cand = lane < E ? g : -INFINITY;
    my_idx = 0; my_p = 0.f; den = 0.f; sel_mask = 0u;
    for (int k = 0; k < K; ++k) {
        const float best = ab_warp_max(cand);
        const unsigned ball = __ballot_sync(0xffffffffu, cand == best);
        const int win = __ffs(ball) - 1;               // lowest expert id among equals
        if (lane == k) { my_idx = win; my_p = best; }
        den += best;                                   // summed in slot order like torch.sum over K
        sel_mask |= 1u << win;
        if (lane == win) cand = -INFINITY;
    }
    den += 1e-6f;
}

__device__ __forceinline__ void write_selection(int s, int lane, int E, int K, float g, float lse, int my_idx, float my_p, float den,
                                                float* gates, int32_t* idx, float* probs, float* w, float* lse_out) {
    if (lane < E) gates[(size_t)s * E + lane] = g;
    if (lane < K) {
        idx[(size_t)s * K + lane] = my_idx;
        probs[(size_t)s * K + lane] = my_p;
        w[(size_t)s * K + lane] = my_p / den;
    }
    if (lane == 0) lse_out[s] = lse;
}

// aux partial layout per CTA: [2E+1] = sum gates[e], count[e], sum lse^2
template <typename T, int EM>
__global__ void __launch_bounds__(WARPS * 32) router_fwd_kernel(const T* __restrict__ x, const float* __restrict__ ln_w,
                                                                const float* __restrict__ ln_b, float eps,
                                                                const float* __restrict__ Wr, const float* __restrict__ br,
                                                                const float* __restrict__ noise,
                                                                const float* __restrict__ noise_scale, float* __restrict__ lclean,
                                                                float* __restrict__ logits, float* __restrict__ gates,
                                                                int32_t* __restrict__ idx, float* __restrict__ probs,
                                                                float* __restrict__ w, float* __restrict__ lse_out,
                                                                float* __restrict__ stats, float* __restrict__ part, int S,
                                                                int Dm, int E, int K, int quant) {
    constexpr int V = ab_vec16<T>::N;
    extern __shared__ float sm[];
    float* G = sm;                 // [E][Dm]
    float* cvec = G + (size_t)E * Dm;   // [E]
    float* red = cvec + 32;        // [WARPS][2E+1]
    float* lnw_s = red + WARPS * (2 * E + 1);      // [Dm], [Dm]: LayerNorm affine (quant modes only)
    float* lnb_s = lnw_s + Dm;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (quant == AB_ROUTER_EXACT) {
        for (int e = 0; e < E; ++e)
            for (int d = tid; d < Dm; d += blockDim.x) G[(size_t)e * Dm + d] = ln_w[d] * Wr[(size_t)e * Dm + d];
        for (int e = warp; e < E; e += WARPS) {
            float acc = 0.f;
            for (int d = lane; d < Dm; d += 32) acc = fmaf(ln_b[d], Wr[(size_t)e * Dm + d], acc);
            acc = ab_warp_sum(acc);
            if (lane == 0) cvec[e] = acc + br[e];
        }
    } else {
        // autocast emulation (core.py:482 under torch.autocast): the router Linear sees its input, weight and bias rounded
        // to the autocast dtype, accumulates in fp32 and rounds its output once
        for (int e = 0; e < E; ++e)
            for (int d = tid; d < Dm; d += blockDim.x) G[(size_t)e * Dm + d] = ab_round_to(Wr[(size_t)e * Dm + d], quant);
        for (int d = tid; d < Dm; d += blockDim.x) { lnw_s[d] = ln_w[d]; lnb_s[d] = ln_b[d]; }
        if (tid < E) cvec[tid] = ab_round_to(br[tid], quant);
    }
    __syncthreads();
    const int nvec = Dm / V;
    float a_g = 0.f, a_cnt = 0.f, a_l2 = 0.f;
    for (int s = blockIdx.x * WARPS + warp; s < S; s += gridDim.x * WARPS) {
        const T* row = x + (size_t)s * Dm;
        float sum = 0.f;
        for (int i = lane; i < nvec; i += 32) {
            float f[V];
            row_load<T>(row, i, f);
#pragma unroll
            for (int v = 0; v < V; ++v) sum += f[v];
        }
        const float mean = ab_warp_sum(sum) / (float)Dm;
        float var = 0.f;
        float dot[EM];
#pragma unroll
        for (int e = 0; e < EM; ++e) dot[e] = 0.f;
        for (int i = lane; i < nvec; i += 32) {
            float f[V];
            row_load<T>(row, i, f);
#pragma unroll
            for (int v = 0; v < V; ++v) { f[v] -= mean; var = fmaf(f[v], f[v], var); }
#pragma unroll
            for (int e = 0; e < EM; ++e) {
                if (e < E) {
#pragma unroll
                    for (int v4 = 0; v4 < V; v4 += 4) {
                        const float4 gq = *reinterpret_cast<const float4*>(G + (size_t)e * Dm + i * V + v4);
                        dot[e] = fmaf(f[v4], gq.x, dot[e]); dot[e] = fmaf(f[v4 + 1], gq.y, dot[e]);
                        dot[e] = fmaf(f[v4 + 2], gq.z, dot[e]); dot[e] = fmaf(f[v4 + 3], gq.w, dot[e]);
                    }
                }
            }
        }
        var = ab_warp_sum(var) / (float)Dm;
        const float rstd = rsqrtf(var + eps);
        if (quant != AB_ROUTER_EXACT) {
            // third pass over the (L1-resident) row: the normalised row rounded element by element, then the dot products
#pragma unroll
            for (int e = 0; e < EM; ++e) dot[e] = 0.f;
            for (int i = lane; i < nvec; i += 32) {
                float f[V];
                row_load<T>(row, i, f);
#pragma unroll
                for (int v = 0; v < V; ++v) f[v] = ab_round_to(fmaf((f[v] - mean) * rstd, lnw_s[i * V + v], lnb_s[i * V + v]), quant);
#pragma unroll
                for (int e = 0; e < EM; ++e) {
                    if (e < E) {
#pragma unroll
                        for (int v = 0; v < V; ++v) dot[e] = fmaf(f[v], G[(size_t)e * Dm + i * V + v], dot[e]);
                    }
                }
            }
        }
        float mylogit = 0.f;
#pragma unroll
        for (int e = 0; e < EM; ++e) {
            if (e < E) {
                const float t = ab_warp_sum(dot[e]);
                if (lane == e) mylogit = t;
            }
        }
        float lc = 0.f;
        if (lane < E) {
            lc = quant == AB_ROUTER_EXACT ? fmaf(rstd, mylogit, cvec[lane]) : ab_round_to(mylogit + cvec[lane], quant);
            mylogit = lc;
            if (noise) mylogit = fmaf(noise[(size_t)s * E + lane], noise_scale[lane], lc);
            if (lclean) lclean[(size_t)s * E + lane] = lc;
            if (logits) logits[(size_t)s * E + lane] = mylogit;
        }
        if (lane == 0) { stats[2 * (size_t)s] = mean; stats[2 * (size_t)s + 1] = rstd; }
        float g, lse, my_p, den;
        int my_idx;
        unsigned sel_mask;
        select_topk(mylogit, lane, E, K, g, lse, my_idx, my_p, den, sel_mask);
        write_selection(s, lane, E, K, g, lse, my_idx, my_p, den, gates, idx, probs, w, lse_out);
        if (lane < E) {
            a_g += g;
            a_cnt += (sel_mask >> lane) & 1u ? 1.f : 0.f;
        }
        if (lane == 0) a_l2 = fmaf(lse, lse, a_l2);
    }
    const int NA = 2 * E + 1;
    if (lane < E) { red[warp * NA + lane] = a_g; red[warp * NA + E + lane] = a_cnt; }
    if (lane == 0) red[warp * NA + 2 * E] = a_l2;
    __syncthreads();
    if (tid < NA) {
        float s2 = 0.f;
        for (int wv = 0; wv < WARPS; ++wv) s2 += red[wv * NA + tid];
        part[(size_t)blockIdx.x * NA + tid] = s2;
    }
}

// Same forward with the token's row held in registers (hidden sizes up to 32 * V * NV): one global read of the row, the
// E dot products read G as 16-byte vectors, and for E <= 8 the E partial sums of the 32 lanes are reduced by recursive
// halving (10 shuffles instead of 5 per expert).  The launcher picks this kernel whenever the row fits.
template <int EM>
__device__ __forceinline__ float reduce_dots_to_lane(float (&dot)[EM], int lane, int E) {
    float mine = 0.f;
    if (EM == 8) {
        // halve the vector while doubling the lanes per value: after xor 16 / 8 / 4 a lane holds ONE expert's partial sum
        float v4[4], v2[2], v1;
        const bool h16 = lane & 16, h8 = lane & 8, h4 = lane & 4;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float keep = h16 ? dot[4 + j] : dot[j], send = h16 ? dot[j] : dot[4 + j];
            v4[j] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const float keep = h8 ? v4[2 + j] : v4[j], send = h8 ? v4[j] : v4[2 + j];
            v2[j] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
        {
            const float keep = h4 ? v2[1] : v2[0], send = h4 ? v2[0] : v2[1];
            v1 = keep + __shfl_xor_sync(0xffffffffu, send, 4);
        }
        v1 += __shfl_xor_sync(0xffffffffu, v1, 2);
        v1 += __shfl_xor_sync(0xffffffffu, v1, 1);
        // lanes with bits (4,3,2) = (e2,e1,e0) hold expert e's total: hand it to lane e
        const int src = ((lane >> 2) & 1) << 4 | ((lane >> 1) & 1) << 3 | (lane & 1) << 2;
        mine = __shfl_sync(0xffffffffu, v1, src);
        if (lane >= E) mine = 0.f;
    } else {
#pragma unroll
        for (int e = 0; e < EM; ++e) {
            if (e < E) {
                const float t = ab_warp_sum(dot[e]);
                if (lane == e) mine = t;
            }
        }
    }
    return mine;
}

template <typename T, int EM, int NV>
#ifndef FWD_MINB
#define FWD_MINB 2
#endif
#ifndef FWD_REGPF
#define FWD_REGPF 1
#endif
#ifndef FWD_PERSIST
#define FWD_PERSIST 1
#endif
__global__ void __launch_bounds__(WARPS * 32, (NV * ab_vec16<T>::N <= 24 && EM <= 8) ? FWD_MINB : 1) router_fwd_reg_kernel(const T* __restrict__ x, const float* __restrict__ ln_w,
                                                                    const float* __restrict__ ln_b, float eps,
                                                                    const float* __restrict__ Wr, const float* __restrict__ br,
                                                                    const float* __restrict__ noise,
                                                                    const float* __restrict__ noise_scale, float* __restrict__ lclean,
                                                                    float* __restrict__ logits, float* __restrict__ gates,
                                                                    int32_t* __restrict__ idx, float* __restrict__ probs,
                                                                    float* __restrict__ w, float* __restrict__ lse_out,
                                                                    float* __restrict__ stats, float* __restrict__ part, int S,
                                                                    int Dm, int E, int K, int quant) {
    constexpr int V = ab_vec16<T>::N;
    extern __shared__ float sm[];
    float* G = sm;                 // [E][Dm]
    float* cvec = G + (size_t)E * Dm;   // [E]
    float* red = cvec + 32;        // [WARPS][2E+1]
    float* lnw_s = red + WARPS * (2 * E + 1);      // [Dm], [Dm]: LayerNorm affine (quant modes only)
    float* lnb_s = lnw_s + Dm;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (quant == AB_ROUTER_EXACT) {
        for (int i = tid; i < E * Dm; i += blockDim.x) G[i] = ln_w[i % Dm] * Wr[i];
        for (int e = warp; e < E; e += WARPS) {
            float acc = 0.f;
            for (int d = lane; d < Dm; d += 32) acc = fmaf(ln_b[d], Wr[(size_t)e * Dm + d], acc);
            acc = ab_warp_sum(acc);
            if (lane == 0) cvec[e] = acc + br[e];
        }
    } else {
        for (int i = tid; i < E * Dm; i += blockDim.x) G[i] = ab_round_to(Wr[i], quant);
        for (int d = tid; d < Dm; d += blockDim.x) { lnw_s[d] = ln_w[d]; lnb_s[d] = ln_b[d]; }
        if (tid < E) cvec[tid] = ab_round_to(br[tid], quant);
    }
    __syncthreads();
    const int nvec = Dm / V;
    const float inv_dm = 1.0f / (float)Dm;
    float a_g = 0.f, a_cnt = 0.f, a_l2 = 0.f;
    // the warp's next row is loaded while the current one is reduced: its loads are in flight during the dependent chain
    // of reductions, dot products and top-K of this row.  Rows of more than 64 values per lane would not fit twice.
    constexpr bool PF = FWD_REGPF && NV * V <= 64;
    float fn[NV][V];
    auto load_row = [&](int s) {
        const T* row = x + (size_t)s * Dm;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int iv = i * 32 + lane;
            if (s < S && iv < nvec) {
                row_load<T>(row, iv, fn[i]);
            } else {
#pragma unroll
                for (int v = 0; v < V; ++v) fn[i][v] = 0.f;
            }
        }
    };
    const int stride = gridDim.x * WARPS;
    if constexpr (PF) load_row(blockIdx.x * WARPS + warp);
    for (int s = blockIdx.x * WARPS + warp; s < S; s += stride) {
        if constexpr (!PF) {
            load_row(s);
            // the warp's next row into L2 while this one is reduced (no registers held)
            const char* nx = reinterpret_cast<const char*>(x + (size_t)(s + stride) * Dm);
            if (s + stride < S)
                for (int o = lane * 128; o < Dm * (int)sizeof(T); o += 32 * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(nx + o));
        }
        float f[NV][V];
#pragma unroll
        for (int i = 0; i < NV; ++i) {
#pragma unroll
            for (int v = 0; v < V; ++v) f[i][v] = fn[i][v];
        }
        if constexpr (PF) load_row(s + stride);
        float sum = 0.f;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            if (i * 32 + lane < nvec) {
#pragma unroll
                for (int v = 0; v < V; ++v) sum += f[i][v];
            }
        }
        const float mean = ab_warp_sum(sum) * inv_dm;
        float var = 0.f;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            if (i * 32 + lane < nvec) {
#pragma unroll
                for (int v = 0; v < V; ++v) { f[i][v] -= mean; var = fmaf(f[i][v], f[i][v], var); }
            }
        }
        var = ab_warp_sum(var) * inv_dm;
        const float rstd = rsqrtf(var + eps);
        float dot[EM];
#pragma unroll
        for (int e = 0; e < EM; ++e) dot[e] = 0.f;
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            const int iv = i * 32 + lane;
            if (iv < nvec) {
                if (quant != AB_ROUTER_EXACT) {
                    // autocast emulation: the normalised row rounded element by element before the Linear
#pragma unroll
                    for (int v4 = 0; v4 < V; v4 += 4) {
                        const float4 lw = *reinterpret_cast<const float4*>(lnw_s + iv * V + v4);
                        const float4 lb = *reinterpret_cast<const float4*>(lnb_s + iv * V + v4);
                        f[i][v4] = ab_round_to(fmaf(f[i][v4] * rstd, lw.x, lb.x), quant);
                        f[i][v4 + 1] = ab_round_to(fmaf(f[i][v4 + 1] * rstd, lw.y, lb.y), quant);
                        f[i][v4 + 2] = ab_round_to(fmaf(f[i][v4 + 2] * rstd, lw.z, lb.z), quant);
                        f[i][v4 + 3] = ab_round_to(fmaf(f[i][v4 + 3] * rstd, lw.w, lb.w), quant);
                    }
                }
#pragma unroll
                for (int e = 0; e < EM; ++e) {
                    if (e < E) {
#pragma unroll
                        for (int v4 = 0; v4 < V; v4 += 4) {
                            const float4 gq = *reinterpret_cast<const float4*>(G + (size_t)e * Dm + iv * V + v4);
                            dot[e] = fmaf(f[i][v4], gq.x, dot[e]); dot[e] = fmaf(f[i][v4 + 1], gq.y, dot[e]);
                            dot[e] = fmaf(f[i][v4 + 2], gq.z, dot[e]); dot[e] = fmaf(f[i][v4 + 3], gq.w, dot[e]);
                        }
                    }
                }
            }
        }
        float mylogit = reduce_dots_to_lane<EM>(dot, lane, E);
        float lc = 0.f;
        if (lane < E) {
            lc = quant == AB_ROUTER_EXACT ? fmaf(rstd, mylogit, cvec[lane]) : ab_round_to(mylogit + cvec[lane], quant);
            mylogit = lc;
            if (noise) mylogit = fmaf(noise[(size_t)s * E + lane], noise_scale[lane], lc);
            if (lclean) lclean[(size_t)s * E + lane] = lc;
            if (logits) logits[(size_t)s * E + lane] = mylogit;
        }
        if (lane == 0) { stats[2 * (size_t)s] = mean; stats[2 * (size_t)s + 1] = rstd; }
        float g, lse, my_p, den;
        int my_idx;
        unsigned sel_mask;
        select_topk(mylogit, lane, E, K, g, lse, my_idx, my_p, den, sel_mask);
        write_selection(s, lane, E, K, g, lse, my_idx, my_p, den, gates, idx, probs, w, lse_out);
        if (lane < E) {
            a_g += g;
            a_cnt += (sel_mask >> lane) & 1u ? 1.f : 0.f;
        }
        if (lane == 0) a_l2 = fmaf(lse, lse, a_l2);
    }
    const int NA = 2 * E + 1;
    if (lane < E) { red[warp * NA + lane] = a_g; red[warp * NA + E + lane] = a_cnt; }
    if (lane == 0) red[warp * NA + 2 * E] = a_l2;
    __syncthreads();
    if (tid < NA) {
        float s2 = 0.f;
        for (int wv = 0; wv < WARPS; ++wv) s2 += red[wv * NA + tid];
        part[(size_t)blockIdx.x * NA + tid] = s2;
    }
}

// out[c] = sum_r part[r][c]; one warp per column, fixed order -> deterministic
__global__ void reduce_rows_kernel(const float* __restrict__ part, int nrows, int ncols, float* __restrict__ out) {
    const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (c >= ncols) return;
    float s = 0.f;
    for (int r = lane; r < nrows; r += 32) s += part[(size_t)r * ncols + c];
    s = ab_warp_sum(s);
    if (lane == 0) out[c] = s;
}

__global__ void __launch_bounds__(WARPS * 32) topk_from_logits_kernel(const float* __restrict__ logits, float* __restrict__ gates,
                                                                      int32_t* __restrict__ idx, float* __restrict__ probs,
                                                                      float* __restrict__ w, float* __restrict__ lse_out, int S,
                                                                      int E, int K) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int s = blockIdx.x * WARPS + warp; s < S; s += gridDim.x * WARPS) {
        const float l = lane < E ? logits[(size_t)s * E + lane] : 0.f;
        float g, lse, my_p, den;
        int my_idx;
        unsigned sel_mask;
        select_topk(l, lane, E, K, g, lse, my_idx, my_p, den, sel_mask);
        write_selection(s, lane, E, K, g, lse, my_idx, my_p, den, gates, idx, probs, w, lse_out);
    }
}

// ---------------------------------------------------------------------------------------------
// backward: per token d logits and dx
// part layout per CTA: [2E] = sum dlogit[e] (-> dbr), sum dlogit[e]*noise[s,e] (-> dnoise_scale)
// ---------------------------------------------------------------------------------------------
// The per-token scalars of the backward (warp per token): lane e < E gets d logit e, lane k < K the row of slot k (-1 if
// dropped); every lane gets mean, rstd and the LayerNorm constants m1 = mean_d(dxhat), m2 = mean_d(dxhat * xhat).
// a_db / a_dn accumulate the lane's d logit and d logit * noise.
__device__ __forceinline__ void router_token_grad(int s, int lane, int E, int K, int Dm, const float* GS, const float* cvec,
                                                  const float* __restrict__ stats, const float* __restrict__ gates,
                                                  const int32_t* __restrict__ idx, const float* __restrict__ probs,
                                                  const float* __restrict__ lse, const float* __restrict__ lclean,
                                                  const float* __restrict__ noise, const float* __restrict__ f, float g_lb,
                                                  float g_rz, const float* __restrict__ dw_row, const int32_t* __restrict__ row_of,
                                                  int& my_r, float& dl, float& mean, float& rstd, float& m1, float& m2,
                                                  float& a_db, float& a_dn) {
    // loads that do not depend on the slot rows first: one memory latency for all of them
    const float g_in = lane < E ? gates[(size_t)s * E + lane] : 0.f;
    const float lse_s = lse[s];
    const float lc_in = lane < E ? lclean[(size_t)s * E + lane] : 0.f;
    const float nz_in = noise != nullptr && lane < E ? noise[(size_t)s * E + lane] : 0.f;
    const float f_in = lane < E ? f[lane] : 0.f;
    mean = stats[2 * (size_t)s]; rstd = stats[2 * (size_t)s + 1];
    // ---- d weights -> d probs (lane k < K holds slot k)
    int my_i = 0;
    float my_dw = 0.f, my_pk = 0.f;
    my_r = -1;
    if (lane < K) {
        my_r = row_of[(size_t)s * K + lane];
        my_i = idx[(size_t)s * K + lane];
        my_pk = probs[(size_t)s * K + lane];
        my_dw = my_r >= 0 ? dw_row[my_r] : 0.f;
    }
    float den = 0.f;
    for (int k = 0; k < K; ++k) den += __shfl_sync(0xffffffffu, my_pk, k);    // slot order, as in the forward
    den += 1e-6f;
    const float dot = ab_warp_sum(my_dw * my_pk);
    const float inv = 1.f / den;
    const float my_dp = my_dw * inv - dot * inv * inv;       // d prob of slot `lane`
    float dgate = 0.f, g = 0.f;
    for (int k = 0; k < K; ++k) {
        const int ik = __shfl_sync(0xffffffffu, my_i, k);
        const float dpk = __shfl_sync(0xffffffffu, my_dp, k);
        if (lane == ik) dgate += dpk;
    }
    if (lane < E) {
        g = g_in;
        dgate = fmaf(g_lb, f_in, dgate);
    } else {
        dgate = 0.f;
    }
    const float gd = ab_warp_sum(g * dgate);
    dl = 0.f;
    if (lane < E) {
        dl = g * (dgate - gd) + g_rz * 2.f * lse_s * g;
        a_db += dl;
        if (noise) a_dn = fmaf(dl, nz_in, a_dn);
    }
    // ---- LayerNorm backward constants
    float t1 = 0.f, t2 = 0.f;
    if (lane < E) {
        t1 = dl * GS[lane];
        t2 = dl * (lc_in - cvec[lane]);    // sum_d G[e,d]*xhat[d]
    }
    m1 = ab_warp_sum(t1) / (float)Dm;
    m2 = ab_warp_sum(t2) / (float)Dm;
}

// Row kernel (warp per token) for the shapes the one-pass kernels below do not take; router_q_kernel then forms Q.
template <typename T, int EM>
__global__ void __launch_bounds__(WARPS * 32) router_bwd_kernel(const T* __restrict__ x, const float* __restrict__ stats,
                                                                const float* __restrict__ ln_w, const float* __restrict__ ln_b,
                                                                const float* __restrict__ Wr, const float* __restrict__ br,
                                                                const float* __restrict__ gates, const int32_t* __restrict__ idx,
                                                                const float* __restrict__ probs, const float* __restrict__ lse,
                                                                const float* __restrict__ lclean, const float* __restrict__ noise,
                                                                const float* __restrict__ f, const float* __restrict__ scal,
                                                                const float* __restrict__ dw_row, const float* __restrict__ dxrow,
                                                                const int32_t* __restrict__ row_of, T* __restrict__ dx,
                                                                float* __restrict__ dlogits, float* __restrict__ part, int S,
                                                                int Dm, int E, int K) {
    constexpr int V = ab_vec16<T>::N;
    extern __shared__ float sm[];
    float* Wsm = sm;                         // [E][Dm] raw router weight
    float* gam = Wsm + (size_t)E * Dm;       // [Dm]
    float* GS = gam + Dm;                    // [32]  sum_d ln_w[d]*Wr[e,d]
    float* cvec = GS + 32;                   // [32]
    float* red = cvec + 32;                  // [WARPS][2E]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < E * Dm; i += blockDim.x) Wsm[i] = Wr[i];
    for (int i = tid; i < Dm; i += blockDim.x) gam[i] = ln_w[i];
    for (int e = warp; e < E; e += WARPS) {
        float a1 = 0.f, a2 = 0.f;
        for (int d = lane; d < Dm; d += 32) {
            a1 = fmaf(ln_w[d], Wr[(size_t)e * Dm + d], a1);
            a2 = fmaf(ln_b[d], Wr[(size_t)e * Dm + d], a2);
        }
        a1 = ab_warp_sum(a1); a2 = ab_warp_sum(a2);
        if (lane == 0) { GS[e] = a1; cvec[e] = a2 + br[e]; }
    }
    __syncthreads();
    const float g_lb = scal[0], g_rz = scal[1];
    const int nvec = Dm / V;
    float a_db = 0.f, a_dn = 0.f;
    for (int s = blockIdx.x * WARPS + warp; s < S; s += gridDim.x * WARPS) {
        int my_r;
        float dl, mean, rstd, m1, m2;
        router_token_grad(s, lane, E, K, Dm, GS, cvec, stats, gates, idx, probs, lse, lclean, noise, f, g_lb, g_rz, dw_row, row_of,
                          my_r, dl, mean, rstd, m1, m2, a_db, a_dn);
        if (lane < E) dlogits[(size_t)s * E + lane] = dl;
        float dle[EM];
#pragma unroll
        for (int e = 0; e < EM; ++e) dle[e] = __shfl_sync(0xffffffffu, dl, e);
        int rk[MAX_K];                                   // rows of the K slots, broadcast once (the vector loop below diverges)
#pragma unroll
        for (int k = 0; k < MAX_K; ++k) { const int r = __shfl_sync(0xffffffffu, my_r, k); rk[k] = k < K ? r : -1; }
        const T* row = x + (size_t)s * Dm;
        T* orow = dx + (size_t)s * Dm;
        for (int i = lane; i < nvec; i += 32) {
            float fx[V], o[V];
            row_load<T>(row, i, fx);
            float dxn[V];
#pragma unroll
            for (int v = 0; v < V; ++v) dxn[v] = 0.f;
#pragma unroll
            for (int e = 0; e < EM; ++e) {
                if (e < E) {
#pragma unroll
                    for (int v4 = 0; v4 < V; v4 += 4) {
                        const float4 wq = *reinterpret_cast<const float4*>(Wsm + (size_t)e * Dm + i * V + v4);
                        dxn[v4] = fmaf(dle[e], wq.x, dxn[v4]); dxn[v4 + 1] = fmaf(dle[e], wq.y, dxn[v4 + 1]);
                        dxn[v4 + 2] = fmaf(dle[e], wq.z, dxn[v4 + 2]); dxn[v4 + 3] = fmaf(dle[e], wq.w, dxn[v4 + 3]);
                    }
                }
            }
#pragma unroll
            for (int v4 = 0; v4 < V; v4 += 4) {
                const float4 gq = *reinterpret_cast<const float4*>(gam + i * V + v4);
                const float gg[4] = {gq.x, gq.y, gq.z, gq.w};
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const float xh = (fx[v4 + u] - mean) * rstd;
                    o[v4 + u] = rstd * (dxn[v4 + u] * gg[u] - m1 - xh * m2);
                }
            }
#pragma unroll
            for (int k = 0; k < MAX_K; ++k) {
                const int rkk = rk[k];
                if (rkk >= 0) {
                    const float* er = dxrow + (size_t)rkk * Dm + i * V;
#pragma unroll
                    for (int v4 = 0; v4 < V; v4 += 4) {
                        const float4 q = __ldg(reinterpret_cast<const float4*>(er + v4));
                        o[v4] += q.x; o[v4 + 1] += q.y; o[v4 + 2] += q.z; o[v4 + 3] += q.w;
                    }
                }
            }
            *(reinterpret_cast<uint4*>(orow) + i) = ab_vec16<T>::pack(o);
        }
    }
    const int NA = 2 * E;
    if (lane < E) { red[warp * NA + lane] = a_db; red[warp * NA + E + lane] = a_dn; }
    __syncthreads();
    if (tid < NA) {
        float s2 = 0.f;
        for (int wv = 0; wv < WARPS; ++wv) s2 += red[wv * NA + tid];
        part[(size_t)blockIdx.x * NA + tid] = s2;
    }
}

// kernel C: Q[e,d] = sum_s dlogits[s,e] * xhat[s,d]; thread per column d, token blocks of QB tokens
constexpr int qb_for(int em) { return 2048 / em; }     // tokens per partial block (smem [QB][EM] floats)
int em_for(int E) { return E <= 8 ? 8 : (E <= 16 ? 16 : 32); }
template <typename T, int EM>
__global__ void __launch_bounds__(256) router_q_kernel(const T* __restrict__ x, const float* __restrict__ stats,
                                                       const float* __restrict__ dlogits, float* __restrict__ qpart, int S,
                                                       int Dm, int E) {
    constexpr int QB = qb_for(EM);
    __shared__ float sdl[QB * EM];
    __shared__ float sst[QB * 2];
    const int s0 = blockIdx.y * QB;
    const int ns = min(QB, S - s0);
    for (int i = threadIdx.x; i < ns * E; i += blockDim.x) sdl[i] = dlogits[(size_t)s0 * E + i];
    for (int i = threadIdx.x; i < ns * 2; i += blockDim.x) sst[i] = stats[(size_t)s0 * 2 + i];
    __syncthreads();
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= Dm) return;
    float acc[EM];
#pragma unroll
    for (int e = 0; e < EM; ++e) acc[e] = 0.f;
    // 8 rows in flight per thread: the loop is a stream of independent, coalesced loads, not a dependent chain
    for (int j0 = 0; j0 < ns; j0 += 8) {
        float xv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) xv[u] = j0 + u < ns ? ab_to_float(x[(size_t)(s0 + j0 + u) * Dm + d]) : 0.f;
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int j = j0 + u;
            if (j < ns) {
                const float xh = (xv[u] - sst[2 * j]) * sst[2 * j + 1];
#pragma unroll
                for (int e = 0; e < EM; ++e)
                    if (e < E) acc[e] = fmaf(sdl[j * E + e], xh, acc[e]);
            }
        }
    }
#pragma unroll
    for (int e = 0; e < EM; ++e)
        if (e < E) qpart[((size_t)blockIdx.y * E + e) * Dm + d] = acc[e];
}

// Backward for E <= 8 and hidden sizes up to 1024 in one pass over x, split in two kernels so that neither waits on the
// other's latency chain.  router_bwd_tok_kernel (warp per token, the whole grid): the per-token scalars of
// router_token_grad -> tsc[s] = {d logits [8], mean, rstd, m1, m2}, and the per-CTA sums for dbr / dnoise_scale.
constexpr int TSC = 12;                      // floats per token in tsc
constexpr int TOK_CTAS_PER_SM = 6;           // 48 warps per SM on the token kernel's latency-bound chains
constexpr int FUSED_EM = 8;
__global__ void __launch_bounds__(WARPS * 32, TOK_CTAS_PER_SM) router_bwd_tok_kernel(const float* __restrict__ stats, const float* __restrict__ ln_w,
                                                                    const float* __restrict__ ln_b, const float* __restrict__ Wr,
                                                                    const float* __restrict__ br, const float* __restrict__ gates,
                                                                    const int32_t* __restrict__ idx, const float* __restrict__ probs,
                                                                    const float* __restrict__ lse, const float* __restrict__ lclean,
                                                                    const float* __restrict__ noise, const float* __restrict__ f,
                                                                    const float* __restrict__ scal, const float* __restrict__ dw_row,
                                                                    const int32_t* __restrict__ row_of, float* __restrict__ tsc,
                                                                    float* __restrict__ part, int S, int Dm, int E, int K) {
    __shared__ float GS[32], cvec[32], red[WARPS][2 * FUSED_EM];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int e = warp; e < E; e += WARPS) {
        float a1 = 0.f, a2 = 0.f;
        for (int d = lane; d < Dm; d += 32) {
            a1 = fmaf(ln_w[d], Wr[(size_t)e * Dm + d], a1);
            a2 = fmaf(ln_b[d], Wr[(size_t)e * Dm + d], a2);
        }
        a1 = ab_warp_sum(a1); a2 = ab_warp_sum(a2);
        if (lane == 0) { GS[e] = a1; cvec[e] = a2 + br[e]; }
    }
    __syncthreads();
    const float g_lb = scal[0], g_rz = scal[1];
    float a_db = 0.f, a_dn = 0.f;
    for (int s = blockIdx.x * WARPS + warp; s < S; s += gridDim.x * WARPS) {
        int my_r;
        float dl, mean, rstd, m1, m2;
        router_token_grad(s, lane, E, K, Dm, GS, cvec, stats, gates, idx, probs, lse, lclean, noise, f, g_lb, g_rz, dw_row, row_of,
                          my_r, dl, mean, rstd, m1, m2, a_db, a_dn);
        float v = dl;                                // lanes < 8: d logit (0 for lanes >= E)
        if (lane == 8) v = mean;
        if (lane == 9) v = rstd;
        if (lane == 10) v = m1;
        if (lane == 11) v = m2;
        if (lane < TSC) tsc[(size_t)s * TSC + lane] = v;
    }
    const int NA = 2 * E;
    if (lane < E) { red[warp][lane] = a_db; red[warp][E + lane] = a_dn; }
    __syncthreads();
    if (tid < NA) {
        float s2 = 0.f;
        for (int wv = 0; wv < WARPS; ++wv) s2 += red[wv][tid];
        part[(size_t)blockIdx.x * NA + tid] = s2;
    }
}

// router_bwd_col_kernel: a persistent CTA takes tiles of BT tokens; thread c owns the columns [4c, 4c+4) of every row of
// the tile, forms dx there and accumulates Q[e,d] = sum_s dlogits[s,e] * xhat[s,d] in registers over all its tiles.  The
// CTA's Q partial is written once at the end; router_param_kernel adds the partials in CTA order.  dx is computed with
// the same operations in the same order as in router_bwd_kernel.  The next tile's scalars and slot rows are copied to
// shared memory asynchronously while the current tile streams.
constexpr int BT = 32;
constexpr int FUSED_MAX_THREADS = 256;
constexpr int FUSED_MAX_REGS = 144;          // no spills; two CTAs of 192 threads (hidden 704) per SM
template <typename T, int KM>
__global__ void __maxnreg__(FUSED_MAX_REGS) router_bwd_col_kernel(const T* __restrict__ x, const float* __restrict__ ln_w,
                                                                  const float* __restrict__ Wr, const float* __restrict__ tsc,
                                                                  const float* __restrict__ dxrow, const int32_t* __restrict__ row_of,
                                                                  T* __restrict__ dx, float* __restrict__ qpart, int S, int Dm,
                                                                  int E, int K) {
    constexpr int EM = FUSED_EM;
    constexpr int U = KM <= 2 ? 4 : 1;       // tokens whose loads are issued together
    constexpr int NSC = BT * TSC, NROW = BT * KM;
    extern __shared__ float sm[];
    float* Wsm = sm;                         // [E][Dm] raw router weight
    float* stile = Wsm + (size_t)E * Dm;     // [2][BT][TSC] scalars of the tile (double buffer)
    int* srow = reinterpret_cast<int*>(stile + 2 * NSC);    // [2][BT][KM] rows of the slots, -1 if dropped
    const int tid = threadIdx.x;
    for (int i = tid; i < E * Dm; i += blockDim.x) Wsm[i] = Wr[i];
    const int d = 4 * tid;
    const bool has_col = d < Dm;
    float gg[4] = {0.f, 0.f, 0.f, 0.f};
    if (has_col) {
        const float4 gq = __ldg(reinterpret_cast<const float4*>(ln_w + d));
        gg[0] = gq.x; gg[1] = gq.y; gg[2] = gq.z; gg[3] = gq.w;
    }
    // one tile's scalars and rows into buffer `buf` by asynchronous copies (no registers held while they are in flight);
    // complete after cp.async.wait_all
    auto fetch = [&](int s0, int buf) {
        const int nt = s0 < S ? min(BT, S - s0) : 0;
        for (int i = tid; i < nt * TSC; i += blockDim.x) {
            const unsigned dst = (unsigned)__cvta_generic_to_shared(stile + buf * NSC + i);
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(tsc + (size_t)s0 * TSC + i));
        }
        for (int i = tid; i < nt * KM; i += blockDim.x) {
            const int j = i / KM, k = i % KM;
            if (k < K) {
                const unsigned dst = (unsigned)__cvta_generic_to_shared(srow + buf * NROW + i);
                asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(row_of + (size_t)(s0 + j) * K + k));
            } else {
                srow[buf * NROW + i] = -1;
            }
        }
    };
    float q[EM][4];
#pragma unroll
    for (int e = 0; e < EM; ++e) { q[e][0] = q[e][1] = q[e][2] = q[e][3] = 0.f; }
    const int step = gridDim.x * BT;
    fetch(blockIdx.x * BT, 0);
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();
    int buf = 0;
    for (int s0 = blockIdx.x * BT; s0 < S; s0 += step, buf ^= 1) {
        const int nt = min(BT, S - s0);
        fetch(s0 + step, buf ^ 1);
        const float* sc = stile + buf * NSC;
        const int* rw = srow + buf * NROW;
        if (has_col) {
            for (int j0 = 0; j0 < nt; j0 += U) {
                // the next batch's x and dxrow lines into L2 (no registers held): its loads then wait on L2, not HBM
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int j = j0 + U + u;
                    if (j < nt && (tid & 7) == 0) {          // one thread per 128-byte line of fp32 rows
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(x + (size_t)(s0 + j) * Dm + d));
#pragma unroll
                        for (int k = 0; k < KM; ++k) {
                            const int r = rw[j * KM + k];
                            if (r >= 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(dxrow + (size_t)r * Dm + d));
                        }
                    }
                }
                float xv[U][4], er[U][KM][4];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int j = j0 + u;
#pragma unroll
                    for (int k = 0; k < KM; ++k) er[u][k][0] = er[u][k][1] = er[u][k][2] = er[u][k][3] = 0.f;
                    xv[u][0] = xv[u][1] = xv[u][2] = xv[u][3] = 0.f;
                    if (j < nt) {
                        ld4g<T>(x + (size_t)(s0 + j) * Dm + d, xv[u]);
#pragma unroll
                        for (int k = 0; k < KM; ++k) {
                            const int r = rw[j * KM + k];
                            if (r >= 0) ld4g<float>(dxrow + (size_t)r * Dm + d, er[u][k]);
                        }
                    }
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int j = j0 + u;
                    if (j >= nt) break;
                    const float* t = sc + j * TSC;
                    const float mean = t[8], rstd = t[9], m1 = t[10], m2 = t[11];
                    float dle[EM];
#pragma unroll
                    for (int e = 0; e < EM; ++e) dle[e] = t[e];
                    float dxn[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                    for (int e = 0; e < EM; ++e) {
                        if (e < E) {
                            const float4 wq = *reinterpret_cast<const float4*>(Wsm + (size_t)e * Dm + d);
                            dxn[0] = fmaf(dle[e], wq.x, dxn[0]); dxn[1] = fmaf(dle[e], wq.y, dxn[1]);
                            dxn[2] = fmaf(dle[e], wq.z, dxn[2]); dxn[3] = fmaf(dle[e], wq.w, dxn[3]);
                        }
                    }
                    float o[4], xh[4];
#pragma unroll
                    for (int v = 0; v < 4; ++v) {
                        xh[v] = (xv[u][v] - mean) * rstd;
                        o[v] = rstd * (dxn[v] * gg[v] - m1 - xh[v] * m2);
                    }
#pragma unroll
                    for (int k = 0; k < KM; ++k) {
                        if (rw[j * KM + k] >= 0) {
#pragma unroll
                            for (int v = 0; v < 4; ++v) o[v] += er[u][k][v];
                        }
                    }
                    ab_st4<T>(dx + (size_t)(s0 + j) * Dm + d, o);
#pragma unroll
                    for (int e = 0; e < EM; ++e) {
#pragma unroll
                        for (int v = 0; v < 4; ++v) q[e][v] = fmaf(dle[e], xh[v], q[e][v]);
                    }
                }
            }
        }
        asm volatile("cp.async.wait_all;" ::: "memory");
        __syncthreads();
    }
    if (has_col) {
#pragma unroll
        for (int e = 0; e < EM; ++e)
            if (e < E) *reinterpret_cast<float4*>(qpart + ((size_t)blockIdx.x * E + e) * Dm + d) = make_float4(q[e][0], q[e][1], q[e][2], q[e][3]);
    }
}

// kernel D: reduce Q partials and derive all router parameter grads.  block = (32 columns, E experts, G row groups)
//   dbr[e] = sum dlogits;  dWr[e,d] = ln_w[d]*Q[e,d] + ln_b[d]*dbr[e]
//   dln_w[d] = sum_e Wr[e,d]*Q[e,d];  dln_b[d] = sum_e Wr[e,d]*dbr[e]
// Group g adds the partial rows g, g+G, ... in order, then the G group sums are added in group order (fixed order ->
// deterministic); the groups put G times as many loads in flight.
int param_groups(int E) { const int g = 1024 / (32 * E); return g < 1 ? 1 : (g > 4 ? 4 : g); }
__global__ void router_param_kernel(const float* __restrict__ qpart, int nqb, const float* __restrict__ part, int nparts,
                                    const float* __restrict__ ln_w, const float* __restrict__ ln_b, const float* __restrict__ Wr,
                                    float* __restrict__ dWr, float* __restrict__ dbr, float* __restrict__ dln_w,
                                    float* __restrict__ dln_b, float* __restrict__ dnoise_scale, int Dm, int E) {
    __shared__ float sdb[64];
    __shared__ float sgw[32][33], sgb[32][33];
    __shared__ float spart[16][64];
    __shared__ float sq[32][33];             // [group * E + e][column]
    const int tx = threadIdx.x, e = threadIdx.y, grp = threadIdx.z, G = blockDim.z;
    const int tid = (grp * E + e) * 32 + tx;
    const int nthr = 32 * E * G;
    // column sums of the per-CTA partials: up to 16 thread groups add interleaved rows, then one thread per column adds
    // the groups in index order (fixed order -> deterministic)
    {
        const int ncol = 2 * E;
        const int ngrp = min(16, nthr / ncol);
        const int col = tid % ncol, pg = tid / ncol;
        if (pg < ngrp) {
            float s = 0.f;
            for (int r0 = pg; r0 < nparts; r0 += ngrp * 4) {
                float v[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) v[u] = r0 + u * ngrp < nparts ? part[(size_t)(r0 + u * ngrp) * ncol + col] : 0.f;
#pragma unroll
                for (int u = 0; u < 4; ++u) s += v[u];
            }
            spart[pg][col] = s;
        }
        __syncthreads();
        if (tid < ncol) {
            float s = 0.f;
            for (int g2 = 0; g2 < ngrp; ++g2) s += spart[g2][tid];
            sdb[tid] = s;
            if (blockIdx.x == 0) {
                if (tid < E) dbr[tid] = s;
                else if (dnoise_scale) dnoise_scale[tid - E] = s;
            }
        }
    }
    const int d = blockIdx.x * 32 + tx;
    {
        float q = 0.f;
        if (d < Dm) {
            for (int r0 = grp; r0 < nqb; r0 += 8 * G) {
                float qv[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) qv[u] = r0 + u * G < nqb ? qpart[((size_t)(r0 + u * G) * E + e) * Dm + d] : 0.f;
#pragma unroll
                for (int u = 0; u < 8; ++u) q += qv[u];
            }
        }
        sq[grp * E + e][tx] = q;
    }
    __syncthreads();
    if (grp == 0) {
        float gw = 0.f, gb = 0.f;
        if (d < Dm) {
            float q = 0.f;
            for (int g2 = 0; g2 < G; ++g2) q += sq[g2 * E + e][tx];
            const float wv = Wr[(size_t)e * Dm + d];
            dWr[(size_t)e * Dm + d] = fmaf(ln_w[d], q, ln_b[d] * sdb[e]);
            gw = wv * q;
            gb = wv * sdb[e];
        }
        sgw[e][tx] = gw;
        sgb[e][tx] = gb;
    }
    __syncthreads();
    if (grp == 0 && e == 0 && d < Dm) {
        float a = 0.f, b = 0.f;
        for (int i = 0; i < E; ++i) { a += sgw[i][tx]; b += sgb[i][tx]; }
        dln_w[d] = a;
        dln_b[d] = b;
    }
}

int router_grid(int S) {
    const int want = (int)ab_ceil_div(S, WARPS);
    const int cap = ab_num_sms() * 4;
    return want < cap ? want : cap;
}

struct FwdWs { size_t part_off, total; int grid; };
FwdWs fwd_ws(int S, int E) {
    FwdWs w;
    w.grid = router_grid(S);
    w.part_off = 0;
    w.total = ab_round_up((int64_t)w.grid * (2 * E + 1) * sizeof(float), 256);
    return w;
}
// the one-pass backward takes E <= 8 and hidden sizes up to 4 * FUSED_MAX_THREADS; its column kernel runs at most
// MAX_FUSED_PER_SM CTAs per SM
constexpr int MAX_FUSED_PER_SM = 4;
// the token kernel in one wave of TOK_CTAS_PER_SM CTAs per SM
int tok_grid(int S) {
    const int want = (int)ab_ceil_div(S, WARPS);
    const int cap = ab_num_sms() * TOK_CTAS_PER_SM;
    return want < cap ? want : cap;
}
bool bwd_fused(int Dm, int E) { return E <= FUSED_EM && Dm % 4 == 0 && Dm / 4 <= FUSED_MAX_THREADS; }
struct BwdWs { size_t part_off, dl_off, q_off, total; int nqb; };
BwdWs bwd_ws(int S, int Dm, int E) {
    BwdWs w;
    const bool fused = bwd_fused(Dm, E);
    w.nqb = fused ? ab_num_sms() * MAX_FUSED_PER_SM : (int)ab_ceil_div(S, qb_for(em_for(E)));
    size_t o = 0;
    w.part_off = o; o += ab_round_up((int64_t)(fused ? tok_grid(S) : router_grid(S)) * 2 * E * sizeof(float), 256);
    w.dl_off = o; o += ab_round_up((int64_t)S * (fused ? TSC : E) * sizeof(float), 256);     // tsc, or the d logits
    w.q_off = o; o += ab_round_up((int64_t)w.nqb * E * Dm * sizeof(float), 256);
    w.total = o;
    return w;
}

int check_router(int S, int Dm, int E, int K, int dtype) {
    AB_REQUIRE(S > 0 && Dm > 0, "moe_router: empty shape S=%d Dm=%d", S, Dm);
    AB_REQUIRE(E >= 1 && E <= 32, "moe_router: num_experts must be in [1,32] (got %d)", E);
    AB_REQUIRE(K >= 1 && K <= MAX_K && K <= E, "moe_router: experts_per_token must be in [1,%d] and <= E (got %d)", MAX_K, K);
    AB_REQUIRE(dtype == AB_F32 || dtype == AB_BF16, "moe_router: bad dtype %d", dtype);
    const int V = dtype == AB_F32 ? 4 : 8;
    AB_REQUIRE(Dm % V == 0, "moe_router: hidden size %d must be a multiple of %d", Dm, V);
    return AB_OK;
}

}  // namespace

extern "C" size_t ab_moe_router_workspace_bytes(int S, int Dm, int E) { (void)Dm; return fwd_ws(S, E).total; }

extern "C" int ab_moe_router_fwd(const void* x, const float* ln_w, const float* ln_b, float eps, const float* Wr,
                                 const float* br, const float* noise, const float* noise_scale, float* lclean, float* logits,
                                 float* gates, int32_t* idx, float* probs, float* w, float* lse, float* stats_out, float* aux,
                                 void* ws, size_t ws_bytes, int S, int Dm, int E, int K, int dtype, int quant, cudaStream_t stream) {
    if (int e = check_router(S, Dm, E, K, dtype)) return e;
    const FwdWs wl = fwd_ws(S, E);
    AB_REQUIRE(ws && ws_bytes >= wl.total, "moe_router_fwd: workspace too small");
    AB_REQUIRE(noise == nullptr || noise_scale != nullptr, "moe_router_fwd: noise without noise_scale");
    AB_REQUIRE(quant == AB_ROUTER_EXACT || quant == AB_ROUTER_BF16 || quant == AB_ROUTER_FP16, "moe_router_fwd: bad logit rounding mode %d", quant);
    // modules.py::router_smem_bytes mirrors this size: AdaptiveExpertSystem refuses, at construction, hidden sizes
    // whose router forward would not fit in a block's shared memory.  Change the two together.
    const size_t smem = ((size_t)E * Dm + 32 + WARPS * (2 * E + 1) + 2 * (size_t)Dm) * sizeof(float);
    float* part = (float*)ws;
    const int V = dtype == AB_F32 ? 4 : 8;
    const int nv = (int)ab_ceil_div(Dm, 32 * V);          // 16-byte vectors of the row per lane
    int grid = wl.grid;
#define AB_ROUTER_LAUNCH(KERNEL)                                                                                        \
    {                                                                                                                    \
        auto k = KERNEL;                                                                                                 \
        AB_CHECK_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                 \
        int occ = 4;                                                                                                     \
        if (FWD_PERSIST) AB_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k, WARPS * 32, smem));       \
        occ = occ < 1 ? 1 : (occ > 4 ? 4 : occ);                                                                        \
        grid = wl.grid < ab_num_sms() * occ ? wl.grid : ab_num_sms() * occ;                                              \
        k<<<grid, WARPS * 32, smem, stream>>>((const TT*)x, ln_w, ln_b, eps, Wr, br, noise, noise_scale, lclean,         \
                                              logits, gates, idx, probs, w, lse, stats_out, part, S, Dm, E, K, quant);    \
    }
    // the row-in-registers kernel whenever the row fits (hidden size <= 2048 fp32 / 4096 bf16), the streaming one otherwise
#define AB_ROUTER_FWD(TT_, EMV)                                                                                         \
    {                                                                                                                    \
        using TT = TT_;                                                                                                  \
        if (nv <= 4) AB_ROUTER_LAUNCH((router_fwd_reg_kernel<TT, EMV, 4>))                                               \
        else if (nv <= 6) AB_ROUTER_LAUNCH((router_fwd_reg_kernel<TT, EMV, 6>))                                          \
        else if (nv <= 8) AB_ROUTER_LAUNCH((router_fwd_reg_kernel<TT, EMV, 8>))                                          \
        else if (nv <= 16 && EMV <= 8) AB_ROUTER_LAUNCH((router_fwd_reg_kernel<TT, EMV, 16>))                            \
        else AB_ROUTER_LAUNCH((router_fwd_kernel<TT, EMV>))                                                              \
    }
    if (dtype == AB_F32) {
        if (E <= 8) AB_ROUTER_FWD(float, 8) else if (E <= 16) AB_ROUTER_FWD(float, 16) else AB_ROUTER_FWD(float, 32)
    } else {
        if (E <= 8) AB_ROUTER_FWD(__nv_bfloat16, 8) else if (E <= 16) AB_ROUTER_FWD(__nv_bfloat16, 16) else AB_ROUTER_FWD(__nv_bfloat16, 32)
    }
#undef AB_ROUTER_LAUNCH
#undef AB_ROUTER_FWD
    AB_LAUNCH_CHECK();
    reduce_rows_kernel<<<(unsigned)ab_ceil_div(2 * E + 1, 4), 128, 0, stream>>>(part, grid, 2 * E + 1, aux);
    AB_LAUNCH_CHECK();
    return AB_OK;
}

extern "C" int ab_moe_topk_from_logits(const float* logits, float* gates, int32_t* idx, float* probs, float* w, float* lse,
                                       int S, int E, int K, cudaStream_t stream) {
    if (int e = check_router(S, 8, E, K, AB_F32)) return e;
    topk_from_logits_kernel<<<router_grid(S), WARPS * 32, 0, stream>>>(logits, gates, idx, probs, w, lse, S, E, K);
    AB_LAUNCH_CHECK();
    return AB_OK;
}

extern "C" size_t ab_moe_router_bwd_workspace_bytes(int S, int Dm, int E) { return bwd_ws(S, Dm, E).total; }

extern "C" int ab_moe_router_bwd(const void* x, const float* stats, const float* ln_w, const float* ln_b, const float* Wr,
                                 const float* br, const float* gates, const int32_t* idx, const float* probs, const float* lse,
                                 const float* lclean, const float* noise, const float* f, const float* scal,
                                 const float* dw_row, const float* dxrow, const int32_t* row_of, void* dx, float* dWr,
                                 float* dbr, float* dln_w, float* dln_b, float* dnoise_scale, void* ws, size_t ws_bytes, int S,
                                 int Dm, int E, int K, int dtype, cudaStream_t stream) {
    if (int e = check_router(S, Dm, E, K, dtype)) return e;
    AB_REQUIRE(Dm % 4 == 0, "moe_router_bwd: hidden size must be a multiple of 4");
    const BwdWs wl = bwd_ws(S, Dm, E);
    AB_REQUIRE(ws && ws_bytes >= wl.total, "moe_router_bwd: workspace too small");
    unsigned char* w8 = (unsigned char*)ws;
    float* part = (float*)(w8 + wl.part_off);
    float* dl = (float*)(w8 + wl.dl_off);
    float* qpart = (float*)(w8 + wl.q_off);
    int nqb = wl.nqb, nparts = router_grid(S);
    if (bwd_fused(Dm, E)) {
        nparts = tok_grid(S);
        router_bwd_tok_kernel<<<nparts, WARPS * 32, 0, stream>>>(stats, ln_w, ln_b, Wr, br, gates, idx, probs, lse, lclean, noise, f,
                                                                 scal, dw_row, row_of, dl, part, S, Dm, E, K);
        AB_LAUNCH_CHECK();
        const int threads = (int)ab_round_up(Dm / 4 > 64 ? Dm / 4 : 64, 32);
        const size_t smem = ((size_t)E * Dm + 2 * BT * TSC + 2 * BT * MAX_K) * sizeof(float);
#define AB_ROUTER_BWD_COL(TT, KMV)                                                                                      \
    {                                                                                                                    \
        auto k = router_bwd_col_kernel<TT, KMV>;                                                                         \
        AB_CHECK_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                 \
        int occ = 0;                                                                                                     \
        AB_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k, threads, smem));                           \
        occ = occ < 1 ? 1 : (occ > MAX_FUSED_PER_SM ? MAX_FUSED_PER_SM : occ);                                          \
        const int64_t want = ab_ceil_div(S, BT);                                                                         \
        nqb = (int)(want < (int64_t)ab_num_sms() * occ ? want : (int64_t)ab_num_sms() * occ);                            \
        k<<<nqb, threads, smem, stream>>>((const TT*)x, ln_w, Wr, dl, dxrow, row_of, (TT*)dx, qpart, S, Dm, E, K);        \
    }
        if (dtype == AB_F32) {
            if (K <= 2) AB_ROUTER_BWD_COL(float, 2) else AB_ROUTER_BWD_COL(float, MAX_K)
        } else {
            if (K <= 2) AB_ROUTER_BWD_COL(__nv_bfloat16, 2) else AB_ROUTER_BWD_COL(__nv_bfloat16, MAX_K)
        }
#undef AB_ROUTER_BWD_COL
        AB_LAUNCH_CHECK();
    } else {
        const size_t smem = ((size_t)E * Dm + Dm + 64 + WARPS * 2 * E) * sizeof(float);
        dim3 qgrid((unsigned)ab_ceil_div(Dm, 256), nqb);
#define AB_ROUTER_BWD(TT, EMV)                                                                                          \
    {                                                                                                                    \
        auto k = router_bwd_kernel<TT, EMV>;                                                                             \
        AB_CHECK_CUDA(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                 \
        k<<<nparts, WARPS * 32, smem, stream>>>((const TT*)x, stats, ln_w, ln_b, Wr, br, gates, idx, probs, lse,        \
                                                lclean, noise, f, scal, dw_row, dxrow, row_of, (TT*)dx, dl, part, S,    \
                                                Dm, E, K);                                                               \
        AB_LAUNCH_CHECK();                                                                                               \
        router_q_kernel<TT, EMV><<<qgrid, 256, 0, stream>>>((const TT*)x, stats, dl, qpart, S, Dm, E);                  \
    }
        if (dtype == AB_F32) {
            if (E <= 8) AB_ROUTER_BWD(float, 8) else if (E <= 16) AB_ROUTER_BWD(float, 16) else AB_ROUTER_BWD(float, 32)
        } else {
            if (E <= 8) AB_ROUTER_BWD(__nv_bfloat16, 8) else if (E <= 16) AB_ROUTER_BWD(__nv_bfloat16, 16) else AB_ROUTER_BWD(__nv_bfloat16, 32)
        }
#undef AB_ROUTER_BWD
        AB_LAUNCH_CHECK();
    }
    const int G = param_groups(E);
    router_param_kernel<<<(unsigned)ab_ceil_div(Dm, 32), dim3(32, E, G), 0, stream>>>(qpart, nqb, part, nparts, ln_w, ln_b, Wr, dWr,
                                                                                     dbr, dln_w, dln_b, dnoise_scale, Dm, E);
    AB_LAUNCH_CHECK();
    return AB_OK;
}
