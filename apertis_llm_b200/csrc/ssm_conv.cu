// Causal depthwise conv1d (k = Kc, 2 <= Kc <= 8) + SiLU, forward and recompute-based backward.
// Replaces core.py:368-375 (two transposes + nn.Conv1d(groups=Di, padding=3)[:, :, :L] + F.silu) and
// their autograd.  Layout is channels-last [B, L, Di]: a thread owns one 16-byte channel vector and
// walks TT consecutive tokens with a sliding window in registers, so every global access is a
// coalesced 128-bit load/store and each input row is fetched from HBM once (halo rows hit L1/L2).
#include "common.cuh"

namespace {

constexpr int KC_MAX = 8;
constexpr int TT = 16;       // tokens per thread
constexpr int ROWS_PER_CTA = 8;   // thread rows (token runs) per CTA

// V channels of T in one 16-byte word, or (bf16, V = 4) in one 8-byte word
template <typename T, int V> struct Chan;
template <> struct Chan<float, 4> {
    typedef uint4 raw;
    __device__ __forceinline__ static void unpack(const raw& r, float* f) { ab_vec16<float>::unpack(r, f); }
    __device__ __forceinline__ static raw pack(const float* f) { return ab_vec16<float>::pack(f); }
};
template <> struct Chan<__nv_bfloat16, 8> {
    typedef uint4 raw;
    __device__ __forceinline__ static void unpack(const raw& r, float* f) { ab_vec16<__nv_bfloat16>::unpack(r, f); }
    __device__ __forceinline__ static raw pack(const float* f) { return ab_vec16<__nv_bfloat16>::pack(f); }
};
template <> struct Chan<__nv_bfloat16, 4> {
    typedef uint2 raw;
    __device__ __forceinline__ static void unpack(const raw& r, float* f) {
        f[0] = __uint_as_float(r.x << 16); f[1] = __uint_as_float(r.x & 0xffff0000u);
        f[2] = __uint_as_float(r.y << 16); f[3] = __uint_as_float(r.y & 0xffff0000u);
    }
    __device__ __forceinline__ static raw pack(const float* f) {
        __nv_bfloat162 a = __floats2bfloat162_rn(f[0], f[1]), b = __floats2bfloat162_rn(f[2], f[3]);
        return make_uint2(*reinterpret_cast<uint32_t*>(&a), *reinterpret_cast<uint32_t*>(&b));
    }
};

// channels per thread of the backward: with Kc > 4 its windows and weight-gradient accumulators would not fit in
// registers at 8 bf16 channels, so it takes 4
template <typename T, int KC> constexpr int bwd_channels() { return (sizeof(T) == 2 && KC > 4) ? 4 : ab_vec16<T>::N; }

template <typename T, int V>
__device__ __forceinline__ void load_vec(const T* p, bool ok, float* f) {
    if (ok) {
        const typename Chan<T, V>::raw r = __ldg(reinterpret_cast<const typename Chan<T, V>::raw*>(p));
        Chan<T, V>::unpack(r, f);
    } else {
#pragma unroll
        for (int i = 0; i < V; ++i) f[i] = 0.f;
    }
}

// weights [Di, KC] of channels c0 .. c0 + V - 1 (V * KC contiguous floats, a multiple of 4 starting at a multiple of 4:
// 16-byte loads whatever KC) and their biases
template <int V, int KC>
__device__ __forceinline__ void load_weights(const float* __restrict__ w, const float* __restrict__ bias, int c0, float (&wr)[V][KC], float (&br)[V]) {
    const float4* w4p = reinterpret_cast<const float4*>(w + (size_t)c0 * KC);
#pragma unroll
    for (int q = 0; q < V * KC / 4; ++q) {
        const float4 w4 = __ldg(w4p + q);
        const float e[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) wr[(4 * q + u) / KC][(4 * q + u) % KC] = e[u];
    }
#pragma unroll
    for (int i = 0; i < V; ++i) br[i] = __ldg(bias + c0 + i);
}

// grid.x = ceil(ncv / blockDim.x), grid.y = ceil(L / (TT*ROWS_PER_CTA)), grid.z = B ; block = (cvx, ROWS_PER_CTA)
// Every width but KC = 4 asks for one resident block per SM: left to its own register target ptxas spills some of them
// (fp32 KC = 5 at 64 registers); KC = 4 keeps the bound, and so the allocation, it had before the other widths existed.
template <typename T, int KC>
__global__ void __launch_bounds__(256, KC == 4 ? 0 : 1) conv_silu_fwd_kernel(const T* __restrict__ xp, int64_t xp_stride,
                                                            const float* __restrict__ w, const float* __restrict__ bias,
                                                            T* __restrict__ xa, int L, int Di) {
    constexpr int V = ab_vec16<T>::N;
    const int cv = blockIdx.x * blockDim.x + threadIdx.x;
    const int c0 = cv * V;
    if (c0 >= Di) return;
    const int b = blockIdx.z;
    const int t0 = (blockIdx.y * ROWS_PER_CTA + threadIdx.y) * TT;
    if (t0 >= L) return;
    float wr[V][KC], br[V];
    load_weights<V, KC>(w, bias, c0, wr, br);
    const T* xrow = xp + (size_t)b * L * xp_stride + c0;
    T* orow = xa + ((size_t)b * L) * Di + c0;
    float win[KC - 1][V];   // x[t-(KC-1)] .. x[t-1]
#pragma unroll
    for (int j = 0; j < KC - 1; ++j) {
        const int t = t0 - (KC - 1) + j;
        load_vec<T, V>(xrow + (size_t)t * xp_stride, t >= 0, win[j]);
    }
#pragma unroll 4
    for (int i = 0; i < TT; ++i) {
        const int t = t0 + i;
        if (t >= L) break;
        float cur[V], o[V];
        load_vec<T, V>(xrow + (size_t)t * xp_stride, true, cur);
#pragma unroll
        for (int v = 0; v < V; ++v) {
            float acc = br[v];
#pragma unroll
            for (int j = 0; j < KC - 1; ++j) acc = fmaf(wr[v][j], win[j][v], acc);
            acc = fmaf(wr[v][KC - 1], cur[v], acc);
            o[v] = acc * ab_sigmoid(acc);
#pragma unroll
            for (int j = 0; j < KC - 2; ++j) win[j][v] = win[j + 1][v];
            win[KC - 2][v] = cur[v];
        }
        *reinterpret_cast<uint4*>(orow + (size_t)t * Di) = ab_vec16<T>::pack(o);
    }
}

// Backward (K = KC).  For the owned tokens t0..t0+TT-1 the thread needs dxc at t..t+K-1, i.e. xc (hence xp rows
// t-K+1..t+K-1) and dxa rows t..t+K-1.  It streams u = t0 .. t0+TT+K-2 computing dxc[u] once each, keeps a
// K-deep window of dxc and a (2K-1)-deep window of xp rows is avoided by re-deriving: dxp[t] needs
// dxc[t..t+K-1]; dw[c,j] += dxc[u]*xp[u-K+1+j] only for owned u (so every (u, j) pair is counted once).
template <typename T, int KC>
__global__ void __launch_bounds__(256) conv_silu_bwd_kernel(const T* __restrict__ xp, int64_t xp_stride,
                                                            const T* __restrict__ dxa, const float* __restrict__ w,
                                                            const float* __restrict__ bias, T* __restrict__ dxp, int64_t dxs,
                                                            float* __restrict__ part, int L, int Di, int n_part_rows) {
    constexpr int V = bwd_channels<T, KC>();
    const int cv = blockIdx.x * blockDim.x + threadIdx.x;
    const int c0 = cv * V;
    const int b = blockIdx.z;
    const int t0 = (blockIdx.y * ROWS_PER_CTA + threadIdx.y) * TT;
    const bool active = (c0 < Di) && (t0 < L);
    float gw[V][KC], gb[V];
#pragma unroll
    for (int v = 0; v < V; ++v) {
        gb[v] = 0.f;
#pragma unroll
        for (int j = 0; j < KC; ++j) gw[v][j] = 0.f;
    }
    if (active) {
        float wr[V][KC], br[V];
        load_weights<V, KC>(w, bias, c0, wr, br);
        const T* xrow = xp + (size_t)b * L * xp_stride + c0;
        const T* grow = dxa + ((size_t)b * L) * Di + c0;
        T* orow = dxp + ((size_t)b * L) * dxs + c0;
        float win[KC - 1][V];      // xp[u-(KC-1)] .. xp[u-1]
#pragma unroll
        for (int j = 0; j < KC - 1; ++j) {
            const int t = t0 - (KC - 1) + j;
            load_vec<T, V>(xrow + (size_t)t * xp_stride, t >= 0, win[j]);
        }
        float dwin[KC - 1][V];     // dxc[u-(KC-1)] .. dxc[u-1]
#pragma unroll
        for (int j = 0; j < KC - 1; ++j)
#pragma unroll
            for (int v = 0; v < V; ++v) dwin[j][v] = 0.f;
        const int u_end = min(t0 + TT + KC - 1, L + KC - 1);
        for (int u = t0; u < u_end; ++u) {
            float cur[V], g[V], dxc[V];
            const bool in_seq = u < L;
            load_vec<T, V>(xrow + (size_t)u * xp_stride, in_seq, cur);
            load_vec<T, V>(grow + (size_t)u * Di, in_seq, g);
            const bool owned = in_seq && (u < t0 + TT);
#pragma unroll
            for (int v = 0; v < V; ++v) {
                float acc = br[v];
#pragma unroll
                for (int j = 0; j < KC - 1; ++j) acc = fmaf(wr[v][j], win[j][v], acc);
                acc = fmaf(wr[v][KC - 1], cur[v], acc);
                const float s = ab_sigmoid(acc);
                // d silu(x)/dx = s * (1 + x * (1 - s))
                dxc[v] = in_seq ? g[v] * s * fmaf(acc, 1.f - s, 1.f) : 0.f;
                if (owned) {
                    gb[v] += dxc[v];
#pragma unroll
                    for (int j = 0; j < KC - 1; ++j) gw[v][j] = fmaf(dxc[v], win[j][v], gw[v][j]);
                    gw[v][KC - 1] = fmaf(dxc[v], cur[v], gw[v][KC - 1]);
                }
            }
            // dxp[t] for t = u-(KC-1): sum_j w[j] * dxc[t + KC-1 - j] = w[KC-1]*dxc[u-(KC-1)] + ... + w[1]*dxc[u-1] + w[0]*dxc[u]
            const int t = u - (KC - 1);
            if (t >= t0 && t < L) {
                float o[V];
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    float acc = wr[v][KC - 1] * dwin[0][v];
#pragma unroll
                    for (int j = 1; j < KC - 1; ++j) acc = fmaf(wr[v][KC - 1 - j], dwin[j][v], acc);
                    acc = fmaf(wr[v][0], dxc[v], acc);
                    o[v] = acc;
                }
                *reinterpret_cast<typename Chan<T, V>::raw*>(orow + (size_t)t * dxs) = Chan<T, V>::pack(o);
            }
#pragma unroll
            for (int v = 0; v < V; ++v) {
#pragma unroll
                for (int j = 0; j < KC - 2; ++j) { win[j][v] = win[j + 1][v]; dwin[j][v] = dwin[j + 1][v]; }
                win[KC - 2][v] = cur[v];
                dwin[KC - 2][v] = dxc[v];
            }
        }
    }
    // CTA reduction over the ROWS_PER_CTA thread rows, then one partial row per CTA: part[prow][c][KC + 1]
    constexpr int NQ = KC + 1;        // dw[c, 0 .. KC-1], dbias[c]
    extern __shared__ float sred[];   // [ROWS_PER_CTA][blockDim.x * V * NQ]
    const int per_row = blockDim.x * V * NQ;
    float* mine = sred + threadIdx.y * per_row + threadIdx.x * V * NQ;
#pragma unroll
    for (int v = 0; v < V; ++v) {
#pragma unroll
        for (int j = 0; j < KC; ++j) mine[v * NQ + j] = gw[v][j];
        mine[v * NQ + KC] = gb[v];
    }
    __syncthreads();
    const int prow = blockIdx.z * gridDim.y + blockIdx.y;
    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    for (int i = tid; i < per_row; i += blockDim.x * blockDim.y) {
        float s = 0.f;
#pragma unroll
        for (int r = 0; r < ROWS_PER_CTA; ++r) s += sred[r * per_row + i];
        const int c = blockIdx.x * blockDim.x * V + i / NQ;
        if (c < Di) part[((size_t)prow * Di + c) * NQ + (i % NQ)] = s;
    }
    (void)n_part_rows;
}

// out[c*(KC+1)+q] = sum over partial rows, fixed order (deterministic)
template <int KC>
__global__ void conv_reduce_kernel(const float* __restrict__ part, int n_rows, int Di, float* __restrict__ dw,
                                   float* __restrict__ dbias) {
    constexpr int NQ = KC + 1;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Di * NQ) return;
    float s = 0.f;
    for (int r = 0; r < n_rows; ++r) s += part[(size_t)r * Di * NQ + i];
    const int c = i / NQ, q = i % NQ;
    if (q < KC) dw[c * KC + q] = s; else dbias[c] = s;
}

template <typename T, int KC>
int launch_fwd(const void* xp, int64_t xs, const float* w, const float* bias, void* xa, int B, int L, int Di, cudaStream_t st) {
    constexpr int V = ab_vec16<T>::N;
    const int ncv = Di / V;
    const int bx = ncv >= 32 ? 32 : ncv;
    dim3 block(bx, ROWS_PER_CTA);
    dim3 grid((unsigned)ab_ceil_div(ncv, bx), (unsigned)ab_ceil_div(L, TT * ROWS_PER_CTA), B);
    conv_silu_fwd_kernel<T, KC><<<grid, block, 0, st>>>((const T*)xp, xs, w, bias, (T*)xa, L, Di);
    AB_LAUNCH_CHECK();
    return AB_OK;
}

template <typename T, int KC>
int launch_bwd(const void* xp, int64_t xs, const void* dxa, const float* w, const float* bias, void* dxp, int64_t dxs, float* dw,
               float* dbias, float* part, int B, int L, int Di, cudaStream_t st) {
    constexpr int V = bwd_channels<T, KC>();
    const int ncv = Di / V;
    const int bx = ncv >= 32 ? 32 : ncv;
    dim3 block(bx, ROWS_PER_CTA);
    dim3 grid((unsigned)ab_ceil_div(ncv, bx), (unsigned)ab_ceil_div(L, TT * ROWS_PER_CTA), B);
    const size_t smem = (size_t)ROWS_PER_CTA * bx * V * (KC + 1) * sizeof(float);      // <= 40 KB for every (T, KC)
    const int n_part = grid.y * grid.z;
    conv_silu_bwd_kernel<T, KC><<<grid, block, smem, st>>>((const T*)xp, xs, (const T*)dxa, w, bias, (T*)dxp, dxs, part, L, Di, n_part);
    AB_LAUNCH_CHECK();
    conv_reduce_kernel<KC><<<(unsigned)ab_ceil_div(Di * (KC + 1), 128), 128, 0, st>>>(part, n_part, Di, dw, dbias);
    AB_LAUNCH_CHECK();
    return AB_OK;
}

template <typename T>
int launch_fwd_kc(const void* xp, int64_t xs, const float* w, const float* bias, void* xa, int B, int L, int Di, int Kc, cudaStream_t st) {
    switch (Kc) {
        case 2: return launch_fwd<T, 2>(xp, xs, w, bias, xa, B, L, Di, st);
        case 3: return launch_fwd<T, 3>(xp, xs, w, bias, xa, B, L, Di, st);
        case 4: return launch_fwd<T, 4>(xp, xs, w, bias, xa, B, L, Di, st);
        case 5: return launch_fwd<T, 5>(xp, xs, w, bias, xa, B, L, Di, st);
        case 6: return launch_fwd<T, 6>(xp, xs, w, bias, xa, B, L, Di, st);
        case 7: return launch_fwd<T, 7>(xp, xs, w, bias, xa, B, L, Di, st);
        default: return launch_fwd<T, 8>(xp, xs, w, bias, xa, B, L, Di, st);
    }
}

template <typename T>
int launch_bwd_kc(const void* xp, int64_t xs, const void* dxa, const float* w, const float* bias, void* dxp, int64_t dxs, float* dw,
                  float* dbias, float* part, int B, int L, int Di, int Kc, cudaStream_t st) {
    switch (Kc) {
        case 2: return launch_bwd<T, 2>(xp, xs, dxa, w, bias, dxp, dxs, dw, dbias, part, B, L, Di, st);
        case 3: return launch_bwd<T, 3>(xp, xs, dxa, w, bias, dxp, dxs, dw, dbias, part, B, L, Di, st);
        case 4: return launch_bwd<T, 4>(xp, xs, dxa, w, bias, dxp, dxs, dw, dbias, part, B, L, Di, st);
        case 5: return launch_bwd<T, 5>(xp, xs, dxa, w, bias, dxp, dxs, dw, dbias, part, B, L, Di, st);
        case 6: return launch_bwd<T, 6>(xp, xs, dxa, w, bias, dxp, dxs, dw, dbias, part, B, L, Di, st);
        case 7: return launch_bwd<T, 7>(xp, xs, dxa, w, bias, dxp, dxs, dw, dbias, part, B, L, Di, st);
        default: return launch_bwd<T, 8>(xp, xs, dxa, w, bias, dxp, dxs, dw, dbias, part, B, L, Di, st);
    }
}

int check_args(int B, int L, int Di, int Kc, int64_t xs, int dtype) {
    AB_REQUIRE(Kc >= 2 && Kc <= KC_MAX, "causal_conv1d: ssm_conv_kernel must be in [2, %d] (got %d)", KC_MAX, Kc);
    AB_REQUIRE(B > 0 && L > 0 && Di > 0, "causal_conv1d: empty shape B=%d L=%d Di=%d", B, L, Di);
    AB_REQUIRE(dtype == AB_F32 || dtype == AB_BF16, "causal_conv1d: bad dtype %d", dtype);
    const int V = dtype == AB_F32 ? 4 : 8;
    AB_REQUIRE(Di % V == 0 && xs % V == 0, "causal_conv1d: Di (%d) and row stride (%lld) must be multiples of %d", Di, (long long)xs, V);
    return AB_OK;
}

}  // namespace

extern "C" int ab_causal_conv1d_silu_fwd(const void* xp, int64_t xp_stride, const float* w, const float* bias, void* xa,
                                         int B, int L, int Di, int Kc, int dtype, cudaStream_t stream) {
    if (int e = check_args(B, L, Di, Kc, xp_stride, dtype)) return e;
    return dtype == AB_F32 ? launch_fwd_kc<float>(xp, xp_stride, w, bias, xa, B, L, Di, Kc, stream)
                           : launch_fwd_kc<__nv_bfloat16>(xp, xp_stride, w, bias, xa, B, L, Di, Kc, stream);
}

// sized for the largest Kc: (KC_MAX + 1) partial sums per channel and partial row
extern "C" size_t ab_causal_conv1d_silu_bwd_workspace_bytes(int B, int L, int Di) {
    return (size_t)B * ab_ceil_div(L, TT * ROWS_PER_CTA) * Di * (KC_MAX + 1) * sizeof(float);
}

extern "C" int ab_causal_conv1d_silu_bwd(const void* xp, int64_t xp_stride, const void* dxa, const float* w,
                                         const float* bias, void* dxp, int64_t dxp_stride, float* dw, float* dbias, void* ws,
                                         size_t ws_bytes, int B, int L, int Di, int Kc, int dtype, cudaStream_t stream) {
    if (int e = check_args(B, L, Di, Kc, xp_stride, dtype)) return e;
    if (int e = check_args(B, L, Di, Kc, dxp_stride, dtype)) return e;
    AB_REQUIRE(dxp_stride >= Di, "causal_conv1d_bwd: dxp row stride smaller than the row");
    AB_REQUIRE(ws_bytes >= ab_causal_conv1d_silu_bwd_workspace_bytes(B, L, Di), "causal_conv1d_bwd: workspace too small");
    return dtype == AB_F32
               ? launch_bwd_kc<float>(xp, xp_stride, dxa, w, bias, dxp, dxp_stride, dw, dbias, (float*)ws, B, L, Di, Kc, stream)
               : launch_bwd_kc<__nv_bfloat16>(xp, xp_stride, dxa, w, bias, dxp, dxp_stride, dw, dbias, (float*)ws, B, L, Di, Kc, stream);
}
