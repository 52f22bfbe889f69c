// MoE dispatch on the device: capacity plan (bit-exact restatement of the reference's slot-major /
// expert-inner loop with keep-the-largest-gate overflow, core.py:508-511, 547-590), token permutation
// with the per-expert LayerNorm fused in (core.py:593 + :436), weighted un-permutation (core.py:605),
// their backward passes and per-expert column sums for the bias gradients.  No host synchronisation:
// everything downstream reads counts / offsets from device memory.
#include "common.cuh"

namespace {

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

// ---- expert parallelism over peer memory (NVLink): rows of the permuted layout that live in ANOTHER rank's buffer.
// The local layout is [W destination ranks][rows_per_peer]; row r belongs to rank d = r / rows_per_peer and sits there in
// block `rank` (the source) of a [W sources][rows_per_peer] buffer whose peer-mapped base address is base[d].
// n == 0: plain local buffer.
constexpr int AB_MAX_PEERS = 16;
struct PeerRows {
    unsigned char* base[AB_MAX_PEERS];
    int n, rows_per_peer, rank;
};
__device__ __forceinline__ unsigned char* peer_row(const PeerRows& pr, void* local, int64_t r, int Dm, int es) {
    if (pr.n == 0) return reinterpret_cast<unsigned char*>(local) + (size_t)r * Dm * es;
    const int d = (int)(r / pr.rows_per_peer);
    const int64_t j = r - (int64_t)d * pr.rows_per_peer;
    return pr.base[d] + ((size_t)pr.rank * pr.rows_per_peer + j) * Dm * es;
}

// four consecutive elements as ONE store (8 bytes bf16 / 16 bytes fp32): whole sectors also when the row is peer memory
template <typename T>
__device__ __forceinline__ void st4(T* p, float a, float b, float c, float d) {
    if constexpr (sizeof(T) == 4) {
        *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
    } else {
        __nv_bfloat162 lo = __floats2bfloat162_rn(a, b), hi = __floats2bfloat162_rn(c, d);
        *reinterpret_cast<uint2*>(p) = make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
    }
}

// Capacity plan over the whole GPU, in four steps that each read idx / w once (launch order = dependency order):
//   (1) plan_hist_kernel, pass 3..0: per (expert, slot) 256-bin histograms of one byte of the weight bits of the candidates
//       that still match the threshold prefix found so far.  The last CTA to finish (atomic ticket) turns the global
//       histograms into the next byte of the threshold; after pass 3 it also fixes each slot's mode and base from the
//       candidate counts: slot k is filled before slot k+1 with the remaining capacity.
//   (2) plan_chunk_count_kernel: per chunk of PLAN_CHUNK tokens and (expert, slot), the candidates above the threshold
//       ("gt") and equal to it ("eq").
//   (3) plan_pos_kernel: a kept (token, slot) sits at base + gt before it + min(eq before it, eq taken): ties at the
//       threshold are taken in token order.  Each CTA adds the counts of the chunks before its own.  Same result as one CTA walking the tokens of each expert in order.
constexpr int PLAN_THREADS = 256;
constexpr int PLAN_CHUNK = PLAN_THREADS;     // tokens per CTA of steps (2) and (3): one per thread
constexpr int HIST_TOKENS = PLAN_THREADS;    // tokens per CTA of step (1): one per thread, loads all in flight at once

// per (expert, slot) state written by the last CTA of each histogram pass
struct PlanSel {
    uint32_t prefix;   // threshold bits found so far (then the threshold itself)
    int need;          // elements equal to the threshold that are still to be taken
    int mode;          // 0 none, 1 all, 2 select the `need` largest
    int base;          // kept rows of the expert in earlier slots
};

// From a 256-bin histogram, by one warp: the bin holding the `need`-th largest element counted from the top, and how many
// are still needed inside it.  Lane l owns bins [8l, 8l+8); suffix sums over the lanes by shuffles.
__device__ __forceinline__ void warp_select_bin(const int* hist, int lane, int& need, int& sel_bin) {
    int h[8], mine = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) { h[i] = hist[lane * 8 + i]; mine += h[i]; }
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_down_sync(0xffffffffu, incl, o);
        if (lane + o < 32) incl += v;
    }
    const int above = incl - mine;
    const int nd0 = need;
    const bool here = above < nd0 && above + mine >= nd0;       // the wanted element lies in this lane's bins
    const unsigned who = __ballot_sync(0xffffffffu, here);
    int bin = 0, nd = 0;
    if (who == 0u) {                                            // fewer than `need` elements in total: lowest bin
        nd = __shfl_sync(0xffffffffu, nd0 - (above + mine) + h[0], 0);
        bin = 0;
    } else {
        const int src = __ffs(who) - 1;
        int b = 7, n2 = nd0 - above;
        for (; b > 0; --b) {
            if (h[b] >= n2) break;
            n2 -= h[b];
        }
        bin = __shfl_sync(0xffffffffu, lane * 8 + b, src);
        nd = __shfl_sync(0xffffffffu, n2, src);
    }
    sel_bin = bin;
    need = nd;
}

// histogram increment with one shared-memory atomic per distinct bin per warp: gate weights share their top bytes, so
// per-element atomics on the same bin would serialise.  Must be reached by all 32 lanes.
__device__ __forceinline__ void hist_add_warp(int* hist, bool valid, int bin) {
    const unsigned act = __ballot_sync(0xffffffffu, valid);
    if (valid) {
        const unsigned peers = __match_any_sync(act, bin);
        if ((__ffs(peers) - 1) == (int)(threadIdx.x & 31)) atomicAdd(&hist[bin], __popc(peers));
    }
}

// true in exactly one CTA of the grid, the last to get here, after all others' global writes are visible
__device__ __forceinline__ bool last_cta(int* ticket) {
    __shared__ bool s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(ticket, 1) == (int)(gridDim.x * gridDim.y) - 1;
    __syncthreads();
    if (s_last) __threadfence();
    return s_last;
}

// grid (ceil(S / HIST_TOKENS), K): slot k = blockIdx.y.  hist: [E*K][256] of this pass, zeroed by the caller.
__global__ void __launch_bounds__(PLAN_THREADS) plan_hist_kernel(const int32_t* __restrict__ idx, const float* __restrict__ w,
                                                                 const int32_t* __restrict__ active, int cap, int pass,
                                                                 int* __restrict__ ghist, PlanSel* __restrict__ sel,
                                                                 int* __restrict__ any_select, int* __restrict__ ticket,
                                                                 int32_t* __restrict__ counts, int S, int K, int E) {
    __shared__ int hist[32 * 256];
    if (pass < 3 && *any_select == 0) return;                  // uniform over the grid: no slot overflows its capacity
    const int k = blockIdx.y, tid = threadIdx.x;
    for (int i = tid; i < E * 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    const int shift = 8 * pass;
    const uint32_t mask = pass == 3 ? 0u : 0xffffffffu << (shift + 8);
    const int s_end = min(S, (int)(blockIdx.x + 1) * HIST_TOKENS);
    for (int s0 = blockIdx.x * HIST_TOKENS; s0 < s_end; s0 += blockDim.x) {
        const int s = s0 + tid;
        bool c = s < s_end;
        int e = 0;
        uint32_t b = 0u;
        if (c) {
            e = idx[(size_t)s * K + k];
            b = __float_as_uint(w[(size_t)s * K + k]);
            if (pass < 3) {
                const PlanSel st = sel[e * K + k];
                c = st.mode == 2 && (b & mask) == st.prefix;
            }
        }
        hist_add_warp(hist, c, e * 256 + (int)((b >> shift) & 0xffu));
    }
    __syncthreads();
    int* gh = ghist + (size_t)k * 256;                         // [E][K][256]: expert e, slot k at (e*K + k)*256
    for (int i = tid; i < E * 256; i += blockDim.x) {
        const int h = hist[i];
        if (h) atomicAdd(&gh[(size_t)(i >> 8) * K * 256 + (i & 255)], h);
    }
    if (!last_cta(ticket)) return;
    // ---- last CTA: one warp per expert
    const int lane = tid & 31, warp = tid >> 5;
    int any = 0;
    for (int e = warp; e < E; e += blockDim.x >> 5) {
        int kept = 0;
        for (int kk = 0; kk < K; ++kk) {
            const int* hk = ghist + ((size_t)e * K + kk) * 256;
            PlanSel st;
            if (pass == 3) {
                int n = 0;
                for (int i = lane; i < 256; i += 32) n += hk[i];
                n = __reduce_add_sync(0xffffffffu, n);
                const bool is_active = active == nullptr || active[e] != 0;
                const int rem = cap - kept;
                st.mode = 0;
                if (is_active && n > 0 && rem > 0) st.mode = n <= rem ? 1 : 2;
                st.base = kept;
                st.need = rem;
                st.prefix = 0u;
                kept += st.mode == 1 ? n : (st.mode == 2 ? rem : 0);
            } else {
                st = sel[e * K + kk];
            }
            if (st.mode == 2) {
                int bin;
                warp_select_bin(hk, lane, st.need, bin);
                st.prefix |= (uint32_t)bin << shift;
                any = 1;
            }
            if (lane == 0) sel[e * K + kk] = st;
        }
        if (pass == 3 && lane == 0) counts[e] = kept;
    }
    if (pass == 3) {
        __shared__ int s_any;
        if (tid == 0) s_any = 0;
        __syncthreads();
        if (any && lane == 0) s_any = 1;
        __syncthreads();
        if (tid == 0) *any_select = s_any;
    }
}

// the class of a candidate under its slot's threshold: 0 above it (or mode 1), 1 equal (mode 2), -1 not kept
__device__ __forceinline__ int plan_class(const PlanSel& st, uint32_t b) {
    if (st.mode == 1) return 0;
    if (st.mode == 2) return b > st.prefix ? 0 : (b == st.prefix ? 1 : -1);
    return -1;
}

// grid (ceil(S / PLAN_CHUNK), K).  cc: [chunks][K][E][2] candidates above / equal to the threshold per chunk
__global__ void __launch_bounds__(PLAN_THREADS) plan_chunk_count_kernel(const int32_t* __restrict__ idx, const float* __restrict__ w,
                                                                        const PlanSel* __restrict__ sel, int* __restrict__ cc,
                                                                        int S, int K, int E) {
    __shared__ int cnt[64];
    const int k = blockIdx.y, tid = threadIdx.x;
    if (tid < 2 * E) cnt[tid] = 0;
    __syncthreads();
    const int s = blockIdx.x * PLAN_CHUNK + tid;
    int cls = -1, e = 0;
    if (s < S) {
        e = idx[(size_t)s * K + k];
        cls = plan_class(sel[e * K + k], __float_as_uint(w[(size_t)s * K + k]));
    }
    hist_add_warp(cnt, cls >= 0, e * 2 + (cls > 0 ? 1 : 0));
    __syncthreads();
    if (tid < 2 * E) cc[((size_t)blockIdx.x * K + k) * 2 * E + tid] = cnt[tid];
}

// grid (ceil(S / PLAN_CHUNK), K): row_local[s,k] = position of the kept (token, slot) inside the expert's segment, -1 if dropped
__global__ void __launch_bounds__(PLAN_THREADS) plan_pos_kernel(const int32_t* __restrict__ idx, const float* __restrict__ w,
                                                                const PlanSel* __restrict__ sel, const int* __restrict__ cc,
                                                                int32_t* __restrict__ row_local, int S, int K, int E) {
    __shared__ int wcnt[PLAN_THREADS / 32][64];                // per warp: [e][gt, eq], then their exclusive prefix over warps
    __shared__ int sbase[PLAN_THREADS];
    const int k = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // counts of the earlier chunks: column (e, gt|eq) = tid % 2E, chunk groups interleaved over the rest of the threads
    {
        const int ncol = 2 * E, ng = PLAN_THREADS / ncol, col = tid % ncol, grp = tid / ncol;
        int sum = 0;
        if (grp < ng)
            for (int c = grp; c < (int)blockIdx.x; c += ng) sum += cc[((size_t)c * K + k) * ncol + col];
        sbase[tid] = sum;
    }
    const int s = blockIdx.x * PLAN_CHUNK + tid;
    int cls = -1, e = 0;
    PlanSel st{0u, 0, 0, 0};
    if (s < S) {
        e = idx[(size_t)s * K + k];
        st = sel[e * K + k];
        cls = plan_class(st, __float_as_uint(w[(size_t)s * K + k]));
    }
    const unsigned valid = __ballot_sync(0xffffffffu, s < S);
    const unsigned same = __match_any_sync(0xffffffffu, s < S ? e : -1) & valid;
    const unsigned gtm = __ballot_sync(0xffffffffu, cls == 0), eqm = __ballot_sync(0xffffffffu, cls == 1);
    const unsigned lt = (1u << lane) - 1u;
    for (int i = tid; i < (PLAN_THREADS / 32) * 64; i += blockDim.x) (&wcnt[0][0])[i] = 0;
    __syncthreads();
    if (s < S && (__ffs(same) - 1) == lane) {
        wcnt[warp][2 * e] = __popc(same & gtm);
        wcnt[warp][2 * e + 1] = __popc(same & eqm);
    }
    __syncthreads();
    if (tid < 2 * E) {
        int run = 0;
        for (int g = 0; g < PLAN_THREADS / (2 * E); ++g) run += sbase[g * 2 * E + tid];
        for (int wv = 0; wv < PLAN_THREADS / 32; ++wv) {
            const int v = wcnt[wv][tid];
            wcnt[wv][tid] = run;
            run += v;
        }
    }
    __syncthreads();
    if (s < S) {
        int r = -1;
        if (cls >= 0) {
            const int gt_before = wcnt[warp][2 * e] + __popc(same & gtm & lt);
            const int eq_before = wcnt[warp][2 * e + 1] + __popc(same & eqm & lt);
            if (cls == 0 || eq_before < st.need) r = st.base + gt_before + min(eq_before, st.need);
        }
        row_local[(size_t)s * K + k] = r;
    }
}

__global__ void plan_finalize_kernel(const int32_t* __restrict__ idx, const int32_t* __restrict__ counts,
                                     const int32_t* __restrict__ row_local, int32_t* __restrict__ seg_off,
                                     int32_t* __restrict__ row_of, int32_t* __restrict__ tok_of_row,
                                     int32_t* __restrict__ slot_of_row, int32_t* __restrict__ tile_expert,
                                     int32_t* __restrict__ n_rows, int S, int K, int E, int align, int64_t max_rows,
                                     int fixed_seg) {
    __shared__ int soff[34];
    if (threadIdx.x == 0) {
        int o = 0, kept = 0;
        for (int e = 0; e < E; ++e) {
            soff[e] = o;
            if (fixed_seg > 0 && counts[e] > fixed_seg) __trap();      // the caller sized the segments too small: never overflow into a neighbour
            o += fixed_seg > 0 ? fixed_seg : (counts[e] + align - 1) / align * align;
            kept += counts[e];
        }
        soff[E] = o;
        soff[E + 1] = kept;
    }
    __syncthreads();
    if (blockIdx.x == 0) {
        for (int i = threadIdx.x; i <= E; i += blockDim.x) seg_off[i] = soff[i];
        if (threadIdx.x == 0) { n_rows[0] = soff[E]; n_rows[1] = soff[E + 1]; }
        const int ntiles = (int)(max_rows / align);
        for (int t = threadIdx.x; t < ntiles; t += blockDim.x) {
            const int r = t * align;
            int ex = -1;
            for (int e = 0; e < E; ++e)
                if (r >= soff[e] && r < soff[e + 1]) ex = e;
            tile_expert[t] = ex;
        }
    }
    const int64_t n = (int64_t)S * K;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int rl = row_local[i];
        if (rl >= 0) {
            const int r = soff[idx[i]] + rl;
            row_of[i] = r;
            tok_of_row[r] = (int)(i / K);
            slot_of_row[r] = (int)(i % K);
        } else {
            row_of[i] = -1;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// permute + LayerNorm (warp per row)
// ---------------------------------------------------------------------------------------------
template <typename TI, typename TO>
__global__ void __launch_bounds__(256) permute_ln_kernel(const TI* __restrict__ x, const float* __restrict__ stats,
                                                         const float* __restrict__ ln_w, const float* __restrict__ ln_b,
                                                         const int32_t* __restrict__ tok_of_row,
                                                         const int32_t* __restrict__ tile_expert,
                                                         const int32_t* __restrict__ n_rows, TO* __restrict__ xn, int Dm,
                                                         int align, const PeerRows pr) {
    const int lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    const int total = n_rows[0];
    for (int r = blockIdx.x * wpb + (threadIdx.x >> 5); r < total; r += gridDim.x * wpb) {
        const int tok = tok_of_row[r];
        TO* orow = reinterpret_cast<TO*>(peer_row(pr, xn, r, Dm, (int)sizeof(TO)));     // the owner's receive buffer under EP
        if (tok < 0) {
            for (int d = lane * 4; d < Dm; d += 128) st4<TO>(orow + d, 0.f, 0.f, 0.f, 0.f);
            continue;
        }
        const int e = tile_expert[r / align];
        const float mean = stats[2 * (size_t)tok], rstd = stats[2 * (size_t)tok + 1];
        const TI* irow = x + (size_t)tok * Dm;
        const float* g = ln_w + (size_t)e * Dm;
        const float* bb = ln_b + (size_t)e * Dm;
        for (int d = lane * 4; d < Dm; d += 128) {
            const float4 gv = __ldg(reinterpret_cast<const float4*>(g + d));
            const float4 bv = __ldg(reinterpret_cast<const float4*>(bb + d));
            float xv[4];
#pragma unroll
            for (int v = 0; v < 4; ++v) xv[v] = ab_to_float(irow[d + v]);
            const float o0 = fmaf((xv[0] - mean) * rstd, gv.x, bv.x), o1 = fmaf((xv[1] - mean) * rstd, gv.y, bv.y);
            const float o2 = fmaf((xv[2] - mean) * rstd, gv.z, bv.z), o3 = fmaf((xv[3] - mean) * rstd, gv.w, bv.w);
            st4<TO>(orow + d, o0, o1, o2, o3);
        }
    }
}

// out[s,:] = sum_k w[s,k] * y[row_of[s,k],:]   (warp per token, fixed slot order).  The loads of a group of chunks - 4
// elements of every one of the K rows each - are all issued before the first is used.
template <typename TY, typename TO, int KM>
__global__ void __launch_bounds__(256) unpermute_kernel(const TY* __restrict__ y, const int32_t* __restrict__ row_of,
                                                        const float* __restrict__ w, const float* __restrict__ res, TO* __restrict__ out,
                                                        const uint32_t* __restrict__ seed, uint32_t thresh, float scale, int S, int K, int Dm) {
    constexpr int DU = 8 / KM;           // chunks in flight (KM = upper bound of the experts per token)
    const int lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    uint32_t s0 = 0, s1 = 0;
    if (seed) { s0 = __ldg(seed); s1 = __ldg(seed + 1); }
    for (int s = blockIdx.x * wpb + (threadIdx.x >> 5); s < S; s += gridDim.x * wpb) {
        TO* orow = out + (size_t)s * Dm;
        const TY* rows[KM];
        float wk[KM];
        int rid[KM];
#pragma unroll
        for (int k = 0; k < KM; ++k) {
            rid[k] = k < K ? row_of[(size_t)s * K + k] : -1;
            wk[k] = rid[k] >= 0 ? w[(size_t)s * K + k] : 0.f;
            rows[k] = rid[k] >= 0 ? y + (size_t)rid[k] * Dm : nullptr;
        }
        for (int d0 = lane * 4; d0 < Dm; d0 += 128 * DU) {
            float yv[DU][KM][4];
#pragma unroll
            for (int u = 0; u < DU; ++u) {
                const int d = d0 + u * 128;
#pragma unroll
                for (int k = 0; k < KM; ++k) {
                    if (k < K && rows[k] != nullptr && d < Dm) ld4g<TY>(rows[k] + d, yv[u][k]);
                    else { yv[u][k][0] = yv[u][k][1] = yv[u][k][2] = yv[u][k][3] = 0.f; }
                }
            }
#pragma unroll
            for (int u = 0; u < DU; ++u) {
                const int d = d0 + u * 128;
                if (d >= Dm) break;
                float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int k = 0; k < KM; ++k) {
                    if (k < K && rows[k] != nullptr) {
#pragma unroll
                        for (int v = 0; v < 4; ++v) acc[v] += yv[u][k][v] * wk[k];   // separate mul and add, as index_add_(y*w)
                    }
                }
                // the caller's output dropout and residual add (core.py:918-919) in the same pass
                if (seed) {
#pragma unroll
                    for (int v = 0; v < 4; ++v) acc[v] = ab_out_keep(s0, s1, (uint64_t)s * Dm + d + v, thresh) ? acc[v] * scale : 0.f;
                }
                if (res) {
                    const float4 rr = *reinterpret_cast<const float4*>(res + (size_t)s * Dm + d);
                    acc[0] += rr.x; acc[1] += rr.y; acc[2] += rr.z; acc[3] += rr.w;
                }
                st4<TO>(orow + d, acc[0], acc[1], acc[2], acc[3]);
            }
        }
    }
}

// dy[r,:] = w[r] * dout[tok,:] ; dw_row[r] = <dout[tok,:], y[r,:]>
template <typename TD, typename TY, typename TO>
__global__ void __launch_bounds__(256) unpermute_bwd_kernel(const TD* __restrict__ dout, const TY* __restrict__ y,
                                                            const float* __restrict__ w, const int32_t* __restrict__ tok_of_row,
                                                            const int32_t* __restrict__ slot_of_row,
                                                            const int32_t* __restrict__ n_rows, TO* __restrict__ dy,
                                                            float* __restrict__ dw_row, const uint32_t* __restrict__ seed, uint32_t thresh,
                                                            float scale, int K, int Dm, const PeerRows pr) {
    const int lane = threadIdx.x & 31;
    const int wpb = blockDim.x >> 5;
    const int total = n_rows[0];
    uint32_t s0 = 0, s1 = 0;
    if (seed) { s0 = __ldg(seed); s1 = __ldg(seed + 1); }
    for (int r = blockIdx.x * wpb + (threadIdx.x >> 5); r < total; r += gridDim.x * wpb) {
        const int tok = tok_of_row[r];
        TO* orow = reinterpret_cast<TO*>(peer_row(pr, dy, r, Dm, (int)sizeof(TO)));     // the owner's receive buffer under EP
        if (tok < 0) {
            for (int d = lane * 4; d < Dm; d += 128) st4<TO>(orow + d, 0.f, 0.f, 0.f, 0.f);
            if (lane == 0) dw_row[r] = 0.f;
            continue;
        }
        const float wk = w[(size_t)tok * K + slot_of_row[r]];
        const TD* drow = dout + (size_t)tok * Dm;
        const TY* yrow = y + (size_t)r * Dm;
        float dot = 0.f;
        for (int d = lane * 4; d < Dm; d += 128) {
            float o[4];
#pragma unroll
            for (int v = 0; v < 4; ++v) {
                float g = ab_to_float(drow[d + v]);
                if (seed) g = ab_out_keep(s0, s1, (uint64_t)tok * Dm + d + v, thresh) ? g * scale : 0.f;      // the forward's output-dropout mask
                dot = fmaf(g, ab_to_float(yrow[d + v]), dot);
                o[v] = g * wk;
            }
            st4<TO>(orow + d, o[0], o[1], o[2], o[3]);
        }
        dot = ab_warp_sum(dot);
        if (lane == 0) dw_row[r] = dot;
    }
}

// ---------------------------------------------------------------------------------------------
// LayerNorm backward per permuted row (warp per row) and per-tile partial sums of the affine grads
// ---------------------------------------------------------------------------------------------
template <typename TX, typename TG>
__global__ void __launch_bounds__(256) permute_ln_bwd_rows_kernel(const TG* __restrict__ dxn, const TX* __restrict__ x,
                                                                  const float* __restrict__ stats, const float* __restrict__ ln_w,
                                                                  const int32_t* __restrict__ tok_of_row,
                                                                  const int32_t* __restrict__ tile_expert,
                                                                  const int32_t* __restrict__ n_rows, float* __restrict__ dxrow,
                                                                  int Dm, int align) {
    const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    const int total = n_rows[0];
    for (int r = blockIdx.x * wpb + (threadIdx.x >> 5); r < total; r += gridDim.x * wpb) {
        const int tok = tok_of_row[r];
        if (tok < 0) continue;
        const int e = tile_expert[r / align];
        const float* g = ln_w + (size_t)e * Dm;
        const float mean = stats[2 * (size_t)tok], rstd = stats[2 * (size_t)tok + 1];
        const TX* xr = x + (size_t)tok * Dm;
        const TG* gr = dxn + (size_t)r * Dm;
        float a1 = 0.f, a2 = 0.f;
        for (int d = lane * 4; d < Dm; d += 128) {
            const float4 gv = __ldg(reinterpret_cast<const float4*>(g + d));
            const float gg[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
            for (int v = 0; v < 4; ++v) {
                const float dh = ab_to_float(gr[d + v]) * gg[v];
                const float xh = (ab_to_float(xr[d + v]) - mean) * rstd;
                a1 += dh;
                a2 = fmaf(dh, xh, a2);
            }
        }
        const float m1 = ab_warp_sum(a1) / (float)Dm, m2 = ab_warp_sum(a2) / (float)Dm;
        float* orow = dxrow + (size_t)r * Dm;
        for (int d = lane * 4; d < Dm; d += 128) {
            const float4 gv = __ldg(reinterpret_cast<const float4*>(g + d));
            const float gg[4] = {gv.x, gv.y, gv.z, gv.w};
            float o[4];
#pragma unroll
            for (int v = 0; v < 4; ++v) {
                const float dh = ab_to_float(gr[d + v]) * gg[v];
                const float xh = (ab_to_float(xr[d + v]) - mean) * rstd;
                o[v] = rstd * (dh - m1 - xh * m2);
            }
            *reinterpret_cast<float4*>(orow + d) = make_float4(o[0], o[1], o[2], o[3]);
        }
    }
}

// Row pass and per-tile column partials in one kernel (hidden sizes up to NIT * 128): one CTA per 128-row tile (one
// expert), a lane always owns the same columns, so dxn * xhat and dxn accumulate in registers while the rows stream; the
// warps then add their sums in warp order.  Replaces the rows + cols kernel pair (one read of dxn and x instead of two).
template <typename TX, typename TG, int NIT>
__global__ void __launch_bounds__(256, NIT <= 6 ? 3 : 2) permute_ln_bwd_fused_kernel(const TG* __restrict__ dxn, const TX* __restrict__ x,
                                                                   const float* __restrict__ stats, const float* __restrict__ ln_w,
                                                                   const int32_t* __restrict__ tok_of_row,
                                                                   const int32_t* __restrict__ tile_expert,
                                                                   const int32_t* __restrict__ n_rows, float* __restrict__ dxrow,
                                                                   float* __restrict__ part, int Dm, int align, int ratio) {
    // `align` = rows of this kernel's work tile, `ratio` work tiles per tile_expert entry (the GEMM's row tile)
    __shared__ float sacc[2][NIT * 128];
    const int t = blockIdx.x;
    if ((int64_t)t * align >= n_rows[0]) return;
    const int e = tile_expert[t / ratio];
    if (e < 0) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const float* g = ln_w + (size_t)e * Dm;
    float gw[NIT][4], gb[NIT][4];
#pragma unroll
    for (int it = 0; it < NIT; ++it) {
#pragma unroll
        for (int v = 0; v < 4; ++v) { gw[it][v] = 0.f; gb[it][v] = 0.f; }
    }
    // The loads of a row are issued piecewise (register budget), each piece a full memory latency when it misses: the
    // NEXT row of this warp (token id looked up two rows ahead) is therefore prefetched into L1 while this one is processed.
    int tok_cur = tok_of_row[t * align + warp];
    int tok_nxt = warp + wpb < align ? tok_of_row[t * align + warp + wpb] : -1;
    for (int i = warp; i < align; i += wpb) {
        const int r = t * align + i;
        const int tok = tok_cur;
        tok_cur = tok_nxt;
        tok_nxt = i + 2 * wpb < align ? tok_of_row[t * align + i + 2 * wpb] : -1;
        if (tok_cur >= 0) {
            const char* px = reinterpret_cast<const char*>(x + (size_t)tok_cur * Dm);
            const char* pg = reinterpret_cast<const char*>(dxn + (size_t)(r + wpb) * Dm);
            for (int o = lane * 128; o < Dm * (int)sizeof(TX); o += 32 * 128) asm volatile("prefetch.global.L1 [%0];" ::"l"(px + o));
            for (int o = lane * 128; o < Dm * (int)sizeof(TG); o += 32 * 128) asm volatile("prefetch.global.L1 [%0];" ::"l"(pg + o));
        }
        if (tok < 0) continue;
        const float mean = stats[2 * (size_t)tok], rstd = stats[2 * (size_t)tok + 1];
        const TX* xr = x + (size_t)tok * Dm;
        const TG* gr = dxn + (size_t)r * Dm;
        // pass 1: column partials and the two row sums (the row is read again in pass 2 from L1: keeping it in
        // registers would halve the resident warps)
        float a1 = 0.f, a2 = 0.f;
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
            const int d = it * 128 + lane * 4;
            if (d < Dm) {
                float fx[4], fg[4], gg[4];
                ld4g<TX>(xr + d, fx);
                ld4g<TG>(gr + d, fg);
                ld4g<float>(g + d, gg);
#pragma unroll
                for (int v = 0; v < 4; ++v) {
                    const float xh = (fx[v] - mean) * rstd;
                    gw[it][v] = fmaf(fg[v], xh, gw[it][v]);
                    gb[it][v] += fg[v];
                    const float dh = fg[v] * gg[v];
                    a1 += dh;
                    a2 = fmaf(dh, xh, a2);
                }
            }
        }
        const float m1 = ab_warp_sum(a1) / (float)Dm, m2 = ab_warp_sum(a2) / (float)Dm;
        float* orow = dxrow + (size_t)r * Dm;
#pragma unroll
        for (int it = 0; it < NIT; ++it) {
            const int d = it * 128 + lane * 4;
            if (d < Dm) {
                float fx[4], fg[4], gg[4], o[4];
                ld4g<TX>(xr + d, fx);
                ld4g<TG>(gr + d, fg);
                ld4g<float>(g + d, gg);
#pragma unroll
                for (int v = 0; v < 4; ++v) o[v] = rstd * (fg[v] * gg[v] - m1 - (fx[v] - mean) * rstd * m2);
                *reinterpret_cast<float4*>(orow + d) = make_float4(o[0], o[1], o[2], o[3]);
            }
        }
    }
    for (int wv = 0; wv < wpb; ++wv) {
        if (warp == wv) {
#pragma unroll
            for (int it = 0; it < NIT; ++it) {
#pragma unroll
                for (int v = 0; v < 4; ++v) {
                    const int i = it * 128 + lane * 4 + v;
                    sacc[0][i] = wv ? sacc[0][i] + gw[it][v] : gw[it][v];
                    sacc[1][i] = wv ? sacc[1][i] + gb[it][v] : gb[it][v];
                }
            }
        }
        __syncthreads();
    }
    for (int i = threadIdx.x; i < 2 * Dm; i += blockDim.x) {
        const int q = i / Dm, d = i % Dm;
        part[((size_t)t * 2 + q) * Dm + d] = sacc[q][d];
    }
}

// grid (tiles, ceil(Dm/128)); block (32 lanes x 4 columns, 8 warps over the tile's rows)
template <typename TX, typename TG>
__global__ void __launch_bounds__(256) permute_ln_bwd_cols_kernel(const TG* __restrict__ dxn, const TX* __restrict__ x,
                                                                  const float* __restrict__ stats,
                                                                  const int32_t* __restrict__ tok_of_row,
                                                                  const int32_t* __restrict__ tile_expert,
                                                                  const int32_t* __restrict__ n_rows, float* __restrict__ part,
                                                                  int Dm, int align, int ratio) {
    __shared__ float red[8][2][128];
    const int t = blockIdx.x;
    if ((int64_t)t * align >= n_rows[0] || tile_expert[t / ratio] < 0) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int d = blockIdx.y * 128 + lane * 4;
    float gw[4] = {0.f, 0.f, 0.f, 0.f}, gb[4] = {0.f, 0.f, 0.f, 0.f};
    if (d < Dm) {
        for (int i = warp; i < align; i += 8) {
            const int r = t * align + i;
            const int tok = tok_of_row[r];
            if (tok < 0) continue;
            const float mean = stats[2 * (size_t)tok], rstd = stats[2 * (size_t)tok + 1];
#pragma unroll
            for (int v = 0; v < 4; ++v) {
                const float dv = ab_to_float(dxn[(size_t)r * Dm + d + v]);
                const float xh = (ab_to_float(x[(size_t)tok * Dm + d + v]) - mean) * rstd;
                gw[v] = fmaf(dv, xh, gw[v]);
                gb[v] += dv;
            }
        }
    }
#pragma unroll
    for (int v = 0; v < 4; ++v) { red[warp][0][lane * 4 + v] = gw[v]; red[warp][1][lane * 4 + v] = gb[v]; }
    __syncthreads();
    const int q = threadIdx.x >> 7, c = threadIdx.x & 127;      // 256 threads: (w|b) x 128 columns
    float s2 = 0.f;
#pragma unroll
    for (int wv = 0; wv < 8; ++wv) s2 += red[wv][q][c];
    const int dd = blockIdx.y * 128 + c;
    if (dd < Dm) part[((size_t)t * 2 + q) * Dm + dd] = s2;
}

// per-tile column sums: grid (tiles, ceil(C/256)); block (32 lanes x 8 columns, 8 warps over the rows)
template <typename T>
__global__ void __launch_bounds__(256) tile_colsum_kernel(const T* __restrict__ a, const int32_t* __restrict__ tile_expert,
                                                          const int32_t* __restrict__ n_rows, float* __restrict__ part, int C,
                                                          int align, int ratio) {
    __shared__ float red[8][256];
    const int t = blockIdx.x;
    if ((int64_t)t * align >= n_rows[0] || tile_expert[t / ratio] < 0) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c0 = blockIdx.y * 256 + lane * 8;
    float acc[8];
#pragma unroll
    for (int v = 0; v < 8; ++v) acc[v] = 0.f;
    if (c0 < C) {
        // 8 columns per thread as whole 16-byte vectors, 4 rows in flight
        constexpr int VN = 16 / (int)sizeof(T);          // elements per vector (8 bf16 / 4 fp32)
        for (int i0 = warp; i0 < align; i0 += 32) {
            uint4 q[4][8 / VN];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + u * 8;
                const uint4* row = reinterpret_cast<const uint4*>(a + ((size_t)t * align + i) * C + c0);
#pragma unroll
                for (int w = 0; w < 8 / VN; ++w) q[u][w] = i < align ? __ldg(row + w) : make_uint4(0u, 0u, 0u, 0u);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
#pragma unroll
                for (int w = 0; w < 8 / VN; ++w) {
                    float f[VN];
                    ab_vec16<T>::unpack(q[u][w], f);
#pragma unroll
                    for (int v = 0; v < VN; ++v) acc[w * VN + v] += f[v];
                }
            }
        }
    }
#pragma unroll
    for (int v = 0; v < 8; ++v) red[warp][lane * 8 + v] = acc[v];
    __syncthreads();
    const int c = threadIdx.x;
    float s2 = 0.f;
#pragma unroll
    for (int wv = 0; wv < 8; ++wv) s2 += red[wv][c];
    if (blockIdx.y * 256 + c < C) part[(size_t)t * C + blockIdx.y * 256 + c] = s2;
}

// out[e][j] = sum over the (contiguous) tiles of expert e of part[t][j], fixed order.  Columns [0, split) go to
// out_a [E][split], columns [split, ncols) to out_b [E][ncols-split].
__global__ void tile_reduce_kernel(const float* __restrict__ part, const int32_t* __restrict__ tile_expert,
                                   const int32_t* __restrict__ n_rows, float* __restrict__ out_a, float* __restrict__ out_b,
                                   int split, int ncols, int align, int ratio) {
    __shared__ int s_t0, s_t1;
    __shared__ int s_list[1024];                       // tile ids of this expert, in order (the common case fits)
    __shared__ int s_n;
    const int e = blockIdx.y;
    const int ntiles = n_rows[0] / align;
    if (threadIdx.x < 32) {                            // one warp builds the ordered list with ballots
        int n = 0, t0 = ntiles, t1 = 0;
        for (int base = 0; base < ntiles; base += 32) {
            const int t = base + (int)threadIdx.x;
            const bool mine = t < ntiles && tile_expert[t / ratio] == e;
            const unsigned m = __ballot_sync(0xffffffffu, mine);
            if (mine) {
                const int pos = n + __popc(m & ((1u << threadIdx.x) - 1u));
                if (pos < 1024) s_list[pos] = t;
            }
            if (m) { t0 = min(t0, base + __ffs(m) - 1); t1 = base + 32 - __clz(m); }
            n += __popc(m);
        }
        if (threadIdx.x == 0) { s_t0 = t0; s_t1 = t1; s_n = n; }
    }
    __syncthreads();
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= ncols) return;
    float s = 0.f;
    if (s_n <= 1024) {
        // loads of 8 tiles are issued before the 8 dependent adds; order = tile order -> deterministic
        for (int i0 = 0; i0 < s_n; i0 += 8) {
            float v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = i0 + u < s_n ? part[(size_t)s_list[i0 + u] * ncols + j] : 0.f;
#pragma unroll
            for (int u = 0; u < 8; ++u) s += v[u];
        }
    } else {
        for (int t = s_t0; t < s_t1; ++t)
            if (tile_expert[t / ratio] == e) s += part[(size_t)t * ncols + j];  // tiles of an expert may be interleaved (EP layout)
    }
    if (j < split) out_a[(size_t)e * split + j] = s;
    else out_b[(size_t)e * (ncols - split) + (j - split)] = s;
}

// The per-tile reduction kernels work on tiles of at most 128 rows whatever the GEMM's row tile is (more, smaller CTAs:
// these kernels are latency-bound streams); tile_expert is looked up through the ratio of the two.
int work_rows(int row_align) { return row_align % 128 == 0 ? 128 : row_align; }

int make_peers(PeerRows* pr, const uint64_t* peer_ptrs, int W, int rank, int64_t rows_per_peer) {
    memset(pr, 0, sizeof(*pr));
    if (peer_ptrs == nullptr) return AB_OK;
    AB_REQUIRE(W >= 1 && W <= AB_MAX_PEERS && rank >= 0 && rank < W && rows_per_peer > 0 && rows_per_peer < (1ll << 31),
               "ep: bad peer table (W=%d, rank=%d, rows_per_peer=%lld; at most %d ranks)", W, rank, (long long)rows_per_peer, AB_MAX_PEERS);
    for (int i = 0; i < W; ++i) {
        AB_REQUIRE(peer_ptrs[i] != 0 && peer_ptrs[i] % 16 == 0, "ep: peer buffer %d is null or not 16-byte aligned", i);
        pr->base[i] = reinterpret_cast<unsigned char*>(peer_ptrs[i]);
    }
    pr->n = W; pr->rows_per_peer = (int)rows_per_peer; pr->rank = rank;
    return AB_OK;
}

int rows_grid(int64_t max_rows) {
    const int64_t want = ab_ceil_div(max_rows, 8);
    const int64_t cap = (int64_t)ab_num_sms() * 8;
    return (int)(want < cap ? want : cap);
}

}  // namespace

extern "C" int64_t ab_moe_max_rows(int S, int K, int E, int cap, int row_align) {
    int64_t kept = (int64_t)S * K;
    if ((int64_t)E * cap < kept) kept = (int64_t)E * cap;
    return ab_round_up(kept + (int64_t)E * (row_align - 1), row_align);
}

namespace {
// plan workspace: row_local [S*K] | zeroed: histograms [4][E*K][256], tickets [8], any_select | sel [E*K] | cc [chunks][K][E][2]
struct PlanWs { size_t hist_off, zero_bytes, sel_off, cc_off, total; };
PlanWs plan_ws(int S, int K, int E) {
    PlanWs p;
    size_t o = ab_round_up((int64_t)S * K * sizeof(int32_t), 256);
    p.hist_off = o;
    p.zero_bytes = ab_round_up(((int64_t)4 * E * K * 256 + 16) * sizeof(int), 256);
    o += p.zero_bytes;
    p.sel_off = o; o += ab_round_up((int64_t)E * K * sizeof(PlanSel), 256);
    p.cc_off = o; o += ab_round_up(ab_ceil_div(S, PLAN_CHUNK) * K * 2 * E * (int64_t)sizeof(int), 256);
    p.total = o;
    return p;
}
}  // namespace

extern "C" size_t ab_moe_plan_workspace_bytes(int S, int K, int E) { return plan_ws(S, K, E).total; }

extern "C" int ab_moe_plan(const int32_t* idx, const float* w, const int32_t* active, int cap, int32_t* counts,
                           int32_t* seg_off, int32_t* row_of, int32_t* tok_of_row, int32_t* slot_of_row,
                           int32_t* tile_expert, int32_t* n_rows, void* ws, size_t ws_bytes, int S, int K, int E,
                           int row_align, int64_t max_rows, int fixed_seg, cudaStream_t stream) {
    AB_REQUIRE(S > 0 && K >= 1 && E >= 1 && E <= 32, "moe_plan: bad shape S=%d K=%d E=%d", S, K, E);
    if (fixed_seg > 0) {
        // with a capacity limit a segment must hold `cap` rows; without one (cap >= S) the caller sizes it from the counts
        // it has reduced over the ranks, and the kernel traps rather than overflow a segment
        AB_REQUIRE(fixed_seg % row_align == 0 && (cap >= S || fixed_seg >= cap) && max_rows == (int64_t)E * fixed_seg,
                   "moe_plan: fixed_seg (%d) must be a multiple of %d, >= cap, and max_rows == E*fixed_seg", fixed_seg, row_align);
    } else {
        AB_REQUIRE(row_align > 0 && max_rows % row_align == 0 && max_rows >= ab_moe_max_rows(S, K, E, cap < S ? cap : S, row_align),
                   "moe_plan: max_rows %lld too small or not a multiple of %d", (long long)max_rows, row_align);
    }
    const PlanWs pw = plan_ws(S, K, E);
    AB_REQUIRE(ws && ws_bytes >= pw.total, "moe_plan: workspace too small");
    unsigned char* w8 = (unsigned char*)ws;
    int32_t* row_local = (int32_t*)ws;
    int* ghist = (int*)(w8 + pw.hist_off);
    int* tickets = ghist + (size_t)4 * E * K * 256;            // [0..3] histogram passes
    int* any_select = tickets + 8;
    PlanSel* sel = (PlanSel*)(w8 + pw.sel_off);
    int* cc = (int*)(w8 + pw.cc_off);
    AB_CHECK_CUDA(cudaMemsetAsync(ghist, 0, pw.zero_bytes, stream));
    AB_CHECK_CUDA(cudaMemsetAsync(tok_of_row, 0xFF, (size_t)max_rows * sizeof(int32_t), stream));
    AB_CHECK_CUDA(cudaMemsetAsync(slot_of_row, 0xFF, (size_t)max_rows * sizeof(int32_t), stream));
    const dim3 hgrid((unsigned)ab_ceil_div(S, HIST_TOKENS), K), cgrid((unsigned)ab_ceil_div(S, PLAN_CHUNK), K);
    for (int pass = 3; pass >= 0; --pass) {
        plan_hist_kernel<<<hgrid, PLAN_THREADS, 0, stream>>>(idx, w, active, cap, pass, ghist + (size_t)(3 - pass) * E * K * 256, sel,
                                                             any_select, tickets + (3 - pass), counts, S, K, E);
        AB_LAUNCH_CHECK();
    }
    plan_chunk_count_kernel<<<cgrid, PLAN_THREADS, 0, stream>>>(idx, w, sel, cc, S, K, E);
    AB_LAUNCH_CHECK();
    plan_pos_kernel<<<cgrid, PLAN_THREADS, 0, stream>>>(idx, w, sel, cc, row_local, S, K, E);
    AB_LAUNCH_CHECK();
    const int64_t want = ab_ceil_div((int64_t)S * K, 256);
    const int grid = (int)(want < ab_num_sms() * 4 ? want : ab_num_sms() * 4);
    plan_finalize_kernel<<<grid, 256, 0, stream>>>(idx, counts, row_local, seg_off, row_of, tok_of_row, slot_of_row, tile_expert,
                                                   n_rows, S, K, E, row_align, max_rows, fixed_seg);
    AB_LAUNCH_CHECK();
    return AB_OK;
}

namespace {
int permute_ln_impl(const void* x, const float* stats, const float* ln_w, const float* ln_b, const int32_t* tok_of_row,
                    const int32_t* tile_expert, const int32_t* n_rows, void* xn, int Dm, int row_align, int64_t max_rows, int dtype,
                    int out_dtype, const PeerRows& pr, cudaStream_t stream) {
    AB_REQUIRE(Dm > 0 && Dm % 4 == 0, "moe_permute_ln: hidden size must be a multiple of 4");
    const int grid = rows_grid(max_rows);
#define AB_PLN(TI, TO) permute_ln_kernel<TI, TO><<<grid, 256, 0, stream>>>((const TI*)x, stats, ln_w, ln_b, tok_of_row, tile_expert, n_rows, (TO*)xn, Dm, row_align, pr)
    if (dtype == AB_F32 && out_dtype == AB_F32) AB_PLN(float, float);
    else if (dtype == AB_F32 && out_dtype == AB_BF16) AB_PLN(float, __nv_bfloat16);
    else if (dtype == AB_BF16 && out_dtype == AB_BF16) AB_PLN(__nv_bfloat16, __nv_bfloat16);
    else if (dtype == AB_BF16 && out_dtype == AB_F32) AB_PLN(__nv_bfloat16, float);
    else AB_REQUIRE(false, "moe_permute_ln: bad dtypes");
#undef AB_PLN
    AB_LAUNCH_CHECK();
    return AB_OK;
}
}  // namespace

extern "C" int ab_moe_permute_ln(const void* x, const float* stats, const float* ln_w, const float* ln_b,
                                 const int32_t* tok_of_row, const int32_t* tile_expert, const int32_t* n_rows, void* xn, int Dm,
                                 int row_align, int64_t max_rows, int dtype, int out_dtype, cudaStream_t stream) {
    PeerRows pr;
    make_peers(&pr, nullptr, 0, 0, 0);
    return permute_ln_impl(x, stats, ln_w, ln_b, tok_of_row, tile_expert, n_rows, xn, Dm, row_align, max_rows, dtype, out_dtype, pr, stream);
}

extern "C" int ab_ep_permute_ln(const void* x, const float* stats, const float* ln_w, const float* ln_b,
                                const int32_t* tok_of_row, const int32_t* tile_expert, const int32_t* n_rows,
                                const uint64_t* peer_xn, int W, int rank, int64_t rows_per_peer, int Dm, int row_align,
                                int64_t max_rows, int dtype, int out_dtype, cudaStream_t stream) {
    AB_REQUIRE(peer_xn != nullptr && max_rows == (int64_t)W * rows_per_peer, "ep_permute_ln: max_rows must equal W * rows_per_peer");
    PeerRows pr;
    if (int e = make_peers(&pr, peer_xn, W, rank, rows_per_peer)) return e;
    return permute_ln_impl(x, stats, ln_w, ln_b, tok_of_row, tile_expert, n_rows, nullptr, Dm, row_align, max_rows, dtype, out_dtype, pr, stream);
}

extern "C" int ab_moe_unpermute(const void* y, const int32_t* row_of, const float* w, const float* res, void* out, float drop_p,
                                const uint32_t* drop_seed, int S, int K, int Dm, int y_dtype, int out_dtype, cudaStream_t stream) {
    AB_REQUIRE(Dm > 0 && Dm % 4 == 0, "moe_unpermute: hidden size must be a multiple of 4");
    AB_REQUIRE(drop_p >= 0.f && drop_p < 1.f && (drop_p == 0.f || drop_seed), "moe_unpermute: dropout p must be in [0,1) and needs a seed when > 0");
    AB_REQUIRE(res == nullptr || ((uintptr_t)res % 16) == 0, "moe_unpermute: the residual must be 16-byte aligned fp32");
    const uint32_t thresh = (uint32_t)((double)drop_p * 4294967296.0);
    const float scale = drop_p > 0.f ? 1.0f / (1.0f - drop_p) : 1.0f;
    const uint32_t* sd = drop_p > 0.f ? drop_seed : nullptr;
    const int grid = rows_grid(S);
#define AB_UNP(TY, TO)                                                                                                          \
    {                                                                                                                            \
        if (K <= 2) unpermute_kernel<TY, TO, 2><<<grid, 256, 0, stream>>>((const TY*)y, row_of, w, res, (TO*)out, sd, thresh, scale, S, K, Dm); \
        else if (K <= 4) unpermute_kernel<TY, TO, 4><<<grid, 256, 0, stream>>>((const TY*)y, row_of, w, res, (TO*)out, sd, thresh, scale, S, K, Dm); \
        else unpermute_kernel<TY, TO, 8><<<grid, 256, 0, stream>>>((const TY*)y, row_of, w, res, (TO*)out, sd, thresh, scale, S, K, Dm); \
    }
    AB_REQUIRE(K >= 1 && K <= 8, "moe_unpermute: experts_per_token must be in [1, 8]");
    if (y_dtype == AB_F32 && out_dtype == AB_F32) AB_UNP(float, float)
    else if (y_dtype == AB_BF16 && out_dtype == AB_F32) AB_UNP(__nv_bfloat16, float)
    else if (y_dtype == AB_BF16 && out_dtype == AB_BF16) AB_UNP(__nv_bfloat16, __nv_bfloat16)
    else if (y_dtype == AB_F32 && out_dtype == AB_BF16) AB_UNP(float, __nv_bfloat16)
    else AB_REQUIRE(false, "moe_unpermute: bad dtypes");
#undef AB_UNP
    AB_LAUNCH_CHECK();
    return AB_OK;
}

namespace {
int unpermute_bwd_impl(const void* dout, const void* y, const float* w, const int32_t* tok_of_row, const int32_t* slot_of_row,
                       const int32_t* n_rows, void* dy, float* dw_row, float drop_p, const uint32_t* drop_seed, int K, int Dm,
                       int64_t max_rows, int dout_dtype, int y_dtype, int dy_dtype, const PeerRows& pr, cudaStream_t stream) {
    AB_REQUIRE(Dm > 0 && Dm % 4 == 0, "moe_unpermute_bwd: hidden size must be a multiple of 4");
    AB_REQUIRE(drop_p >= 0.f && drop_p < 1.f && (drop_p == 0.f || drop_seed), "moe_unpermute_bwd: dropout p must be in [0,1) and needs a seed when > 0");
    const uint32_t thresh = (uint32_t)((double)drop_p * 4294967296.0);
    const float scale = drop_p > 0.f ? 1.0f / (1.0f - drop_p) : 1.0f;
    const uint32_t* sd = drop_p > 0.f ? drop_seed : nullptr;
    const int grid = rows_grid(max_rows);
#define AB_UB(TD, TY, TO) unpermute_bwd_kernel<TD, TY, TO><<<grid, 256, 0, stream>>>((const TD*)dout, (const TY*)y, w, tok_of_row, slot_of_row, n_rows, (TO*)dy, dw_row, sd, thresh, scale, K, Dm, pr)
    const int key = dout_dtype * 4 + y_dtype * 2 + dy_dtype;
    switch (key) {
        case 0: AB_UB(float, float, float); break;
        case 1: AB_UB(float, float, __nv_bfloat16); break;
        case 2: AB_UB(float, __nv_bfloat16, float); break;
        case 3: AB_UB(float, __nv_bfloat16, __nv_bfloat16); break;
        case 4: AB_UB(__nv_bfloat16, float, float); break;
        case 5: AB_UB(__nv_bfloat16, float, __nv_bfloat16); break;
        case 6: AB_UB(__nv_bfloat16, __nv_bfloat16, float); break;
        case 7: AB_UB(__nv_bfloat16, __nv_bfloat16, __nv_bfloat16); break;
        default: AB_REQUIRE(false, "moe_unpermute_bwd: bad dtypes");
    }
#undef AB_UB
    AB_LAUNCH_CHECK();
    return AB_OK;
}
}  // namespace

extern "C" int ab_moe_unpermute_bwd(const void* dout, const void* y, const float* w, const int32_t* tok_of_row,
                                    const int32_t* slot_of_row, const int32_t* n_rows, void* dy, float* dw_row, float drop_p,
                                    const uint32_t* drop_seed, int K, int Dm, int64_t max_rows, int dout_dtype, int y_dtype,
                                    int dy_dtype, cudaStream_t stream) {
    PeerRows pr;
    make_peers(&pr, nullptr, 0, 0, 0);
    return unpermute_bwd_impl(dout, y, w, tok_of_row, slot_of_row, n_rows, dy, dw_row, drop_p, drop_seed, K, Dm, max_rows, dout_dtype,
                              y_dtype, dy_dtype, pr, stream);
}

extern "C" int ab_ep_unpermute_bwd(const void* dout, const void* y, const float* w, const int32_t* tok_of_row,
                                   const int32_t* slot_of_row, const int32_t* n_rows, const uint64_t* peer_dy, int W, int rank,
                                   int64_t rows_per_peer, float* dw_row, float drop_p, const uint32_t* drop_seed, int K, int Dm,
                                   int64_t max_rows, int dout_dtype, int y_dtype, int dy_dtype, cudaStream_t stream) {
    AB_REQUIRE(peer_dy != nullptr && max_rows == (int64_t)W * rows_per_peer, "ep_unpermute_bwd: max_rows must equal W * rows_per_peer");
    PeerRows pr;
    if (int e = make_peers(&pr, peer_dy, W, rank, rows_per_peer)) return e;
    return unpermute_bwd_impl(dout, y, w, tok_of_row, slot_of_row, n_rows, nullptr, dw_row, drop_p, drop_seed, K, Dm, max_rows,
                              dout_dtype, y_dtype, dy_dtype, pr, stream);
}

extern "C" size_t ab_moe_permute_ln_bwd_workspace_bytes(int Dm, int row_align, int64_t max_rows) {
    return (size_t)ab_round_up((max_rows / work_rows(row_align)) * 2 * (int64_t)Dm * sizeof(float), 256);
}

extern "C" int ab_moe_permute_ln_bwd(const void* dxn, const void* x, const float* stats, const float* ln_w,
                                     const int32_t* tok_of_row, const int32_t* tile_expert, const int32_t* n_rows, float* dxrow,
                                     float* dln_w, float* dln_b, void* ws, size_t ws_bytes, int Dm, int E, int row_align,
                                     int64_t max_rows, int dtype, int dxn_dtype, cudaStream_t stream) {
    AB_REQUIRE(ws && ws_bytes >= ab_moe_permute_ln_bwd_workspace_bytes(Dm, row_align, max_rows), "moe_permute_ln_bwd: workspace too small");
    AB_REQUIRE(Dm % 4 == 0, "moe_permute_ln_bwd: hidden size must be a multiple of 4");
    const int sub = work_rows(row_align), ratio = row_align / sub;
    const int ntiles = (int)(max_rows / sub);
    float* part = (float*)ws;
    const int rgrid = rows_grid(max_rows);
    dim3 cgrid(ntiles, (unsigned)ab_ceil_div(Dm, 128));
    const int nit = (int)ab_ceil_div(Dm, 128);
#define AB_LNB_F(TX, TG, NIT)                                                                                                    \
    permute_ln_bwd_fused_kernel<TX, TG, NIT><<<ntiles, 256, 0, stream>>>((const TG*)dxn, (const TX*)x, stats, ln_w, tok_of_row, \
                                                                         tile_expert, n_rows, dxrow, part, Dm, sub, ratio)
#define AB_LNB(TX, TG)                                                                                                           \
    {                                                                                                                            \
        if (nit <= 8) {                                                                                                          \
            if (nit <= 2) AB_LNB_F(TX, TG, 2); else if (nit <= 4) AB_LNB_F(TX, TG, 4);                                           \
            else if (nit <= 6) AB_LNB_F(TX, TG, 6); else AB_LNB_F(TX, TG, 8);                                                    \
        } else {                                                                                                                 \
            permute_ln_bwd_rows_kernel<TX, TG><<<rgrid, 256, 0, stream>>>((const TG*)dxn, (const TX*)x, stats, ln_w, tok_of_row, \
                                                                          tile_expert, n_rows, dxrow, Dm, row_align);            \
            permute_ln_bwd_cols_kernel<TX, TG><<<cgrid, 256, 0, stream>>>((const TG*)dxn, (const TX*)x, stats, tok_of_row,       \
                                                                          tile_expert, n_rows, part, Dm, sub, ratio);            \
        }                                                                                                                        \
    }
    if (dtype == AB_F32 && dxn_dtype == AB_F32) AB_LNB(float, float)
    else if (dtype == AB_F32 && dxn_dtype == AB_BF16) AB_LNB(float, __nv_bfloat16)
    else if (dtype == AB_BF16 && dxn_dtype == AB_BF16) AB_LNB(__nv_bfloat16, __nv_bfloat16)
    else if (dtype == AB_BF16 && dxn_dtype == AB_F32) AB_LNB(__nv_bfloat16, float)
    else AB_REQUIRE(false, "moe_permute_ln_bwd: bad dtypes");
#undef AB_LNB
#undef AB_LNB_F
    AB_LAUNCH_CHECK();
    dim3 grid((unsigned)ab_ceil_div(2 * Dm, 128), E);       // part is [tile][2][Dm]: reduce as 2*Dm columns, split in two
    tile_reduce_kernel<<<grid, 128, 0, stream>>>(part, tile_expert, n_rows, dln_w, dln_b, Dm, 2 * Dm, sub, ratio);
    AB_LAUNCH_CHECK();
    return AB_OK;
}

extern "C" size_t ab_moe_segment_colsum_workspace_bytes(int C, int row_align, int64_t max_rows) {
    return (size_t)ab_round_up((max_rows / work_rows(row_align)) * (int64_t)C * sizeof(float), 256);
}

extern "C" int ab_moe_segment_colsum(const void* a, const int32_t* tile_expert, const int32_t* n_rows, float* out, void* ws,
                                     size_t ws_bytes, int C, int E, int row_align, int64_t max_rows, int dtype,
                                     cudaStream_t stream) {
    AB_REQUIRE(ws && ws_bytes >= ab_moe_segment_colsum_workspace_bytes(C, row_align, max_rows), "moe_segment_colsum: workspace too small");
    const int sub = work_rows(row_align), ratio = row_align / sub;
    const int ntiles = (int)(max_rows / sub);
    float* part = (float*)ws;
    AB_REQUIRE(C % 8 == 0 && ((uintptr_t)a % 16) == 0, "moe_segment_colsum: column count must be a multiple of 8 and the matrix 16-byte aligned");
    dim3 cgrid(ntiles, (unsigned)ab_ceil_div(C, 256));
    if (dtype == AB_F32) tile_colsum_kernel<float><<<cgrid, 256, 0, stream>>>((const float*)a, tile_expert, n_rows, part, C, sub, ratio);
    else tile_colsum_kernel<__nv_bfloat16><<<cgrid, 256, 0, stream>>>((const __nv_bfloat16*)a, tile_expert, n_rows, part, C, sub, ratio);
    AB_LAUNCH_CHECK();
    dim3 grid((unsigned)ab_ceil_div(C, 128), E);
    tile_reduce_kernel<<<grid, 128, 0, stream>>>(part, tile_expert, n_rows, out, nullptr, C, C, sub, ratio);
    AB_LAUNCH_CHECK();
    return AB_OK;
}
