// Selective scan of the Apertis SSM layer (core.py:324-353 scans, :383 softplus, :394-396 skip + gate), forward and
// backward, as ONE persistent kernel each: "rounds" schedule.
//
// The recurrence  h_t = abar_t * h_{t-1} + B_t  (abar = exp(-exp(A_log) * softplus(dt)), one chain per channel) has only
// B * Di independent chains, so the sequence is cut into chunks of Tc tokens.  A warp owns one chunk of one 64-channel
// slab of one sequence at a time: a lane owns two adjacent channels (packed f32x2 arithmetic) and walks the chunk's
// tokens serially.  Up to four warps working on neighbouring slabs of the same chunk form a TEAM that shares its operand
// tiles: one lane issues TMA loads of [8 tokens x (team slabs * 64) channels] boxes into a two-stage ring in shared
// memory (rows / channels past the tensor are zero-filled by the hardware, which is exactly the masking the recurrences
// need), the warps read their slab with immediate offsets, write the results IN PLACE over the consumed operands, and the
// same lane issues the TMA stores (which clip what lies past the tensor).  The token loops hold no address arithmetic,
// predicates or bounds checks.
//
// Every chunk is visited twice:
//   P1  reads only dt and B (forward) / C, z, dout (backward), computes delta = softplus(dt) (32 lanes = 8 tokens x 4 heads,
//       distributed by shuffles, saved for the second visit and for the backward) and the chunk aggregate (P = prod abar,
//       S = state the chunk produces from 0), publishes it;
//   P2  streams the chunk once with the state entering it known: h, y = (C*h + D*x) * silu(z)  (backward: forward
//       recompute of 8 states from the saved checkpoint, reverse sweep, all gradients).
// The persistent grid works in rounds: in round r team g handles chunk r * cpr + g / nteamchains of team-chain
// g % nteamchains, and the order per warp is P1(0), P1(1), P2(0), P1(2), P2(1), ...: the aggregates of round r are
// published a whole P1 pass before anybody needs their prefix.  The prefix over a round's chunk aggregates is a two-level
// scan done by whoever arrives last (segments of 32 chunks, then the segment totals chained to the carry of the previous
// round): fixed association, bitwise reproducible.  All counters / flags are indexed by round and zeroed by a memset node
// ahead of the launch (graph capture safe); waits are bounded (4 s) and trap, so a protocol error is a CUDA error, never a
// silent wrong answer.
//
// The forward saves the state entering every group of 8 tokens (hck, fp32, +0.5 B per element) so that the backward
// needs no forward prefix of its own and recomputes states 8 at a time in registers.
#include <mutex>

#include "common.cuh"

namespace {

// sigmoid of a channel pair.  bf16 activations: single-MUFU tanh form (relative error ~5e-4, below bf16 resolution);
// fp32 activations: ex2 + rcp
template <typename T>
__device__ __forceinline__ f2 f2_sigmoid(f2 z) {
    if constexpr (sizeof(T) == 2) {
        float a, b, ta, tb;
        f2_unpack(f2_mul(z, f2_bcast(0.5f)), a, b);
        asm("tanh.approx.f32 %0, %1;" : "=f"(ta) : "f"(a));
        asm("tanh.approx.f32 %0, %1;" : "=f"(tb) : "f"(b));
        return f2_fma(f2_pack(ta, tb), f2_bcast(0.5f), f2_bcast(0.5f));
    } else {
        float a, b;
        f2_unpack(z, a, b);
        return f2_pack(ab_sigmoid(a), ab_sigmoid(b));
    }
}

// ---- channel pairs in registers / shared memory ----------------------------------------------------------------------
template <typename T> struct Raw;
template <> struct Raw<__nv_bfloat16> { typedef uint32_t type; };
template <> struct Raw<float> { typedef f2 type; };

__device__ __forceinline__ f2 up(uint32_t r) { return f2_pack(__uint_as_float(r << 16), __uint_as_float(r & 0xffff0000u)); }
__device__ __forceinline__ f2 up(f2 r) { return r; }
template <typename T> __device__ __forceinline__ typename Raw<T>::type down(f2 v);
template <> __device__ __forceinline__ uint32_t down<__nv_bfloat16>(f2 v) {
    float a, b;
    f2_unpack(v, a, b);
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
    return r;
}
template <> __device__ __forceinline__ f2 down<float>(f2 v) { return v; }

// ---- TMA: 3-D tiled loads / stores of [channels, tokens, batch] boxes with an L2 eviction policy -------------------------
__device__ __forceinline__ uint64_t policy_evict_last() { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p)); return p; }
__device__ __forceinline__ uint64_t policy_evict_first() { uint64_t p; asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p)); return p; }

__device__ __forceinline__ void tma_load(uint32_t dst, const CUtensorMap* m, uint32_t bar, int c, int t, int b, uint64_t pol) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;"
        ::"r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar), "r"(c), "r"(t), "r"(b), "l"(pol) : "memory");
}
__device__ __forceinline__ void tma_store(const CUtensorMap* m, uint32_t src, int c, int t, int b, uint64_t pol) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group.L2::cache_hint [%0, {%2, %3, %4}], [%1], %5;"
                 ::"l"(reinterpret_cast<uint64_t>(m)), "r"(src), "r"(c), "r"(t), "r"(b), "l"(pol) : "memory");
}
__device__ __forceinline__ void mbar_init_u32(uint32_t bar, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx_u32(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait_u32(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    } while (!ok);
}

__device__ __forceinline__ unsigned long long globaltimer_ns() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }

constexpr int RG = 8;                 // tokens per group: spacing of the saved states, unit of the delta shuffles
constexpr int RSEG = 32;              // chunks per level-1 segment of a round's prefix
constexpr unsigned long long WAIT_LIMIT_NS = 4000000000ull;

struct RoundsParams {
    int B, L, Di, H, nslab, nchains;
    int Tc, nck, cpr, nrounds, nseg, nw_used, nck8, L8;
    int tps, nteamchains;      // teams per sequence, B * tps
    const void *xa, *dlog, *Bm, *Cm, *z, *dout, *dyssm;
    void *y, *yssm, *dxa, *dBm, *dCm, *dz, *ddlog;
    int xa_stride, dlog_stride, bc_stride, z_stride, y_stride, dbc_stride, dz_stride, dxa_stride, ddlog_stride;   // elements (< 2^30, checked on the host)
    const float *dt_bias, *A_log, *D, *h0;
    float* h_last;
    float* hck;        // [B, nck8, Di]     state entering every group of 8 tokens
    float* delta;      // [B, nslab, L8, 4] softplus(dt) of the slab's HPS <= 4 heads (unused slots hold 0)
    float4* agg;       // [2][nchains][cpr][32]   chunk aggregate (P0, P1, S0, S1) per lane; level 1 rewrites it as the exclusive prefix inside the segment
    float4* segagg;    // [2][nchains][nseg][32]
    float2* segcarry;  // [2][nchains][nseg][32]  state entering each segment
    float2* carry;     // [nchains][32]           state at the end of the last prefixed round
    unsigned* cnt1;    // [nrounds][nchains][nseg]
    unsigned* cnt2;    // [nrounds][nchains]
    unsigned* flag;    // [nrounds][nchains]
    unsigned* done;    // teams that have finished; the last one zeroes the counters for the next launch
    int cnt_words, nteams_used;
    float4* part;      // backward: [nw_used][32]  (dA0, dA1, dD0, dD1) accumulated by each warp over its chunks
    float* part_b;     // backward: [nw_used][32]  d dt_bias share of lane (head lane / (32 / HPS), token lane & 7); zero in
                       //           the lanes of a head past its first 8
    int ddlog_cols;    // backward: columns [H, ddlog_cols) of the d dlog rows are written as zero (padding of a fused buffer)
};

__device__ __forceinline__ void wait_flag(const unsigned* f, int lane) {
    if (lane == 0) {
        unsigned v;
        unsigned long long t0 = 0;
        for (int it = 0;; ++it) {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
            if (v != 0u) break;
            if (it >= 32) {
                __nanosleep(100);
                if (t0 == 0) t0 = globaltimer_ns();
                else if (globaltimer_ns() - t0 > WAIT_LIMIT_NS) {
                    __trap();          // protocol error: surfaces as a CUDA error at the next synchronisation, never as a wrong answer
                }
            }
        }
    }
    __syncwarp();
}

// Publishes this warp's chunk aggregate and, when it is the last of its segment / of the round, runs the level-1 /
// level-2 prefix.  `init` = state entering the chain (forward: h0; backward: 0), used by round 0.
__device__ __forceinline__ void publish_and_prefix(const RoundsParams& p, int r, int chain, int slot, int n_r, int lane, f2 P, f2 S, f2 init,
                                                   float* final_out /* this lane's pair of the chain's final state, or null */) {
    const int par = r & 1;
    const int seg = slot / RSEG;
    const int nseg_r = (n_r + RSEG - 1) / RSEG;
    float4* agg = p.agg + ((size_t)(par * p.nchains + chain) * p.cpr) * 32;
    {
        float p0, p1, s0, s1;
        f2_unpack(P, p0, p1);
        f2_unpack(S, s0, s1);
        __stcg(&agg[(size_t)slot * 32 + lane], make_float4(p0, p1, s0, s1));
    }
    __syncwarp();
    unsigned last1 = 0;
    if (lane == 0) {
        __threadfence();
        const int n_in_seg = min(RSEG, n_r - seg * RSEG);
        const unsigned old = atomicAdd(&p.cnt1[((size_t)r * p.nchains + chain) * p.nseg + seg], 1u);
        last1 = (old == (unsigned)(n_in_seg - 1));
        if (last1) __threadfence();
    }
    last1 = __shfl_sync(0xffffffffu, last1, 0);
    if (!last1) return;
    // ---- level 1: exclusive prefixes inside the segment, segment total (loads in batches of 8: each is an L2 round trip)
    f2 Pex = f2_bcast(1.f), Sex = f2_bcast(0.f);
    {
        const int n_in_seg = min(RSEG, n_r - seg * RSEG);
        float4* a = agg + (size_t)(seg * RSEG) * 32 + lane;
        for (int j0 = 0; j0 < n_in_seg; j0 += 8) {
            float4 v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) v[u] = (j0 + u < n_in_seg) ? __ldcg(a + (size_t)(j0 + u) * 32) : make_float4(1.f, 1.f, 0.f, 0.f);
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                if (j0 + u < n_in_seg) {
                    float e0, e1, g0, g1;
                    f2_unpack(Pex, e0, e1);
                    f2_unpack(Sex, g0, g1);
                    __stcg(a + (size_t)(j0 + u) * 32, make_float4(e0, e1, g0, g1));
                    const f2 vp = f2_pack(v[u].x, v[u].y), vs = f2_pack(v[u].z, v[u].w);
                    Sex = f2_fma(vp, Sex, vs);
                    Pex = f2_mul(Pex, vp);
                }
            }
        }
    }
    float4* segagg = p.segagg + ((size_t)(par * p.nchains + chain) * p.nseg) * 32;
    {
        float e0, e1, g0, g1;
        f2_unpack(Pex, e0, e1);
        f2_unpack(Sex, g0, g1);
        __stcg(&segagg[(size_t)seg * 32 + lane], make_float4(e0, e1, g0, g1));
    }
    __syncwarp();
    unsigned last2 = 0;
    if (lane == 0) {
        __threadfence();
        const unsigned old = atomicAdd(&p.cnt2[(size_t)r * p.nchains + chain], 1u);
        last2 = (old == (unsigned)(nseg_r - 1));
        if (last2) __threadfence();
    }
    last2 = __shfl_sync(0xffffffffu, last2, 0);
    if (!last2) return;
    // ---- level 2: chain the segment totals to the carry of the previous round
    f2 h = init;
    if (r > 0) {
        wait_flag(&p.flag[(size_t)(r - 1) * p.nchains + chain], lane);
        const float2 c = __ldcg(&p.carry[(size_t)chain * 32 + lane]);
        h = f2_pack(c.x, c.y);
    }
    float2* segcarry = p.segcarry + ((size_t)(par * p.nchains + chain) * p.nseg) * 32;
    for (int s0 = 0; s0 < nseg_r; s0 += 8) {
        float4 v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = (s0 + u < nseg_r) ? __ldcg(&segagg[(size_t)(s0 + u) * 32 + lane]) : make_float4(1.f, 1.f, 0.f, 0.f);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            if (s0 + u < nseg_r) {
                float h0, h1;
                f2_unpack(h, h0, h1);
                __stcg(&segcarry[(size_t)(s0 + u) * 32 + lane], make_float2(h0, h1));
                h = f2_fma(f2_pack(v[u].x, v[u].y), h, f2_pack(v[u].z, v[u].w));
            }
        }
    }
    {
        float h0, h1;
        f2_unpack(h, h0, h1);
        __stcg(&p.carry[(size_t)chain * 32 + lane], make_float2(h0, h1));
        if (final_out != nullptr && r == p.nrounds - 1) { final_out[0] = h0; final_out[1] = h1; }
    }
    __syncwarp();
    if (lane == 0) {
        __threadfence();
        asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(&p.flag[(size_t)r * p.nchains + chain]), "r"(1u) : "memory");
    }
}

// state entering chunk `slot` of round r (after wait_flag)
__device__ __forceinline__ f2 incoming_state(const RoundsParams& p, int r, int chain, int slot, int lane) {
    const int par = r & 1;
    const float4 ex = __ldcg(&p.agg[((size_t)(par * p.nchains + chain) * p.cpr + slot) * 32 + lane]);
    const float2 sc = __ldcg(&p.segcarry[((size_t)(par * p.nchains + chain) * p.nseg + slot / RSEG) * 32 + lane]);
    return f2_fma(f2_pack(ex.x, ex.y), f2_pack(sc.x, sc.y), f2_pack(ex.z, ex.w));
}

// ====================================================================================================================
// team TMA pipeline
//   A team's work is one stream of ITEMS: P1 of round 0, P1 of round 1, P2 of round 0, P1 of round 2, ... each phase cut
//   into items of one ring stage (forward P1: 32 tokens of B; everything else: 8 tokens of every operand of the phase).
//   The team leader issues the loads of item k - 1 + NST while item k is being computed, ACROSS phase boundaries (the
//   addresses of a phase do not depend on the prefix it waits for), so the ring never drains and a visit of a chunk
//   costs no cold start.  Results are written in place over the consumed operands and stored by TMA from the stage.
// ====================================================================================================================
template <typename T, int TS> struct Tile {
    static constexpr int ROW_RAW = TS * 32;                          // row pitch in channel pairs
    static constexpr int BYTES = RG * TS * 64 * (int)sizeof(T);      // one operand of one group of 8 tokens
};

struct Pipe {
    unsigned char* base;     // generic address of stage 0 + this lane's channel pair
    uint32_t sbase;          // shared-space address of stage 0
    uint32_t bar;            // shared-space address of mbarrier 0
    uint32_t phases;         // bit s: parity the next wait on stage s expects
    uint32_t stage_bytes;
    int k;                   // items consumed so far (item k lives in stage k % NST)
    __device__ __forceinline__ uint32_t saddr(int st, int off) const { return sbase + (uint32_t)st * stage_bytes + (uint32_t)off; }
    __device__ __forceinline__ unsigned char* gaddr(int st) const { return base + (size_t)st * stage_bytes; }
    __device__ __forceinline__ uint32_t baddr(int st) const { return bar + 8u * (uint32_t)st; }
    __device__ __forceinline__ void wait(int st) {
        mbar_wait_u32(baddr(st), (phases >> st) & 1u);
        phases ^= 1u << st;
    }
};
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
template <int TS> __device__ __forceinline__ void team_sync(int team_in_cta) {
    if (TS == 1) __syncwarp();
    else asm volatile("bar.sync %0, %1;" ::"r"(team_in_cta + 1), "n"(TS * 32) : "memory");
}

// `stage` already points at this lane's channel pair of row 0 of operand 0
template <typename T, int TS>
__device__ __forceinline__ typename Raw<T>::type lds_pair(const unsigned char* stage, int arr, int row) {
    return reinterpret_cast<const typename Raw<T>::type*>(stage)[(arr * RG + row) * Tile<T, TS>::ROW_RAW];
}
template <typename T, int TS>
__device__ __forceinline__ void sts_pair(unsigned char* stage, int arr, int row, f2 v) {
    reinterpret_cast<typename Raw<T>::type*>(stage)[(arr * RG + row) * Tile<T, TS>::ROW_RAW] = down<T>(v);
}

// what a warp knows about its place
struct Who {
    int lane, member, team_in_cta;     // member: slab inside the team (the team's lane 0 of member 0 drives TMA)
    int b, ch0_team, slab, chain, slot;
    bool real, leader, cv;             // real: the slab exists (teams are padded to TS slabs); cv: this lane's channel pair exists
};

constexpr int P1_ROWS = 4 * RG;       // forward P1 reads B in pieces of 32 tokens (one stage = 4 operand tiles = 32 rows)

// Walks a team's phases in execution order: P1(0), then for r = 0 .. R-1: P1(r+1) (if any), P2(r).  Used twice per team:
// by every warp to run the phases, and by the leader, NST items ahead, to issue their loads.
template <bool BWD>
struct Cursor {
    int ph, kind, r, i, n, t0, tend, n_r;      // kind: 0 = P1, 1 = P2, -1 = end;  item i of n in chunk [t0, tend)
    __device__ __forceinline__ void begin(const RoundsParams& p, int slot) { ph = -1; kind = 0; next_phase(p, slot); }
    __device__ __forceinline__ void next_phase(const RoundsParams& p, int slot) {
        for (;;) {
            ++ph;
            if (ph == 0) { kind = 0; r = 0; }
            else {
                const int q = (ph - 1) >> 1;
                if (q >= p.nrounds) { kind = -1; n = 0; i = 0; return; }
                if ((ph - 1) & 1) { kind = 1; r = q; }
                else { kind = 0; r = q + 1; if (r >= p.nrounds) continue; }
            }
            n_r = min(p.cpr, p.nck - r * p.cpr);
            if (slot >= n_r) continue;                       // the last round may not reach this team
            const int pos = BWD ? p.nck - 1 - (r * p.cpr + slot) : r * p.cpr + slot;
            t0 = pos * p.Tc;
            tend = min(t0 + p.Tc, p.L);
            const int rows = (!BWD && kind == 0) ? P1_ROWS : RG;
            n = (tend - t0 + rows - 1) / rows;
            i = 0;
            if (n > 0) return;
        }
    }
    // first token of item i (the backward walks a chunk's groups last to first)
    __device__ __forceinline__ int token() const {
        if (BWD) return t0 + (n - 1 - i) * RG;
        return t0 + i * (kind == 0 ? P1_ROWS : RG);
    }
    __device__ __forceinline__ void advance(const RoundsParams& p, int slot) { if (++i >= n) next_phase(p, slot); }
};


// A team that has run all its phases signs off; the last one zeroes every counter / flag of this launch, so the next launch
// on the workspace starts clean without a memset node (the workspace is zero-filled once, when it is allocated).
__device__ __forceinline__ void team_finish(const RoundsParams& p, int member, int lane) {
    if (member != 0) return;
    unsigned last = 0;
    if (lane == 0) {
        __threadfence();
        last = atomicAdd(p.done, 1u) == (unsigned)(p.nteams_used - 1);
        if (last) __threadfence();
    }
    last = __shfl_sync(0xffffffffu, last, 0);
    if (!last) return;
    for (int i = lane; i < p.cnt_words; i += 32) p.cnt1[i] = 0u;
    if (lane == 0) *p.done = 0u;
}

// ====================================================================================================================
// forward
// ====================================================================================================================
template <typename T>
struct FwdCtx {
    const T* dlog;     // this lane's (token lane >> 2, head slot lane & 3) column of row 0 of the sequence
    float* delta;      // this (sequence, slab)'s [L8, 4] block + head slot (lane & 3)
    float* hck;        // this sequence's [nck8, Di] block + channel pair
    f2 A2, Dv;
    float bias;        // dt bias of the head this lane computes delta for
    bool hv;           // head slot (lane & 3) holds a head: slot < HPS and head < H
    int L;
};

// operand tiles of a forward P2 stage
constexpr int FA_B = 0, FA_X = 1, FA_C = 2, FA_Z = 3;

struct FwdMaps {
    const CUtensorMap *xa, *b, *b32, *c, *z, *y, *ys;
};

template <typename T, int TS, int NST>
struct FwdFeeder {
    const RoundsParams& p;
    const Who& w;
    Pipe& pp;
    const FwdMaps& m;
    Cursor<false> cur;
    uint64_t pol_keep, pol_stream;
    __device__ __forceinline__ FwdFeeder(const RoundsParams& p_, const Who& w_, Pipe& pp_, const FwdMaps& m_, uint64_t pk, uint64_t ps)
        : p(p_), w(w_), pp(pp_), m(m_), pol_keep(pk), pol_stream(ps) {}
    __device__ __forceinline__ void issue_one(int st) {
        if (cur.kind < 0) return;
        constexpr int TB = Tile<T, TS>::BYTES;
        const int t = cur.token();
        mbar_expect_tx_u32(pp.baddr(st), 4 * TB);
        if (cur.kind == 0) {
            tma_load(pp.saddr(st, 0), m.b32, pp.baddr(st), w.ch0_team, t, w.b, pol_keep);
        } else {
            tma_load(pp.saddr(st, FA_B * TB), m.b, pp.baddr(st), w.ch0_team, t, w.b, pol_stream);
            tma_load(pp.saddr(st, FA_X * TB), m.xa, pp.baddr(st), w.ch0_team, t, w.b, pol_stream);
            tma_load(pp.saddr(st, FA_C * TB), m.c, pp.baddr(st), w.ch0_team, t, w.b, pol_stream);
            tma_load(pp.saddr(st, FA_Z * TB), m.z, pp.baddr(st), w.ch0_team, t, w.b, pol_stream);
        }
        cur.advance(p, w.slot);
    }
    __device__ __forceinline__ void prime() {
        cur.begin(p, w.slot);
#pragma unroll
        for (int i = 0; i < NST; ++i) issue_one(i);
    }
    // called by the leader while item k (k >= 1) is being computed: the stage of item k - 1 (consumed, its stores issued
    // when it finished) takes item k - 1 + NST
    __device__ __forceinline__ void refill(int k) {
        if (k < 1) return;
        bulk_wait_read<0>();
        issue_one((k - 1) % NST);
    }
};

template <typename T>
__device__ __forceinline__ float dlog_fetch(const FwdCtx<T>& c, const Who& w, int dls, int tb, int tend) {
    const int tok = tb + (w.lane >> 2);
    return (w.real && c.hv && tb < tend && tok < c.L) ? ab_to_float(c.dlog[(int64_t)tok * dls]) : -1e30f;
}
// delta of 8 tokens x 4 head slots, one (token, slot) per lane; saved for P2 and the backward
template <typename T>
__device__ __forceinline__ float delta_finish(const FwdCtx<T>& c, const Who& w, float raw, int tb, int tend) {
    const float d = raw > -1e29f ? ab_softplus_fast(raw + c.bias) : 0.f;
    if (w.real && tb < tend) c.delta[(int64_t)(tb + (w.lane >> 2)) * 4] = d;        // rows < L8 always (tb < L, tb a multiple of 8)
    return d;
}

template <typename T, int TS, int NST, int HPS, typename Feeder>
__device__ __forceinline__ void fwd_p1(const RoundsParams& p, const FwdCtx<T>& c, const Who& w, Pipe& pp, Feeder& fd, const Cursor<false>& ph, f2 init) {
    const int t0 = ph.t0, tend = ph.tend, npieces = ph.n;
    const int dls = p.dlog_stride;
    const int hsel = w.lane / (32 / HPS);
    f2 S = f2_bcast(0.f);
    float sumd = 0.f;
    float raw[4];
#pragma unroll
    for (int g = 0; g < 4; ++g) raw[g] = dlog_fetch<T>(c, w, dls, t0 + g * RG, tend);
    for (int pc = 0; pc < npieces; ++pc) {
        const int st = pp.k % NST;
        const int tp = t0 + pc * P1_ROWS;
        float dm[4];
#pragma unroll
        for (int g = 0; g < 4; ++g) dm[g] = delta_finish<T>(c, w, raw[g], tp + g * RG, tend);
#pragma unroll
        for (int g = 0; g < 4; ++g) raw[g] = dlog_fetch<T>(c, w, dls, tp + P1_ROWS + g * RG, tend);     // next piece: in flight during this one
        pp.wait(st);
        if (w.leader) fd.refill(pp.k);
        const unsigned char* sb = pp.gaddr(st);
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            if (tp + g * RG < tend) {
#pragma unroll
                for (int j = 0; j < RG; ++j) {
                    const float d = __shfl_sync(0xffffffffu, dm[g], j * 4 + hsel);
                    const f2 a = f2_ex2(f2_mul(f2_bcast(d), c.A2));
                    S = f2_fma(a, S, up(lds_pair<T, TS>(sb, g, j)));
                    sumd += d;
                }
            }
        }
        team_sync<TS>(w.team_in_cta);
        ++pp.k;
    }
    if (!w.real) return;
    const f2 P = f2_ex2(f2_mul(f2_bcast(sumd), c.A2));
    float* fin = (p.h_last != nullptr && w.cv) ? p.h_last + (size_t)w.b * p.Di + w.slab * 64 + 2 * w.lane : nullptr;
    publish_and_prefix(p, ph.r, w.chain, w.slot, ph.n_r, w.lane, P, S, init, fin);
}

template <typename T, bool YSSM, int TS, int NST, int HPS, typename Feeder>
__device__ __forceinline__ void fwd_p2(const RoundsParams& p, const FwdCtx<T>& c, const Who& w, Pipe& pp, Feeder& fd, const FwdMaps& m,
                                       const Cursor<false>& ph, uint64_t pol_stream) {
    const int t0 = ph.t0, ngroups = ph.n, r = ph.r;
    const int hsel = w.lane / (32 / HPS);
    constexpr int TB = Tile<T, TS>::BYTES;
    const float* dsrc = c.delta + (int64_t)(t0 + (w.lane >> 2)) * 4;
    float dnext = w.real ? __ldcg(dsrc) : 0.f;
    f2 h = f2_bcast(0.f);
    if (w.real) {
        wait_flag(&p.flag[(size_t)r * p.nchains + w.chain], w.lane);
        h = incoming_state(p, r, w.chain, w.slot, w.lane);
    }
    float* hck = c.hck + (size_t)(t0 >> 3) * p.Di;
    for (int g = 0; g < ngroups; ++g) {
        const int st = pp.k % NST;
        const int tb = t0 + g * RG;
        const float dmine = dnext;
        dsrc += RG * 4;
        if (w.real && g + 1 < ngroups) dnext = __ldcg(dsrc);          // next group's delta: in flight during this group
        if (w.cv) {
            float h0, h1;
            f2_unpack(h, h0, h1);
            *reinterpret_cast<float2*>(hck) = make_float2(h0, h1);
        }
        hck += p.Di;
        pp.wait(st);
        unsigned char* sb = pp.gaddr(st);
#pragma unroll
        for (int j = 0; j < RG; ++j) {
            const float d = __shfl_sync(0xffffffffu, dmine, j * 4 + hsel);
            const f2 a = f2_ex2(f2_mul(f2_bcast(d), c.A2));
            h = f2_fma(a, h, up(lds_pair<T, TS>(sb, FA_B, j)));
            const f2 ys = f2_mul(up(lds_pair<T, TS>(sb, FA_C, j)), h);
            const f2 yv = f2_fma(c.Dv, up(lds_pair<T, TS>(sb, FA_X, j)), ys);
            const f2 zv = up(lds_pair<T, TS>(sb, FA_Z, j));
            sts_pair<T, TS>(sb, FA_X, j, f2_mul(yv, f2_mul(zv, f2_sigmoid<T>(zv))));      // y over the consumed x
            if (YSSM) sts_pair<T, TS>(sb, FA_C, j, ys);
            if (j == RG / 2 - 1 && w.leader) fd.refill(pp.k);      // half a group after the previous item's stores were issued
        }
        fence_async_smem();
        team_sync<TS>(w.team_in_cta);
        if (w.leader) {
            tma_store(m.y, pp.saddr(st, FA_X * TB), w.ch0_team, tb, w.b, pol_stream);
            if (YSSM) tma_store(m.ys, pp.saddr(st, FA_C * TB), w.ch0_team, tb, w.b, pol_stream);
            bulk_commit();
        }
        ++pp.k;
    }
}

template <typename T, int TS, int NST>
__device__ __forceinline__ void who_am_i(const RoundsParams& p, Who& w, Pipe& pp, unsigned char* smem_raw, int ntiles) {
    const int wic = threadIdx.x >> 5, nteams_cta = (blockDim.x >> 5) / TS;
    w.lane = threadIdx.x & 31;
    w.member = wic % TS;
    w.team_in_cta = wic / TS;
    const int gt = blockIdx.x * nteams_cta + w.team_in_cta;            // global team
    const int tc = gt % p.nteamchains;
    w.slot = gt / p.nteamchains;
    w.b = tc / p.tps;
    const int tslab = tc % p.tps;
    w.ch0_team = tslab * TS * 64;
    w.slab = tslab * TS + w.member;
    w.real = w.slab < p.nslab;
    w.chain = w.b * p.nslab + (w.real ? w.slab : 0);
    w.leader = w.member == 0 && w.lane == 0;
    w.cv = w.real && (w.slab * 64 + 2 * w.lane) < p.Di;
    pp.stage_bytes = (uint32_t)ntiles * Tile<T, TS>::BYTES;
    unsigned char* ring = smem_raw + (size_t)w.team_in_cta * NST * pp.stage_bytes;
    pp.sbase = ab_smem_u32(ring);
    pp.base = ring + (size_t)(w.member * 32 + w.lane) * sizeof(typename Raw<T>::type);
    pp.bar = ab_smem_u32(smem_raw + (size_t)nteams_cta * NST * pp.stage_bytes) + (uint32_t)w.team_in_cta * NST * 8u;
    pp.phases = 0;
    pp.k = 0;
    if (w.leader) {
#pragma unroll
        for (int i = 0; i < NST; ++i) mbar_init_u32(pp.baddr(i), 1);
        ab_fence_mbar_init();
    }
    __syncthreads();
}

template <typename T, bool YSSM, int TS, int NST, int HPS>
__global__ void __launch_bounds__(sizeof(T) == 2 ? 768 : 512, 1)
scan_rounds_fwd_kernel(const __grid_constant__ CUtensorMap tm_xa, const __grid_constant__ CUtensorMap tm_b, const __grid_constant__ CUtensorMap tm_b32,
                       const __grid_constant__ CUtensorMap tm_c, const __grid_constant__ CUtensorMap tm_z, const __grid_constant__ CUtensorMap tm_y,
                       const __grid_constant__ CUtensorMap tm_ys, const RoundsParams p) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    Who w;
    Pipe pp;
    who_am_i<T, TS, NST>(p, w, pp, smem_raw, 4);
    if (w.slot >= p.cpr) return;              // whole teams past the grid's share leave together
    const int lane = w.lane;
    const int c0 = w.slab * 64 + 2 * lane;
    FwdCtx<T> c;
    c.L = p.L;
    // head slots past the slab's HPS heads get head H (invalid): one test in the loops, not two
    const int head = (HPS == 4 || (lane & 3) < HPS) ? w.slab * HPS + (lane & 3) : p.H;
    c.hv = w.real && head < p.H;
    c.bias = (c.hv && p.dt_bias != nullptr) ? p.dt_bias[head] : 0.f;
    const int cs = w.cv ? c0 : 0;
    c.A2 = w.cv ? f2_pack(-__expf(p.A_log[c0]) * AB_LOG2E, -__expf(p.A_log[c0 + 1]) * AB_LOG2E) : f2_bcast(0.f);
    c.Dv = w.cv ? f2_pack(p.D[c0], p.D[c0 + 1]) : f2_bcast(0.f);
    c.dlog = reinterpret_cast<const T*>(p.dlog) + (int64_t)w.b * p.L * p.dlog_stride + (c.hv ? head : 0);
    c.delta = p.delta + (size_t)w.chain * p.L8 * 4 + (lane & 3);
    c.hck = p.hck + (size_t)w.b * p.nck8 * p.Di + cs;
    f2 init = f2_bcast(0.f);
    if (p.h0 != nullptr && w.cv) init = f2_pack(p.h0[(size_t)w.b * p.Di + c0], p.h0[(size_t)w.b * p.Di + c0 + 1]);
    const FwdMaps m{&tm_xa, &tm_b, &tm_b32, &tm_c, &tm_z, &tm_y, &tm_ys};
    const uint64_t pol_keep = policy_evict_last(), pol_stream = policy_evict_first();
    FwdFeeder<T, TS, NST> fd(p, w, pp, m, pol_keep, pol_stream);
    if (w.leader) fd.prime();
    Cursor<false> ph;
    for (ph.begin(p, w.slot); ph.kind >= 0; ph.next_phase(p, w.slot)) {
        if (ph.kind == 0) fwd_p1<T, TS, NST, HPS>(p, c, w, pp, fd, ph, init);
        else fwd_p2<T, YSSM, TS, NST, HPS>(p, c, w, pp, fd, m, ph, pol_stream);
    }
    if (w.leader) bulk_wait_all();
    team_finish(p, w.member, w.lane);
}

// ====================================================================================================================
// backward
//   dyv = dout * silu(z);  dz = dout * (C h + D x) * silu'(z);  dys = dyv (+ dyssm);  dxa = dyv * D;  dD += dyv * x
//   dC = dys * h;  E_t = C_t dys_t + F_{t+1};  dB = E;  F_t = abar_t E_t   (F: what a token hands to its predecessor)
//   d abar = E * h_{t-1};  w = d abar * abar;  d delta[head] += sum_c w * A_c;  dA_log_c += w * delta * A_c
//   d dlog = d delta * sigmoid(dlog) = d delta * (1 - exp(-delta))
// Chunks are visited from the end of the sequence; the reverse chunk aggregate is F_first = Pr * F_in + Sr.
// Rows past the sequence arrive as zeros (TMA fill): dout = 0 and delta = 0 make them hand F on unchanged.
// ====================================================================================================================
template <typename T>
struct BwdCtx {
    T* ddlog;
    const float* delta;
    const float* hck;
    f2 A2, Dv, An;      // An = natural-log A = -exp(A_log)
    int L;
};

// operand tiles of a backward stage (P1 fills C, Z, G (, S); P2 all); the results overwrite B, X, C, Z in place
constexpr int BA_B = 0, BA_X = 1, BA_C = 2, BA_Z = 3, BA_G = 4, BA_S = 5;

struct BwdMaps {
    const CUtensorMap *xa, *b, *c, *z, *g, *s, *dxa, *db, *dc, *dz;
};

template <typename T, bool YSSM, int TS, int NST>
struct BwdFeeder {
    const RoundsParams& p;
    const Who& w;
    Pipe& pp;
    const BwdMaps& m;
    Cursor<true> cur;
    uint64_t pol_keep, pol_stream;
    __device__ __forceinline__ BwdFeeder(const RoundsParams& p_, const Who& w_, Pipe& pp_, const BwdMaps& m_, uint64_t pk, uint64_t ps)
        : p(p_), w(w_), pp(pp_), m(m_), pol_keep(pk), pol_stream(ps) {}
    __device__ __forceinline__ void issue_one(int st) {
        if (cur.kind < 0) return;
        constexpr int TB = Tile<T, TS>::BYTES;
        const int t = cur.token();
        if (cur.kind == 0) {
            mbar_expect_tx_u32(pp.baddr(st), (YSSM ? 4 : 3) * TB);
            tma_load(pp.saddr(st, BA_C * TB), m.c, pp.baddr(st), w.ch0_team, t, w.b, pol_keep);
            tma_load(pp.saddr(st, BA_Z * TB), m.z, pp.baddr(st), w.ch0_team, t, w.b, pol_keep);
            tma_load(pp.saddr(st, BA_G * TB), m.g, pp.baddr(st), w.ch0_team, t, w.b, pol_keep);
            if (YSSM) tma_load(pp.saddr(st, BA_S * TB), m.s, pp.baddr(st), w.ch0_team, t, w.b, pol_keep);
        } else {
            mbar_expect_tx_u32(pp.baddr(st), (YSSM ? 6 : 5) * TB);
            tma_load(pp.saddr(st, BA_B * TB), m.b, pp.baddr(st), w.ch0_team, t, w.b, pol_stream);
            tma_load(pp.saddr(st, BA_G * TB), m.g, pp.baddr(st), w.ch0_team, t, w.b, pol_stream);
            tma_load(pp.saddr(st, BA_Z * TB), m.z, pp.baddr(st), w.ch0_team, t, w.b, pol_stream);
            tma_load(pp.saddr(st, BA_C * TB), m.c, pp.baddr(st), w.ch0_team, t, w.b, pol_stream);
            tma_load(pp.saddr(st, BA_X * TB), m.xa, pp.baddr(st), w.ch0_team, t, w.b, pol_stream);
            if (YSSM) tma_load(pp.saddr(st, BA_S * TB), m.s, pp.baddr(st), w.ch0_team, t, w.b, pol_stream);
        }
        cur.advance(p, w.slot);
    }
    __device__ __forceinline__ void prime() {
        cur.begin(p, w.slot);
#pragma unroll
        for (int i = 0; i < NST; ++i) issue_one(i);
    }
    __device__ __forceinline__ void refill(int k) {
        if (k < 1) return;
        bulk_wait_read<0>();
        issue_one((k - 1) % NST);
    }
};

template <typename T, bool YSSM, int TS, int NST, int HPS, typename Feeder>
__device__ __forceinline__ void bwd_p1(const RoundsParams& p, const BwdCtx<T>& c, const Who& w, Pipe& pp, Feeder& fd, const Cursor<true>& ph) {
    const int t0 = ph.t0, ngroups = ph.n;          // groups are visited last to first: step i handles group ngroups - 1 - i
    const int hsel = w.lane / (32 / HPS);
    f2 F = f2_bcast(0.f);
    float sumd = 0.f;
    const float* dsrc = c.delta + (int64_t)(t0 + (ngroups - 1) * RG + (w.lane >> 2)) * 4;
    float dnext = w.real ? __ldg(dsrc) : 0.f;
    for (int i = 0; i < ngroups; ++i) {
        const int st = pp.k % NST;
        const float dmine = dnext;
        dsrc -= RG * 4;
        if (w.real && i + 1 < ngroups) dnext = __ldg(dsrc);
        pp.wait(st);
        const unsigned char* sb = pp.gaddr(st);
#pragma unroll
        for (int j = RG - 1; j >= 0; --j) {
            const float d = __shfl_sync(0xffffffffu, dmine, j * 4 + hsel);
            const f2 a = f2_ex2(f2_mul(f2_bcast(d), c.A2));
            const f2 zv = up(lds_pair<T, TS>(sb, BA_Z, j));
            f2 dys = f2_mul(up(lds_pair<T, TS>(sb, BA_G, j)), f2_mul(zv, f2_sigmoid<T>(zv)));
            if (YSSM) dys = f2_add(dys, up(lds_pair<T, TS>(sb, BA_S, j)));
            F = f2_mul(a, f2_fma(up(lds_pair<T, TS>(sb, BA_C, j)), dys, F));
            sumd += d;
            if (j == RG / 2 && w.leader) fd.refill(pp.k);
        }
        team_sync<TS>(w.team_in_cta);
        ++pp.k;
    }
    if (!w.real) return;
    const f2 P = f2_ex2(f2_mul(f2_bcast(sumd), c.A2));
    publish_and_prefix(p, ph.r, w.chain, w.slot, ph.n_r, w.lane, P, F, f2_bcast(0.f), nullptr);
}

template <typename T, bool YSSM, int TS, int NST, int HPS, typename Feeder>
__device__ __forceinline__ void bwd_p2(const RoundsParams& p, const BwdCtx<T>& c, const Who& w, Pipe& pp, Feeder& fd, const BwdMaps& m,
                                       const Cursor<true>& ph, f2& accA, f2& accD, float& accB, uint64_t pol_stream) {
    const int t0 = ph.t0, ngroups = ph.n, r = ph.r;
    constexpr int LPH = 32 / HPS;                  // lanes per head
    const int hsel = w.lane / LPH;
    constexpr int TB = Tile<T, TS>::BYTES;
    const float* hck = c.hck + (size_t)((t0 >> 3) + ngroups - 1) * p.Di;
    const float* dsrc = c.delta + (int64_t)(t0 + (ngroups - 1) * RG + (w.lane >> 2)) * 4;
    float dnext = w.real ? __ldg(dsrc) : 0.f;
    float2 hnext = make_float2(0.f, 0.f);
    if (w.cv) hnext = __ldg(reinterpret_cast<const float2*>(hck));
    f2 F = f2_bcast(0.f);
    if (w.real) {
        wait_flag(&p.flag[(size_t)r * p.nchains + w.chain], w.lane);
        F = incoming_state(p, r, w.chain, w.slot, w.lane);
    }
    for (int i = 0; i < ngroups; ++i) {
        const int st = pp.k % NST;
        const int tb = t0 + (ngroups - 1 - i) * RG;
        const float dmine = dnext;
        const float2 hp = hnext;
        dsrc -= RG * 4;
        hck -= p.Di;
        if (i + 1 < ngroups) {
            if (w.real) dnext = __ldg(dsrc);
            if (w.cv) hnext = __ldg(reinterpret_cast<const float2*>(hck));
        }
        pp.wait(st);
        unsigned char* sb = pp.gaddr(st);
        // ---- forward recompute of the 8 states
        f2 a[RG], h[RG + 1];
        float dl[RG];
        h[0] = f2_pack(hp.x, hp.y);
#pragma unroll
        for (int j = 0; j < RG; ++j) {
            dl[j] = __shfl_sync(0xffffffffu, dmine, j * 4 + hsel);
            a[j] = f2_ex2(f2_mul(f2_bcast(dl[j]), c.A2));
            h[j + 1] = f2_fma(a[j], h[j], up(lds_pair<T, TS>(sb, BA_B, j)));
        }
        if (w.leader) fd.refill(pp.k);            // the previous item's stores were issued a recompute ago
        // ---- reverse sweep; every result goes over the operand it replaces
        float dd[RG];          // this lane's share (2 channels) of d delta of each token
#pragma unroll
        for (int j = RG - 1; j >= 0; --j) {
            const f2 zv = up(lds_pair<T, TS>(sb, BA_Z, j)), go = up(lds_pair<T, TS>(sb, BA_G, j));
            const f2 xx = up(lds_pair<T, TS>(sb, BA_X, j)), cc = up(lds_pair<T, TS>(sb, BA_C, j));
            const f2 sg = f2_sigmoid<T>(zv);
            const f2 dyv = f2_mul(go, f2_mul(zv, sg));
            const f2 yv = f2_fma(c.Dv, xx, f2_mul(cc, h[j + 1]));
            // silu'(z) = sg * (1 + z * (1 - sg)) = sg * (1 + z - z * sg)
            const f2 dsilu = f2_mul(sg, f2_fma(f2_mul(zv, sg), f2_bcast(-1.f), f2_add(zv, f2_bcast(1.f))));
            sts_pair<T, TS>(sb, BA_Z, j, f2_mul(f2_mul(go, yv), dsilu));
            sts_pair<T, TS>(sb, BA_X, j, f2_mul(dyv, c.Dv));
            accD = f2_fma(dyv, xx, accD);
            f2 dys = dyv;
            if (YSSM) dys = f2_add(dys, up(lds_pair<T, TS>(sb, BA_S, j)));
            sts_pair<T, TS>(sb, BA_C, j, f2_mul(dys, h[j + 1]));
            const f2 E = f2_fma(cc, dys, F);
            sts_pair<T, TS>(sb, BA_B, j, E);
            const f2 wv = f2_mul(f2_mul(E, h[j]), a[j]);
            dd[j] = f2_hsum(f2_mul(wv, c.An));
            accA = f2_fma(wv, f2_bcast(dl[j]), accA);
            F = f2_mul(a[j], E);
        }
        fence_async_smem();
        team_sync<TS>(w.team_in_cta);
        if (w.leader) {
            tma_store(m.db, pp.saddr(st, BA_B * TB), w.ch0_team, tb, w.b, pol_stream);
            tma_store(m.dxa, pp.saddr(st, BA_X * TB), w.ch0_team, tb, w.b, pol_stream);
            tma_store(m.dc, pp.saddr(st, BA_C * TB), w.ch0_team, tb, w.b, pol_stream);
            tma_store(m.dz, pp.saddr(st, BA_Z * TB), w.ch0_team, tb, w.b, pol_stream);
            bulk_commit();
        }
        ++pp.k;
        // ---- d delta: transposing butterfly over the 8 tokens inside each group of 8 lanes (16 channels), so that lane
        //      (head hsel, k = lane & 7) holds its group's share of token k, then the sum over the LPH / 8 groups of the head;
        //      every lane of a head then holds the same totals and only its first 8 lanes write them
        {
            const int k = w.lane & 7;
            float s4[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float keep = (k & 4) ? dd[q + 4] : dd[q];
                const float send = (k & 4) ? dd[q] : dd[q + 4];
                s4[q] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
            }
            float s2[2];
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const float keep = (k & 2) ? s4[q + 2] : s4[q];
                const float send = (k & 2) ? s4[q] : s4[q + 2];
                s2[q] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
            }
            const float keep = (k & 1) ? s2[1] : s2[0];
            const float send = (k & 1) ? s2[0] : s2[1];
            float tot = keep + __shfl_xor_sync(0xffffffffu, send, 1);            // token k of head hsel
#pragma unroll
            for (int m = 8; m < LPH; m <<= 1) tot += __shfl_xor_sync(0xffffffffu, tot, m);
            const float dk = __shfl_sync(0xffffffffu, dmine, k * 4 + hsel);       // delta of (token k, head hsel)
            const int head = w.slab * HPS + hsel;
            const int tok = tb + k;
            if (w.real && tok < c.L && (w.lane & (LPH - 1)) < 8) {
                if (head < p.H) {
                    // softplus'(x) = sigmoid(x) = 1 - exp(-softplus(x))
                    const float gq = tot * (1.0f - ab_ex2(-dk * AB_LOG2E));
                    accB += gq;
                    c.ddlog[(int64_t)tok * p.ddlog_stride + head] = ab_from_float<T>(gq);
                }
                int hh = head;
                if constexpr (HPS < 4) { if (hh < p.H) hh += (p.H - hh + HPS - 1) / HPS * HPS; }      // first padding column of this head's class
                for (; hh < p.ddlog_cols; hh += HPS)     // padding columns (covered by the last slab's lanes)
                    if (hh >= p.H) c.ddlog[(int64_t)tok * p.ddlog_stride + hh] = ab_from_float<T>(0.f);
            }
        }
    }
}

template <typename T, bool YSSM, int TS, int NST, int HPS>
__global__ void __launch_bounds__(sizeof(T) == 2 ? 512 : 256, 1)
scan_rounds_bwd_kernel(const __grid_constant__ CUtensorMap tm_xa, const __grid_constant__ CUtensorMap tm_b, const __grid_constant__ CUtensorMap tm_c,
                       const __grid_constant__ CUtensorMap tm_z, const __grid_constant__ CUtensorMap tm_g, const __grid_constant__ CUtensorMap tm_s,
                       const __grid_constant__ CUtensorMap tm_dxa, const __grid_constant__ CUtensorMap tm_db, const __grid_constant__ CUtensorMap tm_dc,
                       const __grid_constant__ CUtensorMap tm_dz, const RoundsParams p) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    Who w;
    Pipe pp;
    who_am_i<T, TS, NST>(p, w, pp, smem_raw, YSSM ? 6 : 5);
    const int gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (w.slot >= p.cpr) return;
    const int lane = w.lane;
    const int c0 = w.slab * 64 + 2 * lane;
    BwdCtx<T> c;
    c.L = p.L;
    const int cs = w.cv ? c0 : 0;
    const float a0 = w.cv ? -__expf(p.A_log[c0]) : 0.f, a1 = w.cv ? -__expf(p.A_log[c0 + 1]) : 0.f;
    c.An = f2_pack(a0, a1);
    c.A2 = f2_pack(a0 * AB_LOG2E, a1 * AB_LOG2E);
    c.Dv = w.cv ? f2_pack(p.D[c0], p.D[c0 + 1]) : f2_bcast(0.f);
    c.ddlog = reinterpret_cast<T*>(p.ddlog) + (int64_t)w.b * p.L * p.ddlog_stride;
    c.delta = p.delta + (size_t)w.chain * p.L8 * 4 + (lane & 3);
    c.hck = p.hck + (size_t)w.b * p.nck8 * p.Di + cs;
    const BwdMaps m{&tm_xa, &tm_b, &tm_c, &tm_z, &tm_g, &tm_s, &tm_dxa, &tm_db, &tm_dc, &tm_dz};
    const uint64_t pol_keep = policy_evict_last(), pol_stream = policy_evict_first();
    f2 accA = f2_bcast(0.f), accD = f2_bcast(0.f);
    float accB = 0.f;
    BwdFeeder<T, YSSM, TS, NST> fd(p, w, pp, m, pol_keep, pol_stream);
    if (w.leader) fd.prime();
    Cursor<true> ph;
    for (ph.begin(p, w.slot); ph.kind >= 0; ph.next_phase(p, w.slot)) {
        if (ph.kind == 0) bwd_p1<T, YSSM, TS, NST, HPS>(p, c, w, pp, fd, ph);
        else bwd_p2<T, YSSM, TS, NST, HPS>(p, c, w, pp, fd, m, ph, accA, accD, accB, pol_stream);
    }
    if (w.leader) bulk_wait_all();
    {
        // dA_log = A * sum(w * delta): accA holds sum(w * delta); phantom slabs contribute zeros
        const f2 da = f2_mul(accA, c.An);
        float x0, x1, y0, y1;
        f2_unpack(da, x0, x1);
        f2_unpack(accD, y0, y1);
        p.part[(size_t)gw * 32 + lane] = make_float4(x0, x1, y0, y1);
        p.part_b[(size_t)gw * 32 + lane] = accB;
    }
    team_finish(p, w.member, w.lane);
}

// dA_log[c], dD[c] (and d dt_bias[head]) = sum over the warps that worked on the channel's slab (all sequences, all chunk
// slots), fixed order: bitwise reproducible.  RED_SPLIT CTAs of 8 warps per slab each sum a fixed share of the partials
// (eight loads in flight per lane); the CTA that finishes last adds the RED_SPLIT shares in index order.
constexpr int RED_SPLIT = 8;

template <int HPS>
__global__ void __launch_bounds__(256) scan_rounds_param_reduce_kernel(const float4* __restrict__ part, const float* __restrict__ part_b, float* __restrict__ dA,
                                                                        float* __restrict__ dD, float* __restrict__ dbias, float4* __restrict__ stage2,
                                                                        float* __restrict__ stage2_b, unsigned* __restrict__ arrive, int Di, int H, int B,
                                                                        int TS, int tps, int nteamchains, int cpr) {
    __shared__ float4 red[8][32];
    __shared__ float redb[8][32];
    __shared__ unsigned is_last;
    const int slab = blockIdx.x, share = blockIdx.y, lane = threadIdx.x & 31, v = threadIdx.x >> 5;
    const int tslab = slab / TS, member = slab % TS;
    const int n = cpr * B;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    float accb = 0.f;
    // partial q belongs to share q % RED_SPLIT, warp (q / RED_SPLIT) % 8
    for (int i0 = v; ; i0 += 64) {
        const int qbase = i0 * RED_SPLIT + share;
        if (qbase >= n) break;
        float4 t[8];
        float tb[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int q = (i0 + u * 8) * RED_SPLIT + share;
            t[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            tb[u] = 0.f;
            if (q < n) {
                const int slot = q / B, b = q % B;
                const size_t gw = ((size_t)slot * nteamchains + (size_t)b * tps + tslab) * TS + member;
                t[u] = __ldcg(&part[gw * 32 + lane]);
                tb[u] = __ldcg(&part_b[gw * 32 + lane]);
            }
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) { acc.x += t[u].x; acc.y += t[u].y; acc.z += t[u].z; acc.w += t[u].w; accb += tb[u]; }
    }
    red[v][lane] = acc;
    redb[v][lane] = accb;
    __syncthreads();
    if (v == 0) {
        float4 sum = red[0][lane];
        float sb = redb[0][lane];
#pragma unroll
        for (int i = 1; i < 8; ++i) { sum.x += red[i][lane].x; sum.y += red[i][lane].y; sum.z += red[i][lane].z; sum.w += red[i][lane].w; sb += redb[i][lane]; }
        __stcg(&stage2[((size_t)slab * RED_SPLIT + share) * 32 + lane], sum);
        __stcg(&stage2_b[((size_t)slab * RED_SPLIT + share) * 32 + lane], sb);
        __syncwarp();
        if (lane == 0) {
            __threadfence();
            const unsigned old = atomicAdd(&arrive[slab], 1u);
            is_last = old == RED_SPLIT - 1;
            if (is_last) { __threadfence(); arrive[slab] = 0u; }      // left clean for the next launch
        }
        __syncwarp();
        if (is_last) {
            float4 tot = make_float4(0.f, 0.f, 0.f, 0.f);
            float tb2 = 0.f;
#pragma unroll
            for (int i = 0; i < RED_SPLIT; ++i) {
                const float4 q = __ldcg(&stage2[((size_t)slab * RED_SPLIT + i) * 32 + lane]);
                tot.x += q.x; tot.y += q.y; tot.z += q.z; tot.w += q.w;
                tb2 += __ldcg(&stage2_b[((size_t)slab * RED_SPLIT + i) * 32 + lane]);
            }
            const int c0 = slab * 64 + 2 * lane;
            if (c0 < Di) { dA[c0] = tot.x; dA[c0 + 1] = tot.y; dD[c0] = tot.z; dD[c0 + 1] = tot.w; }
            // lanes (head lane / (32 / HPS), token lane & 7): sum the 8 token lanes of a head (its other lanes hold zeros)
            tb2 += __shfl_xor_sync(0xffffffffu, tb2, 4);
            tb2 += __shfl_xor_sync(0xffffffffu, tb2, 2);
            tb2 += __shfl_xor_sync(0xffffffffu, tb2, 1);
            const int head = slab * HPS + lane / (32 / HPS);
            if (dbias != nullptr && (lane & (32 / HPS - 1)) == 0 && head < H) dbias[head] = tb2;
        }
    }
}

// ---- host ----------------------------------------------------------------------------------------------------------
struct RoundsCfg {
    int nslab, nchains, TS, NST, tps, nteamchains, teams_per_cta, nteams, cpr, Tc, nck, nrounds, nseg, nck8, L8, grid, block, nw_total;
    size_t smem, off_agg, off_segagg, off_segcarry, off_carry, off_cnt, cnt_bytes, off_part, off_part_b, off_stage2, total;
};

constexpr size_t SMEM_MAX = 227 * 1024;
constexpr size_t CNT_REGION = 1 << 20;      // head of the workspace: sign-off word, then the per-round counters / flags

// slabs per team: wide boxes (few, large TMA requests) against slabs lost to padding the last team of a sequence
int choose_ts(int nslab) {
    int best = 1;
    double best_score = -1.0;
    for (int ts = 1; ts <= 4 && ts <= nslab; ++ts) {
        const int tps = (nslab + ts - 1) / ts;
        const double score = (double)nslab / (tps * ts) * (ts >= 3 ? 1.0 : ts == 2 ? 0.9 : 0.75);
        if (score >= best_score) { best_score = score; best = ts; }
    }
    return best;
}

// Chunk length: few, well-filled rounds (the grid is persistent: a partly filled last round idles warps), at least two
// rounds where the sequence allows it (the prefix of round r hides behind P1 of round r + 1); every visit of a chunk
// starts its TMA ring cold, so short chunks pay a latency per visit.
int choose_tc(int L, int cpr, int tc_hint) {
    if (tc_hint >= RG) return (tc_hint / RG) * RG;
    int best = RG;
    double best_score = -1.0;
    for (int tc = RG; tc <= 256; tc += RG) {
        const int nck = (int)ab_ceil_div(L, tc);
        const int rounds = (int)ab_ceil_div(nck, cpr);
        double score = (double)L / ((double)rounds * cpr * tc);            // fill
        score *= (double)tc / (tc + 24.0);                                 // per-visit overhead ~ 3 groups of work (ring fill, prefix wait)
        if (rounds == 1 && nck > 1) score *= 0.9;                          // exposed prefix
        if (score > best_score) { best_score = score; best = tc; }
    }
    return best;
}

int g_nst_fwd = 0, g_nst_bwd = 0;

int make_cfg(int B, int L, int Di, int dtype, bool bwd, bool yssm, int warp_cap, int tc_hint, RoundsCfg& c) {
    const int es = dtype == AB_F32 ? 4 : 2;
    c.nslab = (int)ab_ceil_div(Di, 64);
    c.nchains = B * c.nslab;
    c.TS = choose_ts(c.nslab);
    c.tps = (c.nslab + c.TS - 1) / c.TS;
    c.nteamchains = B * c.tps;
    const size_t tile = (size_t)RG * c.TS * 64 * es;
    int reg_cap = bwd ? (es == 2 ? 16 : 8) : (es == 2 ? 24 : 16);          // warps per CTA under the kernels' __launch_bounds__
    if (warp_cap > 0 && reg_cap > warp_cap) reg_cap = warp_cap;
    // ring depth: three stages (two items in flight per team) when that still leaves the register-limited number of
    // teams or at least four of them, else two
    const int want = bwd ? g_nst_bwd : g_nst_fwd;
    const size_t stage = (size_t)(bwd ? (yssm ? 6 : 5) : 4) * tile;
    const int tpc3 = (int)((SMEM_MAX - 1024) / (3 * stage + 24));
    c.NST = want == 2 || want == 3 ? want : ((tpc3 >= reg_cap / c.TS || tpc3 >= 4) ? 3 : 2);
    const size_t per_team = (size_t)c.NST * stage + c.NST * 8;
    int tpc = (int)((SMEM_MAX - 1024) / per_team);
    if (tpc > reg_cap / c.TS) tpc = reg_cap / c.TS;
    if (tpc > 15) tpc = 15;                                                 // named barriers 1..15
    if (tpc < 1) tpc = 1;
    c.teams_per_cta = tpc;
    c.smem = (size_t)tpc * per_team + 128;
    c.block = tpc * c.TS * 32;
    c.nteams = ab_num_sms() * tpc;
    AB_REQUIRE(c.nteamchains <= c.nteams, "selective scan: %d (sequence, slab group) chains exceed the %d resident teams; split the batch", c.nteamchains, c.nteams);
    c.cpr = c.nteams / c.nteamchains;
    c.nck8 = (int)ab_ceil_div(L, RG);
    c.L8 = c.nck8 * RG;
    if (c.cpr > c.nck8) c.cpr = c.nck8;
    c.Tc = choose_tc(L, c.cpr, tc_hint);
    c.nck = (int)ab_ceil_div(L, c.Tc);
    if (c.cpr > c.nck) c.cpr = c.nck;
    c.grid = (int)ab_ceil_div((int64_t)c.cpr * c.nteamchains, tpc);
    c.nw_total = c.grid * tpc * c.TS;
    c.nrounds = (int)ab_ceil_div(c.nck, c.cpr);
    c.nseg = (int)ab_ceil_div(c.cpr, RSEG);
    // counters first, at a fixed place: a launch leaves them zeroed for the next one whatever its shape
    c.cnt_bytes = (size_t)c.nrounds * c.nchains * (c.nseg + 2) * sizeof(unsigned);
    AB_REQUIRE(c.cnt_bytes + 4096 <= CNT_REGION && c.nslab <= 1000, "selective scan: %zu bytes of round counters exceed the reserved %zu", c.cnt_bytes, (size_t)CNT_REGION);
    c.off_cnt = 4096;                    // [0]: sign-off word; [64 ..): one arrival word per slab of the parameter reduce
    size_t o = CNT_REGION;
    c.off_agg = o;      o += (size_t)2 * c.nchains * c.cpr * 32 * sizeof(float4);
    c.off_segagg = o;   o += (size_t)2 * c.nchains * c.nseg * 32 * sizeof(float4);
    c.off_segcarry = o; o += (size_t)2 * c.nchains * c.nseg * 32 * sizeof(float2);
    c.off_carry = o;    o += (size_t)c.nchains * 32 * sizeof(float2);
    c.off_part = o;     o += (size_t)c.nw_total * 32 * sizeof(float4);
    c.off_part_b = o;   o += (size_t)c.nw_total * 32 * sizeof(float);
    c.off_stage2 = o;   o += (size_t)c.nslab * RED_SPLIT * 32 * (sizeof(float4) + sizeof(float));
    c.total = o;
    return AB_OK;
}

void fill_sync(RoundsParams& p, const RoundsCfg& c, void* ws) {
    unsigned char* w = reinterpret_cast<unsigned char*>(ws);
    p.agg = reinterpret_cast<float4*>(w + c.off_agg);
    p.segagg = reinterpret_cast<float4*>(w + c.off_segagg);
    p.segcarry = reinterpret_cast<float2*>(w + c.off_segcarry);
    p.carry = reinterpret_cast<float2*>(w + c.off_carry);
    p.part = reinterpret_cast<float4*>(w + c.off_part);
    p.part_b = reinterpret_cast<float*>(w + c.off_part_b);
    p.cnt1 = reinterpret_cast<unsigned*>(w + c.off_cnt);
    p.cnt2 = p.cnt1 + (size_t)c.nrounds * c.nchains * c.nseg;
    p.flag = p.cnt2 + (size_t)c.nrounds * c.nchains;
    p.done = reinterpret_cast<unsigned*>(w);
    p.cnt_words = (int)(c.cnt_bytes / sizeof(unsigned));
    p.nteams_used = c.cpr * c.nteamchains;
    p.nslab = c.nslab; p.nchains = c.nchains; p.Tc = c.Tc; p.nck = c.nck; p.cpr = c.cpr; p.nrounds = c.nrounds; p.nseg = c.nseg;
    p.nw_used = c.nw_total; p.nck8 = c.nck8; p.L8 = c.L8; p.tps = c.tps; p.nteamchains = c.nteamchains;
}

int g_tc_hint_fwd = 0, g_tc_hint_bwd = 0, g_warp_cap = 0;

// A 64-channel slab holds 64 / N whole heads of N = Di / H channels (ssm_d_state); N = 16, 32, 64 -> 4, 2, 1 heads per slab.
int heads_per_slab(int Di, int H) { return 64 * H / Di; }

int common_checks(const char* who, int B, int L, int Di, int H, int dtype) {
    AB_REQUIRE(B > 0 && L > 0 && Di > 0 && H > 0, "%s: B, L, Di, H must be positive", who);
    AB_REQUIRE(Di == 16 * H || Di == 32 * H || Di == 64 * H,
               "%s: Di (%d) must be N * H (H = %d) with ssm_d_state N in {16, 32, 64}", who, Di, H);
    AB_REQUIRE(dtype == AB_F32 || dtype == AB_BF16, "%s: bad dtype %d", who, dtype);
    return AB_OK;
}

// 3-D tensor map over [B, L, Di] rows (row stride in elements), box = `cols` channels x `rows` tokens.  Encoding costs a
// few microseconds of host time per map and a launch uses up to ten: recently used maps are kept (a training loop presents
// the same buffers again and again through torch's caching allocator).
struct MapKey {
    const void* base; int dtype, B, L, Di, rows, cols; int64_t stride;
    bool operator==(const MapKey& o) const {
        return base == o.base && dtype == o.dtype && B == o.B && L == o.L && Di == o.Di && rows == o.rows && cols == o.cols && stride == o.stride;
    }
};
constexpr int MAP_CACHE = 128;
struct MapCache { MapKey key[MAP_CACHE]; CUtensorMap map[MAP_CACHE]; int used = 0, next = 0; };
MapCache g_maps;
std::mutex g_maps_mutex;

int map3(CUtensorMap* m, const void* base, int dtype, int B, int L, int Di, int64_t stride, int rows, int cols) {
    const int es = dtype == AB_F32 ? 4 : 2;
    AB_REQUIRE(((uintptr_t)base % 16) == 0 && (stride * es) % 16 == 0 && stride >= Di,
               "selective scan: activations must be 16-byte aligned with a 16-byte aligned row stride >= Di (stride %lld elements)", (long long)stride);
    const MapKey k{base, dtype, B, L, Di, rows, cols, stride};
    {
        std::lock_guard<std::mutex> g(g_maps_mutex);
        for (int i = 0; i < g_maps.used; ++i)
            if (g_maps.key[i] == k) { *m = g_maps.map[i]; return AB_OK; }
    }
    uint64_t dims[3] = {(uint64_t)Di, (uint64_t)L, (uint64_t)B};
    uint64_t strides[2] = {(uint64_t)stride * es, (uint64_t)stride * es * L};
    uint32_t box[3] = {(uint32_t)cols, (uint32_t)rows, 1u};
    if (int e = ab_encode_tmap(m, dtype == AB_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, base, dims, strides, box,
                               CU_TENSOR_MAP_SWIZZLE_NONE)) return e;
    std::lock_guard<std::mutex> g(g_maps_mutex);
    const int slot = g_maps.used < MAP_CACHE ? g_maps.used++ : (g_maps.next++ % MAP_CACHE);
    g_maps.key[slot] = k;
    g_maps.map[slot] = *m;
    return AB_OK;
}

template <typename K>
int set_smem(K kernel, size_t bytes) {
    AB_CHECK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return AB_OK;
}

struct FwdLaunch {
    CUtensorMap xa, b, b32, c, z, y, ys;
};
template <typename T, bool YS, int TS, int NST, int HPS>
int launch_fwd_n(const FwdLaunch& m, const RoundsParams& p, const RoundsCfg& c, cudaStream_t stream) {
    static size_t configured = 0;          // cudaFuncSetAttribute is a driver call: only when the requirement grows
    if (c.smem > configured) {
        if (int e = set_smem(scan_rounds_fwd_kernel<T, YS, TS, NST, HPS>, c.smem)) return e;
        configured = c.smem;
    }
    scan_rounds_fwd_kernel<T, YS, TS, NST, HPS><<<c.grid, c.block, c.smem, stream>>>(m.xa, m.b, m.b32, m.c, m.z, m.y, m.ys, p);
    AB_LAUNCH_CHECK();
    return AB_OK;
}
template <typename T, bool YS, int TS, int HPS>
int launch_fwd(const FwdLaunch& m, const RoundsParams& p, const RoundsCfg& c, cudaStream_t stream) {
    return c.NST == 3 ? launch_fwd_n<T, YS, TS, 3, HPS>(m, p, c, stream) : launch_fwd_n<T, YS, TS, 2, HPS>(m, p, c, stream);
}
template <typename T, bool YS, int HPS>
int launch_fwd_ts(const FwdLaunch& m, const RoundsParams& p, const RoundsCfg& c, cudaStream_t stream) {
    switch (c.TS) {
        case 1: return launch_fwd<T, YS, 1, HPS>(m, p, c, stream);
        case 2: return launch_fwd<T, YS, 2, HPS>(m, p, c, stream);
        case 3: return launch_fwd<T, YS, 3, HPS>(m, p, c, stream);
        default: return launch_fwd<T, YS, 4, HPS>(m, p, c, stream);
    }
}
template <typename T, bool YS>
int launch_fwd_hps(const FwdLaunch& m, const RoundsParams& p, const RoundsCfg& c, int hps, cudaStream_t stream) {
    switch (hps) {
        case 4: return launch_fwd_ts<T, YS, 4>(m, p, c, stream);
        case 2: return launch_fwd_ts<T, YS, 2>(m, p, c, stream);
        default: return launch_fwd_ts<T, YS, 1>(m, p, c, stream);
    }
}
struct BwdLaunch {
    CUtensorMap xa, b, c, z, g, s, dxa, db, dc, dz;
};
template <typename T, bool YS, int TS, int NST, int HPS>
int launch_bwd_n(const BwdLaunch& m, const RoundsParams& p, const RoundsCfg& c, cudaStream_t stream) {
    static size_t configured = 0;
    if (c.smem > configured) {
        if (int e = set_smem(scan_rounds_bwd_kernel<T, YS, TS, NST, HPS>, c.smem)) return e;
        configured = c.smem;
    }
    scan_rounds_bwd_kernel<T, YS, TS, NST, HPS><<<c.grid, c.block, c.smem, stream>>>(m.xa, m.b, m.c, m.z, m.g, m.s, m.dxa, m.db, m.dc, m.dz, p);
    AB_LAUNCH_CHECK();
    return AB_OK;
}
template <typename T, bool YS, int TS, int HPS>
int launch_bwd(const BwdLaunch& m, const RoundsParams& p, const RoundsCfg& c, cudaStream_t stream) {
    return c.NST == 3 ? launch_bwd_n<T, YS, TS, 3, HPS>(m, p, c, stream) : launch_bwd_n<T, YS, TS, 2, HPS>(m, p, c, stream);
}
template <typename T, bool YS, int HPS>
int launch_bwd_ts(const BwdLaunch& m, const RoundsParams& p, const RoundsCfg& c, cudaStream_t stream) {
    switch (c.TS) {
        case 1: return launch_bwd<T, YS, 1, HPS>(m, p, c, stream);
        case 2: return launch_bwd<T, YS, 2, HPS>(m, p, c, stream);
        case 3: return launch_bwd<T, YS, 3, HPS>(m, p, c, stream);
        default: return launch_bwd<T, YS, 4, HPS>(m, p, c, stream);
    }
}
template <typename T, bool YS>
int launch_bwd_hps(const BwdLaunch& m, const RoundsParams& p, const RoundsCfg& c, int hps, cudaStream_t stream) {
    switch (hps) {
        case 4: return launch_bwd_ts<T, YS, 4>(m, p, c, stream);
        case 2: return launch_bwd_ts<T, YS, 2>(m, p, c, stream);
        default: return launch_bwd_ts<T, YS, 1>(m, p, c, stream);
    }
}

}  // namespace

// ---- C ABI ---------------------------------------------------------------------------------------------------------
extern "C" int ab_ssm_scan_tune(int tc_fwd, int tc_bwd, int warps_per_sm, int stages_fwd, int stages_bwd) {
    g_tc_hint_fwd = tc_fwd; g_tc_hint_bwd = tc_bwd; g_warp_cap = warps_per_sm; g_nst_fwd = stages_fwd; g_nst_bwd = stages_bwd;
    return AB_OK;
}

extern "C" int ab_ssm_scan_plan(int B, int L, int Di, int dtype, int64_t* state_floats, size_t* ws_bytes) {
    if (int e = common_checks("ssm_scan_plan", B, L, Di, Di / 16, dtype)) return e;
    size_t total = 0;
    for (int bwd = 0; bwd < 2; ++bwd)
        for (int ys = 0; ys < 2; ++ys) {
            RoundsCfg c;
            if (int e = make_cfg(B, L, Di, dtype, bwd != 0, ys != 0, g_warp_cap, bwd ? g_tc_hint_bwd : g_tc_hint_fwd, c)) return e;
            if (c.total > total) total = c.total;
        }
    const int64_t nck8 = ab_ceil_div(L, RG), nslab = ab_ceil_div(Di, 64);
    if (state_floats) *state_floats = (int64_t)B * nck8 * Di + (int64_t)B * nslab * nck8 * RG * 4;
    if (ws_bytes) *ws_bytes = total;
    return AB_OK;
}

extern "C" int ab_ssm_scan_fwd(const void* xa, int64_t xa_stride, const void* dlog, int64_t dlog_stride, const float* dt_bias,
                               const void* Bm, const void* Cm, int64_t bc_stride, const void* z, int64_t z_stride,
                               const float* A_log, const float* D, const float* h0, void* y, void* y_ssm, float* h_last,
                               float* state, void* ws, size_t ws_bytes, int B, int L, int Di, int H, int dtype,
                               cudaStream_t stream) {
    if (int e = common_checks("ssm_scan_fwd", B, L, Di, H, dtype)) return e;
    const int es = dtype == AB_F32 ? 4 : 2;
    AB_REQUIRE(xa && dlog && Bm && Cm && z && A_log && D && y && state && ws, "ssm_scan_fwd: null argument");
    AB_REQUIRE(xa_stride >= Di && bc_stride >= Di && z_stride >= Di && dlog_stride >= H, "ssm_scan_fwd: a row stride is smaller than its row");
    AB_REQUIRE(((xa_stride | bc_stride | z_stride) % 2) == 0, "ssm_scan_fwd: row strides must be even (channel pairs are loaded as one word)");
    AB_REQUIRE((xa_stride | bc_stride | z_stride | dlog_stride) < (1 << 30), "ssm_scan_fwd: row strides must be below 2^30 elements");
    AB_REQUIRE(((uintptr_t)xa | (uintptr_t)Bm | (uintptr_t)Cm | (uintptr_t)z | (uintptr_t)y | (uintptr_t)y_ssm) % (2 * es) == 0,
               "ssm_scan_fwd: activations must be aligned to a channel pair");
    RoundsCfg c;
    if (int e = make_cfg(B, L, Di, dtype, false, y_ssm != nullptr, g_warp_cap, g_tc_hint_fwd, c)) return e;
    AB_REQUIRE(ws_bytes >= c.total, "ssm_scan_fwd: workspace too small (%zu < %zu)", ws_bytes, c.total);
    RoundsParams p;
    memset(&p, 0, sizeof(p));
    fill_sync(p, c, ws);
    p.B = B; p.L = L; p.Di = Di; p.H = H;
    p.dlog = dlog; p.dlog_stride = (int)dlog_stride;
    p.dt_bias = dt_bias; p.A_log = A_log; p.D = D; p.h0 = h0; p.h_last = h_last;
    p.hck = state;
    p.delta = state + (size_t)B * c.nck8 * Di;
    FwdLaunch m;
    const int cols = c.TS * 64;
    if (int e = map3(&m.xa, xa, dtype, B, L, Di, xa_stride, RG, cols)) return e;
    if (int e = map3(&m.b, Bm, dtype, B, L, Di, bc_stride, RG, cols)) return e;
    if (int e = map3(&m.b32, Bm, dtype, B, L, Di, bc_stride, P1_ROWS, cols)) return e;
    if (int e = map3(&m.c, Cm, dtype, B, L, Di, bc_stride, RG, cols)) return e;
    if (int e = map3(&m.z, z, dtype, B, L, Di, z_stride, RG, cols)) return e;
    if (int e = map3(&m.y, y, dtype, B, L, Di, Di, RG, cols)) return e;
    m.ys = m.y;
    if (y_ssm) { if (int e = map3(&m.ys, y_ssm, dtype, B, L, Di, Di, RG, cols)) return e; }
    const int hps = heads_per_slab(Di, H);
    if (dtype == AB_F32) return y_ssm ? launch_fwd_hps<float, true>(m, p, c, hps, stream) : launch_fwd_hps<float, false>(m, p, c, hps, stream);
    return y_ssm ? launch_fwd_hps<__nv_bfloat16, true>(m, p, c, hps, stream) : launch_fwd_hps<__nv_bfloat16, false>(m, p, c, hps, stream);
}

extern "C" int ab_ssm_scan_bwd(const void* xa, int64_t xa_stride, const void* Bm, const void* Cm, int64_t bc_stride,
                               const void* z, int64_t z_stride, const void* dout, const void* dyssm, const float* A_log,
                               const float* D, const float* state, void* dxa, int64_t dxa_stride, void* dBm, void* dCm,
                               int64_t dbc_stride, void* dz, int64_t dz_stride, void* ddlog, int64_t ddlog_stride, int ddlog_cols,
                               float* ddt_bias, float* dA_log, float* dD, void* ws, size_t ws_bytes, int B, int L, int Di, int H, int dtype,
                               cudaStream_t stream) {
    if (int e = common_checks("ssm_scan_bwd", B, L, Di, H, dtype)) return e;
    const int es = dtype == AB_F32 ? 4 : 2;
    AB_REQUIRE(xa && Bm && Cm && z && dout && A_log && D && state && dxa && dBm && dCm && dz && ddlog && dA_log && dD && ws,
               "ssm_scan_bwd: null argument");
    AB_REQUIRE(xa_stride >= Di && bc_stride >= Di && z_stride >= Di && dxa_stride >= Di && dbc_stride >= Di && dz_stride >= Di && ddlog_stride >= H && ddlog_cols <= ddlog_stride,
               "ssm_scan_bwd: a row stride is smaller than its row");
    AB_REQUIRE(((xa_stride | bc_stride | z_stride | dxa_stride | dbc_stride | dz_stride) % 2) == 0, "ssm_scan_bwd: row strides must be even");
    AB_REQUIRE((xa_stride | bc_stride | z_stride | dxa_stride | dbc_stride | dz_stride | ddlog_stride) < (1 << 30), "ssm_scan_bwd: row strides must be below 2^30 elements");
    AB_REQUIRE(((uintptr_t)xa | (uintptr_t)Bm | (uintptr_t)Cm | (uintptr_t)z | (uintptr_t)dout | (uintptr_t)dyssm | (uintptr_t)dxa | (uintptr_t)dBm |
                (uintptr_t)dCm | (uintptr_t)dz) % (2 * es) == 0, "ssm_scan_bwd: activations must be aligned to a channel pair");
    RoundsCfg c;
    if (int e = make_cfg(B, L, Di, dtype, true, dyssm != nullptr, g_warp_cap, g_tc_hint_bwd, c)) return e;
    AB_REQUIRE(ws_bytes >= c.total, "ssm_scan_bwd: workspace too small (%zu < %zu)", ws_bytes, c.total);
    RoundsParams p;
    memset(&p, 0, sizeof(p));
    fill_sync(p, c, ws);
    p.B = B; p.L = L; p.Di = Di; p.H = H;
    p.ddlog = ddlog; p.ddlog_stride = (int)ddlog_stride; p.ddlog_cols = ddlog_cols;
    p.A_log = A_log; p.D = D;
    p.hck = const_cast<float*>(state);
    p.delta = const_cast<float*>(state) + (size_t)B * c.nck8 * Di;
    BwdLaunch m;
    const int cols = c.TS * 64;
    if (int e = map3(&m.xa, xa, dtype, B, L, Di, xa_stride, RG, cols)) return e;
    if (int e = map3(&m.b, Bm, dtype, B, L, Di, bc_stride, RG, cols)) return e;
    if (int e = map3(&m.c, Cm, dtype, B, L, Di, bc_stride, RG, cols)) return e;
    if (int e = map3(&m.z, z, dtype, B, L, Di, z_stride, RG, cols)) return e;
    if (int e = map3(&m.g, dout, dtype, B, L, Di, Di, RG, cols)) return e;
    m.s = m.g;
    if (dyssm) { if (int e = map3(&m.s, dyssm, dtype, B, L, Di, Di, RG, cols)) return e; }
    if (int e = map3(&m.dxa, dxa, dtype, B, L, Di, dxa_stride, RG, cols)) return e;
    if (int e = map3(&m.db, dBm, dtype, B, L, Di, dbc_stride, RG, cols)) return e;
    if (int e = map3(&m.dc, dCm, dtype, B, L, Di, dbc_stride, RG, cols)) return e;
    if (int e = map3(&m.dz, dz, dtype, B, L, Di, dz_stride, RG, cols)) return e;
    const int hps = heads_per_slab(Di, H);
    int e;
    if (dtype == AB_F32) e = dyssm ? launch_bwd_hps<float, true>(m, p, c, hps, stream) : launch_bwd_hps<float, false>(m, p, c, hps, stream);
    else e = dyssm ? launch_bwd_hps<__nv_bfloat16, true>(m, p, c, hps, stream) : launch_bwd_hps<__nv_bfloat16, false>(m, p, c, hps, stream);
    if (e) return e;
    unsigned char* w8 = reinterpret_cast<unsigned char*>(ws);
    float4* stage2 = reinterpret_cast<float4*>(w8 + c.off_stage2);
    float* stage2_b = reinterpret_cast<float*>(stage2 + (size_t)c.nslab * RED_SPLIT * 32);
    auto reduce = hps == 4 ? scan_rounds_param_reduce_kernel<4> : hps == 2 ? scan_rounds_param_reduce_kernel<2> : scan_rounds_param_reduce_kernel<1>;
    reduce<<<dim3(c.nslab, RED_SPLIT), 256, 0, stream>>>(p.part, p.part_b, dA_log, dD, ddt_bias, stage2, stage2_b, reinterpret_cast<unsigned*>(w8 + 64),
                                                         Di, H, B, c.TS, c.tps, c.nteamchains, c.cpr);
    AB_LAUNCH_CHECK();
    return AB_OK;
}
