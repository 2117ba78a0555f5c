// Fused iteration kernels for onesided fp32 with 16 (8) complex values per lane (gl_warp_core.cuh), hop = n_fft/OV
// with OV = 2, 4 or 8 frames overlapping on every sample (template parameter; 4 is the reference's default hop):
//   n_fft =  512 : one warp per frame, 8 values per lane (LANES = 32, VV = 8)
//   n_fft = 1024 : one warp per frame    (LANES = 32)   -- the headline shape (cfg2: hop = 256)
//   n_fft = 2048 : two warps per frame   (LANES = 64)   -- cfg1, cfg4 (hop = 512)
//   n_fft = 4096 : four warps per frame  (LANES = 128)  -- cfg5 (hop = 1024)
//
// One launch = one whole Griffin-Lim (or ADMM) iteration.  Every group of LANES/32 warps walks through a
// contiguous range of the B*T frames (crossing signal boundaries if need be) and for each frame does,
// entirely on chip:
//   window -> real FFT (M-point complex FFT in three passes, gl_warp_core.cuh) -> momentum / ADMM update and
//   magnitude projection on the FFT outputs in registers -> inverse FFT -> windowed overlap-add.
//   * 16 complex values per lane: <= 168 registers, 12 free-running warps per SM (no CTA-wide barriers; the
//     warps of a frame group meet at a named barrier per exchange), and the unrolled frame body fits the
//     instruction cache;
//   * the lane-constant tables (windows, twiddles), the lane-private input ring and the overlap-add carry
//     live in TENSOR MEMORY and move with tcgen05.ld / tcgen05.st (one instruction per 8..32 registers, no
//     shared-memory bandwidth); shared memory only carries the four FFT exchanges (swizzled, conflict free);
//   * the q / X and magnitude rows of the NEXT frame and the next hop of input samples are fetched by the TMA
//     (cp.async.bulk, one elected lane, mbarrier completion) into per-group staging rows one frame ahead, so
//     the compute never waits on DRAM; the new state is written straight from registers, 256 contiguous
//     bytes per warp instruction.
// A range re-computes the OV - 1 frames before it as a halo (state not written, output not stored), so ranges are
// independent: no atomics, deterministic.  State arrays are ping-ponged (q_in != q_out).
#pragma once
#include <cstdlib>

#include "specinv_common.cuh"
#include "gl_warp_core.cuh"
#include "sm100_ptx.cuh"

namespace specinv {
namespace wfast {

struct WArgs {
    const float* x_in; float* x_out;
    const float2* s0_in;  const float2* s0_in_nyq;  float2* s0_out; float2* s0_out_nyq;
    const float2* s1_in;  const float2* s1_in_nyq;  float2* s1_out; float2* s1_out_nyq;
    const float* mag;     const float* mag_nyq;
    const float2* tw;     const float2* twr;        // plan tables: W_M^j (M entries), W_N^k (k <= M/2)
    const float* wa; const float* ws; const float* inv_env;
    double* sums;
    float coef, coef2;
    int B, T, P, pad_mode;
    long long L;
    long long frames_total;     // B * T
    int ranges;                 // number of warp groups that get a frame range
};

// TMEM columns (per lane): constant tables shared by the warps of one sub-partition, then per-warp state
constexpr int TC_WA = 0, TC_WS = 32, TC_TW1 = 64, TC_TW2 = 96, TC_TWR = 128, TC_IE = 144;
// One-warp-per-frame variants (LANES = 32) also keep the CONJUGATES of the three twiddle tables (fft_regs.cuh: cmul2t):
// 64 more columns, which is exactly what 12 warps x 96 columns of ring / carry leave of the 512.
constexpr int TC_TW1C = 160, TC_TW2C = 192, TC_TWRC = 208;
constexpr bool has_conj_tables(int lanes) { return lanes == 32; }
constexpr int tc_warp(int lanes) { return has_conj_tables(lanes) ? 224 : 160; }
// per warp: the input ring (OV - 1 hops) then the overlap-add carry (OV - 1 hops), a hop = 2 VV / OV words per lane
// (OV = n_fft / hop = 2, 4 or 8 overlapping frames per sample; 48 words for OV = 4 and 16 values per lane)
constexpr int ring_words(int vv, int ov) { return (ov - 1) * 2 * vv / ov; }
constexpr int TMEM_COLS = 512;
// 12 warps x 168 registers (no spills), 12 x 15 KB of staging fills the shared memory; the 8-values-per-lane variant
// needs <= 128 registers and half the staging: 16 warps (measured at B = 512, T = 1251: GL 0.722 -> 0.678 ms; ADMM,
// whose 36 B/bin are already HBM-bound, is faster with 12: 1.07 vs 1.12 ms)
constexpr int warps_of(int vv, int op) { return vv == 8 && op != OP_ADMM ? 16 : 12; }
// float2 of shared memory per frame group: E1, E2 (M float2 each), staged input block (HOP floats = M/OV float2),
// magnitude row (M floats = M/2 float2), q / X row (M float2)
constexpr int group_f2(int m, int ov) { return 2 * m + m / ov + m / 2 + m; }
// W words of tensor memory per lane, W any even number: pieces of 32, 16, 8, 4, 2
template <int W> __device__ __forceinline__ void tmem_ldn(unsigned taddr, float* r) {
    if constexpr (W >= 32) { tmem_ld32(taddr, r); tmem_ldn<W - 32>(taddr + 32, r + 32); }
    else if constexpr (W >= 16) { tmem_ld16(taddr, r); tmem_ldn<W - 16>(taddr + 16, r + 16); }
    else if constexpr (W >= 8) { tmem_ld8(taddr, r); tmem_ldn<W - 8>(taddr + 8, r + 8); }
    else if constexpr (W >= 4) { tmem_ld4(taddr, r); tmem_ldn<W - 4>(taddr + 4, r + 4); }
    else if constexpr (W >= 2) { tmem_ld2(taddr, r); }
}
template <int W> __device__ __forceinline__ void tmem_stn(unsigned taddr, const float* r) {
    if constexpr (W >= 32) { tmem_st32(taddr, r); tmem_stn<W - 32>(taddr + 32, r + 32); }
    else if constexpr (W >= 16) { tmem_st16(taddr, r); tmem_stn<W - 16>(taddr + 16, r + 16); }
    else if constexpr (W >= 8) { tmem_st8(taddr, r); tmem_stn<W - 8>(taddr + 8, r + 8); }
    else if constexpr (W >= 4) { tmem_st4(taddr, r); tmem_stn<W - 4>(taddr + 4, r + 4); }
    else if constexpr (W >= 2) { tmem_st2(taddr, r); }
}

// Synchronise the warps that share a frame (named barrier per group) or just the warp.
template <int LANES>
__device__ __forceinline__ void group_sync(int bar_id) {
    if constexpr (LANES == 32) __syncwarp();
    else asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "n"(LANES) : "memory");
}

// Fetch block u (padded samples [HOP u, HOP u + HOP)) of signal x: lane l gets the pairs at 2 LANES j + 2 l.
template <int LANES, int VV, int OV>
__device__ __forceinline__ void fetch_block_regs(const WArgs& a, const float* __restrict__ x, int u, int l, float2* nb) {
    constexpr int HOP = Cfg<LANES, VV>::N / OV, HP = VV / OV;
    const long long base = (long long)u * HOP - a.P;
    if (base >= 0 && base + HOP <= a.L) {
#pragma unroll
        for (int j = 0; j < HP; ++j) nb[j] = __ldg(reinterpret_cast<const float2*>(x + base + 2 * LANES * j + 2 * l));
    } else {
#pragma unroll
        for (int j = 0; j < HP; ++j) {
            const long long pp = (long long)u * HOP + 2 * LANES * j + 2 * l;
            const long long i0 = pad_index(pp, a.P, a.L, a.pad_mode), i1 = pad_index(pp + 1, a.P, a.L, a.pad_mode);
            nb[j] = f2(i0 >= 0 ? x[i0] : 0.f, i1 >= 0 ? x[i1] : 0.f);
        }
    }
}
// Same into the staging buffer xs[LANES j + l] (= the block's bytes in memory order): interior blocks by one TMA
// bulk copy issued by the group's first warp (returns true: the data arrives on `bar`), padded edge blocks
// element by element.
template <int LANES, int VV, int OV>
__device__ __forceinline__ bool fetch_block_staged(const WArgs& a, const float* __restrict__ x, int u, int l, float2* xs,
                                                   unsigned xs_s, unsigned bar) {
    constexpr int HOP = Cfg<LANES, VV>::N / OV, HP = VV / OV;
    const long long base = (long long)u * HOP - a.P;
    if (base >= 0 && base + HOP <= a.L) {
        if (l < 32) { if (elect_one()) { mbar_expect_tx(bar, HOP * 4); bulk_g2s(xs_s, x + base, HOP * 4, bar); } }
        return true;
    }
#pragma unroll
    for (int j = 0; j < HP; ++j) {
        const long long pp = (long long)u * HOP + 2 * LANES * j + 2 * l;
        const long long i0 = pad_index(pp, a.P, a.L, a.pad_mode), i1 = pad_index(pp + 1, a.P, a.L, a.pad_mode);
        xs[LANES * j + l] = f2(i0 >= 0 ? x[i0] : 0.f, i1 >= 0 ? x[i1] : 0.f);
    }
    return false;
}
template <int LANES, int VV, int OV>
__device__ __forceinline__ bool block_valid(const WArgs& a, int u) {
    constexpr int HOP = Cfg<LANES, VV>::N / OV;
    const long long base = (long long)u * HOP - a.P;
    return base >= 0 && base + HOP <= a.L;
}
template <int LANES, int VV, int OV>
__device__ __forceinline__ void load_inv_env(const WArgs& a, int u, int l, float2* ie) {
    const long long base = (long long)u * (Cfg<LANES, VV>::N / OV) - a.P;
#pragma unroll
    for (int j = 0; j < VV / OV; ++j) {
        // volatile + "memory": the compiler must not sink these loads down to their use
        asm volatile("ld.global.nc.v2.f32 {%0, %1}, [%2];" : "=f"(ie[j].x), "=f"(ie[j].y)
                     : "l"(a.inv_env + base + 2 * LANES * j + 2 * l) : "memory");
    }
}
template <int LANES, int VV, int OV>
__device__ __forceinline__ void store_block_ie(const WArgs& a, float* __restrict__ xo, int u, int l, const float2* blk,
                                               const float2* ie) {
    const long long base = (long long)u * (Cfg<LANES, VV>::N / OV) - a.P;
#pragma unroll
    for (int j = 0; j < VV / OV; ++j)
        *reinterpret_cast<float2*>(xo + base + 2 * LANES * j + 2 * l) = pmul(blk[j], ie[j]);
}
// Fetch the q / X row and the magnitude row of frame `row` into the staging rows (one elected lane, TMA).
template <int OP, int LANES, int VV>
__device__ __forceinline__ void stage_rows(const WArgs& a, long long row, int l, unsigned qstage_s, unsigned mstage_s, unsigned bar) {
    constexpr int M = Cfg<LANES, VV>::M;
    if (l < 32) {
        if (elect_one()) {
            mbar_expect_tx(bar, OP == OP_ISTFT ? M * 8 : OP == OP_GLP ? M * 4 : M * 8 + M * 4);
            if constexpr (OP != OP_GLP) bulk_g2s(qstage_s, a.s0_in + row * M, M * 8, bar);
            if constexpr (OP != OP_ISTFT) bulk_g2s(mstage_s, a.mag + row * M, M * 4, bar);
        }
    }
}

template <int OP, bool SUMS, int LANES, int VV, int OV>
__global__ void __launch_bounds__(warps_of(VV, OP) * 32, 1) warp_iter_kernel(const WArgs a) {
    using C = Cfg<LANES, VV>;
    constexpr int M = C::M;
    constexpr int V = VV;                         // complex values per lane (shadows wfast::V)
    constexpr int HOP = C::N / OV;                // samples per hop; OV frames overlap on every interior sample
    constexpr int HP = VV / OV;                   // sample pairs per hop and lane
    constexpr int NR = OV - 1;                    // hops in the input ring = hops in the carry = halo frames
    constexpr int RING_W = ring_words(VV, OV);    // words per lane of the ring (and of the carry)
    constexpr int TC_PER_WARP = 2 * RING_W;
    constexpr int RC = C::RC;                     // pair slots per lane
    constexpr int GROUP_F2 = group_f2(M, OV);
    constexpr int G = LANES / 32;                 // warps per frame group
    constexpr int WARPS = warps_of(VV, OP);
    constexpr int GROUPS = WARPS / G;
    constexpr bool HC = has_conj_tables(LANES);
    constexpr int TC_WARP = tc_warp(LANES);
    static_assert(TC_WARP + ((WARPS + 3) / 4) * TC_PER_WARP <= TMEM_COLS && TC_IE + 2 * HP <= 160, "TMEM columns");
    extern __shared__ __align__(16) float2 sm[];
    __shared__ unsigned s_tmem_base;
    __shared__ __align__(8) unsigned long long s_bar[GROUPS][3];   // per group: input block, state rows, ADMM U row
    const int tid = threadIdx.x, warp = tid >> 5;
    const int grp = warp / G;                     // frame group inside the CTA
    const int l = tid - grp * LANES;              // lane inside the group, 0 .. LANES-1
    const int bar_id = 1 + grp;
    if (warp == 0) tmem_alloc(&s_tmem_base, TMEM_COLS);
    const unsigned xbar = (unsigned)__cvta_generic_to_shared(&s_bar[grp][0]), sbar = xbar + 8, ubar = xbar + 16;
    if (l == 0) { mbar_init(xbar, 1); mbar_init(sbar, 1); mbar_init(ubar, 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    // this warp's TMEM window: lanes 32 * (warp % 4) .. +31.  A group's warps sit on consecutive sub-partitions
    // (G divides 4), so the position inside the group, hence the lane-constant tables, depend on warp % 4 only.
    const unsigned tlane = s_tmem_base + ((unsigned)(32 * (warp & 3)) << 16);
    if (warp < 4) {
        const int tl = 32 * (warp % G) + (tid & 31);       // group lane served by this sub-partition
        float t[32];
#pragma unroll
        for (int i = 0; i < V; ++i) { t[2 * i] = 0.5f * a.wa[2 * LANES * i + 2 * tl]; t[2 * i + 1] = 0.5f * a.wa[2 * LANES * i + 2 * tl + 1]; }
        tmem_stw<2 * V>(tlane + TC_WA, t);
#pragma unroll
        for (int i = 0; i < V; ++i) { t[2 * i] = a.ws[2 * LANES * i + 2 * tl]; t[2 * i + 1] = a.ws[2 * LANES * i + 2 * tl + 1]; }
        tmem_stw<2 * V>(tlane + TC_WS, t);
#pragma unroll
        for (int i = 0; i < V; ++i) {       // [R1 s + ka]: W_M^((tl + LANES s) ka)
            const float2 w = a.tw[((tl + LANES * (i / C::R1)) * (i % C::R1)) & (M - 1)];
            t[2 * i] = w.x; t[2 * i + 1] = w.y;
        }
        tmem_stw<2 * V>(tlane + TC_TW1, t);
#pragma unroll
        for (int kb = 0; kb < 16; ++kb) {   // W_(RC R2)^(c kb) = W_M^(R1 c kb), c = tl & (RC - 1)
            const float2 w = a.tw[(C::R1 * (tl & (RC - 1)) * (kb % C::R2)) & (M - 1)];
            t[2 * kb] = w.x; t[2 * kb + 1] = w.y;
        }
        tmem_st32(tlane + TC_TW2, t);
#pragma unroll
        for (int j = 0; j < RC; ++j) {
            const int k = slot_bin_rt<LANES, VV>(tl, j);
            float2 w;
            if (k <= M / 2) w = a.twr[k];
            else { w = a.twr[M - k]; w.x = -w.x; }                  // W_N^k = -conj(W_N^(M-k))
            t[2 * j] = w.x; t[2 * j + 1] = w.y;
        }
        tmem_stw<2 * RC>(tlane + TC_TWR, t);
        if constexpr (HC) {
#pragma unroll
            for (int j = 0; j < RC; ++j) t[2 * j + 1] = -t[2 * j + 1];
            tmem_stw<2 * RC>(tlane + TC_TWRC, t);
#pragma unroll
            for (int i = 0; i < V; ++i) {
                const float2 w = a.tw[((tl + LANES * (i / C::R1)) * (i % C::R1)) & (M - 1)];
                t[2 * i] = w.x; t[2 * i + 1] = -w.y;
            }
            tmem_stw<2 * V>(tlane + TC_TW1C, t);
#pragma unroll
            for (int kb = 0; kb < C::R2; ++kb) {
                const float2 w = a.tw[(C::R1 * (tl & (RC - 1)) * kb) & (M - 1)];
                t[2 * kb] = w.x; t[2 * kb + 1] = -w.y;
            }
            tmem_stw<2 * C::R2>(tlane + TC_TW2C, t);
        }
        tmem_wait_st();
    }
    // Programmatic dependent launch: everything above touched only this CTA's own resources and the plan's window /
    // twiddle tables, so it may run under the tail of the previous kernel of the stream (the previous iteration).
    // The tables are written by plan_tables_kernel only; the host side enforces that this kernel is never launched
    // with the programmatic attribute right behind it (note_tables_launch / pdl_prologue_safe, specinv_common.cuh).  Let the next launch start as early as SM resources allow, then
    // wait until the previous grid has completed and its writes are visible before the first access to anything it
    // may have written (the 1/envelope, the signal, the state) or may still be reading (the ping-pong buffers).
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
    // 1/envelope of an INTERIOR hop (OV overlapping frames): the envelope is periodic with the hop there, so
    // blocks OV-1 .. T-1 take it from here instead of streaming it from memory (block OV-1 is the first such block)
    if (warp < 4 && a.T >= OV) {
        const int tl = 32 * (warp % G) + (tid & 31);
        float t[2 * HP];
#pragma unroll
        for (int j = 0; j < HP; ++j) {
            const float2 e = *reinterpret_cast<const float2*>(a.inv_env + ((long long)NR * HOP - a.P) + 2 * LANES * j + 2 * tl);
            t[2 * j] = e.x; t[2 * j + 1] = e.y;
        }
        tmem_stw<2 * HP>(tlane + TC_IE, t);
        tmem_wait_st();
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    const unsigned twarp = tlane + TC_WARP + TC_PER_WARP * (warp >> 2);   // ring (RING_W columns) then carry (RING_W)
    float2* e1 = sm + grp * GROUP_F2;
    float2* e2 = e1 + M;
    float2* xs = e2 + M;                                            // HOP floats = M / OV float2
    float* mstage = reinterpret_cast<float*>(xs + M / OV);          // magnitudes of the coming frame (M floats)
    float2* qstage = xs + M / OV + M / 2;                           // q / X row of the coming frame
    const unsigned grp_s = (unsigned)__cvta_generic_to_shared(sm) + grp * (GROUP_F2 * 8);   // shared-window addresses
    const unsigned xs_s = grp_s + 2 * M * 8, mstage_s = xs_s + (M / OV) * 8, qstage_s = mstage_s + (M / 2) * 8;
    unsigned xpar = 0, spar = 0, upar = 0;                          // mbarrier phase parities

    // bin offsets of the lane's pair slots inside a main row
    const int hi_adj = l == 0 ? -(RC - 1) * LANES : 0;  // lane 0, slots j >= RC/2: LANES + 2 LANES (j - RC/2)
    const int kq0 = l == 0 ? M / 2 : M - l;

    double dacc = 0.0, eacc = 0.0;
    const int gg = blockIdx.x + gridDim.x * grp;                    // global group index
    long long g = 0, g1 = 0;
    if (gg < a.ranges) {
        g = a.frames_total * gg / a.ranges;
        g1 = a.frames_total * (gg + 1) / a.ranges;
    }
    while (g < g1) {
        const int b = (int)(g / a.T);
        const int t0 = (int)(g - (long long)b * a.T);
        const int t1 = (int)min((long long)a.T, t0 + (g1 - g));
        g += t1 - t0;
        const int tf0 = max(0, t0 - NR);
        const float* x = a.x_in + (long long)b * a.L;
        float* xo = a.x_out + (long long)b * a.L;

        // ---- prologue: empty carry, ring = blocks tf0 .. tf0 + NR - 1, block tf0 + NR and the first rows on their way
        tmem_wait_st();
        {
            float z[RING_W];
#pragma unroll
            for (int i = 0; i < RING_W; ++i) z[i] = 0.f;
            tmem_stn<RING_W>(twarp + RING_W, z);
        }
        int m = tf0 % NR;                                           // ring slot of block t
        if constexpr (OP != OP_ISTFT) {
            int mm = m;
#pragma unroll
            for (int i = 0; i < NR; ++i) {
                float2 nb[HP];
                fetch_block_regs<LANES, VV, OV>(a, x, tf0 + i, l, nb);
                tmem_stw<2 * HP>(twarp + 2 * HP * mm, reinterpret_cast<const float*>(nb));
                mm = mm == NR - 1 ? 0 : mm + 1;
            }
        }
        group_sync<LANES>(bar_id);                 // nobody still reads the staging rows of an earlier range
        bool x_async = false;
        if constexpr (OP != OP_ISTFT) x_async = fetch_block_staged<LANES, VV, OV>(a, x, tf0 + NR, l, xs, xs_s, xbar);
        stage_rows<OP, LANES, VV>(a, (long long)b * a.T + tf0, l, qstage_s, mstage_s, sbar);
        // Nyquist scalars of the coming frame (lane 0), fetched one frame ahead like the rows
        float2 s0n_next = f2(0.f, 0.f), s1n_next = f2(0.f, 0.f);
        float mgn_next = 0.f;
        if (l == 0) {
            const long long r0 = (long long)b * a.T + tf0;
            if constexpr (OP != OP_GLP) s0n_next = __ldg(a.s0_in_nyq + r0);
            if constexpr (OP != OP_ISTFT) mgn_next = __ldg(a.mag_nyq + r0);
            if constexpr (OP == OP_ADMM) s1n_next = __ldg(a.s1_in_nyq + r0);
        }
        if constexpr (OP == OP_ADMM) {             // U rows are read straight from global memory: pull them into L2
            const char* u0 = reinterpret_cast<const char*>(a.s1_in + ((long long)b * a.T + tf0) * M);
            if (128 * l < M * 8) prefetch_l2(u0 + 128 * l);
        }

        for (int t = tf0; t < t1; ++t) {
            const long long row = (long long)b * a.T + t;
            const bool owned = t >= t0;
            float2 v[V];
            float2 A[RC], Bv[RC];
            if constexpr (OP != OP_ISTFT) {
            // ---- assemble the frame: blocks t .. t+NR-1 from the ring, block t+NR from the staging buffer
            {
                tmem_wait_st();
                int mm = m;
#pragma unroll
                for (int i = 0; i < NR; ++i) {
                    tmem_ldw<2 * HP>(twarp + 2 * HP * mm, reinterpret_cast<float*>(v + i * HP));
                    mm = mm == NR - 1 ? 0 : mm + 1;
                }
                if (x_async) { mbar_wait(xbar, xpar); xpar ^= 1; }
#pragma unroll
                for (int j = 0; j < HP; ++j) v[NR * HP + j] = xs[LANES * j + l];
                tmem_stw<2 * HP>(twarp + 2 * HP * m, reinterpret_cast<const float*>(v + NR * HP));   // block t+NR replaces block t
                m = m == NR - 1 ? 0 : m + 1;
            }
            group_sync<LANES>(bar_id);             // xs consumed by every lane; the previous frame's reads of E1 are done
            if (t + 1 < t1) {
                x_async = fetch_block_staged<LANES, VV, OV>(a, x, t + OV, l, xs, xs_s, xbar);
                if constexpr (OP == OP_ADMM) {
                    const char* u1 = reinterpret_cast<const char*>(a.s1_in + (row + 1) * M);
                    if (128 * l < M * 8) prefetch_l2(u1 + 128 * l);
                }
            }
            {
                float2 w[V];
                tmem_ldw<2 * V>(tlane + TC_WA, reinterpret_cast<float*>(w));
#pragma unroll
                for (int i = 0; i < V; ++i) v[i] = pmul(v[i], w[i]);
            }
            {
                float2 tw1[V], tw1c[HC ? V : 1];
                tmem_ldw<2 * V>(tlane + TC_TW1, reinterpret_cast<float*>(tw1));
                if constexpr (HC) tmem_ldw<2 * V>(tlane + TC_TW1C, reinterpret_cast<float*>(tw1c));
                fwd_pass1<LANES, VV, HC>(l, v, tw1, e1, tw1c);
            }
            group_sync<LANES>(bar_id);
            {
                float2 tw2[C::R2], tw2c[HC ? C::R2 : 1];
                if constexpr (C::R2 == 8) tmem_ld16(tlane + TC_TW2, reinterpret_cast<float*>(tw2));
                else tmem_ld32(tlane + TC_TW2, reinterpret_cast<float*>(tw2));
                if constexpr (HC) tmem_ldw<2 * C::R2>(tlane + TC_TW2C, reinterpret_cast<float*>(tw2c));
                fwd_pass2<LANES, VV, HC>(l, e1, tw2, e2, tw2c);
            }
            group_sync<LANES>(bar_id);
            if constexpr (OP == OP_ADMM) {
                // E1 is idle until the inverse pass 2: stage this frame's U row (L2-prefetched a frame ago) in it
                if (l < 32) { if (elect_one()) { mbar_expect_tx(ubar, M * 8); bulk_g2s(grp_s, a.s1_in + row * M, M * 8, ubar); } }
            }
            fwd_pass3<LANES, VV>(l, e2, A, Bv);
            }  // OP != OP_ISTFT
            const float2 s0n = s0n_next, s1n = s1n_next;
            const float mgn = mgn_next;
            mbar_wait(sbar, spar); spar ^= 1;      // this frame's staged rows have landed
            if constexpr (OP == OP_ADMM) { mbar_wait(ubar, upar); upar ^= 1; }
            {
                // ---- point-wise stage on the lane's 16 bins (+ Nyquist for lane 0), state fetched where it is used.
                // Element e = 2 j / 2 j + 1 is the P / Q bin of slot j: bins l + 2 LANES j and M - l - 2 LANES j, except
                // for lane 0 (slots 4..7: 2 LANES j - 7 LANES and its mirror; slot 0: bins 0 and M/2).  Four per-lane
                // base offsets turn every access into base + compile-time offset.
                struct IO {
                    const float2* q; const float* mg; const float2* u; float2* o0; float2* o1;
                    float2* o0n; float2* o1n;
                    int pl, ph, ql, qh, q0; bool owned;
                    float2 s0n, s1n; float mgn;
                    __device__ __forceinline__ int bin(int e) const {
                        const int j = e >> 1;
                        return (e & 1) ? (j == 0 ? q0 : (j >= RC / 2 ? qh : ql) - 2 * LANES * j)
                                       : (j >= RC / 2 ? ph : pl) + 2 * LANES * j;
                    }
                    __device__ __forceinline__ float2 s0(int e) const { return e < 0 ? s0n : q[bin(e)]; }
                    __device__ __forceinline__ float2 s1(int e) const { return e < 0 ? s1n : u[bin(e)]; }
                    __device__ __forceinline__ float mag(int e) const { return e < 0 ? mgn : mg[bin(e)]; }
                    __device__ __forceinline__ void put(int e, float2 v0, float2 v1) const {
                        if (!owned) return;
                        if (e < 0) {
                            *o0n = v0;
                            if constexpr (OP == OP_ADMM) *o1n = v1;
                        } else {
                            o0[bin(e)] = v0;
                            if constexpr (OP == OP_ADMM) o1[bin(e)] = v1;
                        }
                    }
                } io{qstage, mstage, e1, OP == OP_GLP ? nullptr : a.s0_out + row * M,
                     OP == OP_ADMM ? a.s1_out + row * M : nullptr, a.s0_out_nyq + row,
                     OP == OP_ADMM ? a.s1_out_nyq + row : nullptr, l, l + hi_adj, M - l, M - l - hi_adj, kq0, owned,
                     s0n, s1n, mgn};
                float2 twr[RC], twrc[HC ? RC : 1];
                tmem_ldw<2 * RC>(tlane + TC_TWR, reinterpret_cast<float*>(twr));
                if constexpr (HC) tmem_ldw<2 * RC>(tlane + TC_TWRC, reinterpret_cast<float*>(twrc));
                if constexpr (OP == OP_ISTFT) {
                    spectrum_pairs<VV, HC>(l, A, Bv, twr, io, twrc);
                } else {
                    float dsum = 0.f, esum = 0.f;
                    pointwise<OP, SUMS, VV, HC>(l, A, Bv, twr, io, a.coef, a.coef2, dsum, esum, twrc);
                    if constexpr (SUMS) { if (owned) { dacc += (double)dsum; eacc += (double)esum; } }
                }
            }
            group_sync<LANES>(bar_id);             // every lane has read its classes from E2 and its staged state
            if (t + 1 < t1) {
                stage_rows<OP, LANES, VV>(a, row + 1, l, qstage_s, mstage_s, sbar);
                if (l == 0) {
                    if constexpr (OP != OP_GLP) s0n_next = __ldg(a.s0_in_nyq + row + 1);
                    if constexpr (OP != OP_ISTFT) mgn_next = __ldg(a.mag_nyq + row + 1);
                    if constexpr (OP == OP_ADMM) s1n_next = __ldg(a.s1_in_nyq + row + 1);
                }
            }
            inv_pass3<LANES, VV>(l, A, Bv, e2);
            group_sync<LANES>(bar_id);
            const bool emit = owned && block_valid<LANES, VV, OV>(a, t);
            float2 ie[HP];
            if (emit && t < NR) load_inv_env<LANES, VV, OV>(a, t, l, ie);   // edge blocks; early: hidden behind the last two passes
            {
                float2 tw2[C::R2], tw2c[HC ? C::R2 : 1];
                if constexpr (C::R2 == 8) tmem_ld16(tlane + TC_TW2, reinterpret_cast<float*>(tw2));
                else tmem_ld32(tlane + TC_TW2, reinterpret_cast<float*>(tw2));
                if constexpr (HC) tmem_ldw<2 * C::R2>(tlane + TC_TW2C, reinterpret_cast<float*>(tw2c));
                inv_pass2<LANES, VV, HC>(l, e2, tw2, e1, tw2c);
            }
            group_sync<LANES>(bar_id);
            {
                float2 tw1[V], tw1c[HC ? V : 1];
                tmem_ldw<2 * V>(tlane + TC_TW1, reinterpret_cast<float*>(tw1));
                if constexpr (HC) tmem_ldw<2 * V>(tlane + TC_TW1C, reinterpret_cast<float*>(tw1c));
                inv_pass1<LANES, VV, HC>(l, e1, tw1, v, tw1c);
            }
            // ---- windowed overlap-add: out = carry (NR hops from earlier frames) + ws * v; the first hop
            // (HP pairs) of `out` is a finished block, the other NR * HP pairs are the new carry
            {
                float2 w[V], carry[NR * HP];
                tmem_ldw<2 * V>(tlane + TC_WS, reinterpret_cast<float*>(w));
                tmem_ldn<RING_W>(twarp + RING_W, reinterpret_cast<float*>(carry));
#pragma unroll
                for (int i = 0; i < V; ++i) v[i] = i < NR * HP ? pfma(w[i], v[i], carry[i]) : pmul(w[i], v[i]);
                tmem_stn<RING_W>(twarp + RING_W, reinterpret_cast<const float*>(v + HP));
                if (emit) {
                    if (t >= NR) tmem_ldw<2 * HP>(tlane + TC_IE, reinterpret_cast<float*>(ie));   // interior: periodic envelope
                    store_block_ie<LANES, VV, OV>(a, xo, t, l, v, ie);
                }
            }
        }
        if (t1 == a.T) {      // tail of the signal: blocks T .. T+NR-1 are complete now
            float2 carry[NR * HP];
            tmem_wait_st();
            tmem_ldn<RING_W>(twarp + RING_W, reinterpret_cast<float*>(carry));
#pragma unroll
            for (int k = 0; k < NR; ++k)
                if (block_valid<LANES, VV, OV>(a, a.T + k)) {
                    float2 ie[HP];
                    load_inv_env<LANES, VV, OV>(a, a.T + k, l, ie);
                    store_block_ie<LANES, VV, OV>(a, xo, a.T + k, l, carry + HP * k, ie);
                }
        }
    }

    if constexpr (SUMS) {
        double d = dacc, e = eacc;
        for (int o = 16; o > 0; o >>= 1) {
            d += __shfl_xor_sync(0xffffffffu, d, o);
            e += __shfl_xor_sync(0xffffffffu, e, o);
        }
        if ((tid & 31) == 0 && (d != 0.0 || e != 0.0)) { atomicAdd(a.sums, d); atomicAdd(a.sums + 1, e); }
    }
    tmem_wait_st();
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) tmem_dealloc(s_tmem_base, TMEM_COLS);
}

static int g_sms = 0;

template <int OP, int OV, int LANES, int VV = V>
static int launch(const WArgs& a0, cudaStream_t st) {
    WArgs a = a0;
    if (g_sms == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return SPECINV_ERR_NO_DEVICE;
        if (cudaDeviceGetAttribute(&g_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return SPECINV_ERR_NO_DEVICE;
    }
    // the TMA bulk copies need 16-byte aligned rows
    // (s0_in is NULL for OP_GLP, s1_in for everything but ADMM, whose U rows are bulk-copied too)
    if ((((uintptr_t)a.x_in | (uintptr_t)a.s0_in | (uintptr_t)a.s1_in | (uintptr_t)a.mag) & 15) != 0) return SPECINV_ERR_UNSUPPORTED;
    if (OP == OP_ISTFT && a.sums) return SPECINV_ERR_INVALID;
    a.frames_total = (long long)a.B * a.T;
    constexpr int WARPS = warps_of(VV, OP);
    constexpr int GROUPS = WARPS / (LANES / 32);
    const int slots = g_sms * GROUPS;
    // One frame range per group slot.  A range re-computes OV - 1 halo frames, which costs ~1.5 % when the ranges are
    // long (the batched configs) and buys parallelism when the problem is small (one short signal).
    long long ranges = a.frames_total < slots ? a.frames_total : slots;
    a.ranges = (int)ranges;
    const int grid = (int)min((long long)g_sms, ranges);
    // with fewer ranges than group slots, spread them over all CTAs of the grid: range index = blockIdx + grid * group
    const size_t smem = (size_t)GROUPS * group_f2(Cfg<LANES, VV>::M, OV) * sizeof(float2);
    // launched with programmatic stream serialization: the kernel's prologue may overlap the previous kernel's tail
    // (see griddepcontrol.wait in the kernel)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(WARPS * 32); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    // ... unless the library's last launch on this stream was the kernel that WRITES the plan tables the prologue reads
    // (specinv_common.cuh: pdl_prologue_safe); then this launch is fully serialised behind it.
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = pdl_prologue_safe(st) ? 1 : 0;
    cfg.attrs = attr; cfg.numAttrs = 1;
    cudaError_t e;
    if (a.sums) {
        e = cudaFuncSetAttribute(warp_iter_kernel<OP, true, LANES, VV, OV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        e = cudaLaunchKernelEx(&cfg, warp_iter_kernel<OP, true, LANES, VV, OV>, a);
    } else {
        e = cudaFuncSetAttribute(warp_iter_kernel<OP, false, LANES, VV, OV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        e = cudaLaunchKernelEx(&cfg, warp_iter_kernel<OP, false, LANES, VV, OV>, a);
    }
    return (int)e;
}

template <int OP, int OV>
static int launch_any(const WArgs& a, int n_fft, cudaStream_t st) {
    switch (n_fft) {
        case 512: return launch<OP, OV, 32, 8>(a, st);
        case 1024: return launch<OP, OV, 32>(a, st);
        case 2048: return launch<OP, OV, 64>(a, st);
        case 4096: return launch<OP, OV, 128>(a, st);
        default: return SPECINV_ERR_UNSUPPORTED;
    }
}

// One translation unit per overlap factor (they compile in parallel): fastw_launch_ov<OV>(op, args, n_fft, stream)
#define SPECINV_FASTW_DEFINE_LAUNCH(OV)                                                        \
    int fastw_launch_ov##OV(int op, const WArgs& a, int n_fft, cudaStream_t st) {              \
        switch (op) {                                                                          \
            case OP_GL: return launch_any<OP_GL, OV>(a, n_fft, st);                            \
            case OP_ADMM: return launch_any<OP_ADMM, OV>(a, n_fft, st);                        \
            case OP_ISTFT: return launch_any<OP_ISTFT, OV>(a, n_fft, st);                      \
            case OP_GLP: return launch_any<OP_GLP, OV>(a, n_fft, st);                          \
            case OP_GLR: return launch_any<OP_GLR, OV>(a, n_fft, st);                          \
            default: return SPECINV_ERR_INVALID;                                               \
        }                                                                                      \
    }
int fastw_launch_ov2(int op, const WArgs& a, int n_fft, cudaStream_t st);
int fastw_launch_ov4(int op, const WArgs& a, int n_fft, cudaStream_t st);
int fastw_launch_ov8(int op, const WArgs& a, int n_fft, cudaStream_t st);

}  // namespace wfast
}  // namespace specinv
