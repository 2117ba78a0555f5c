// RTISI-LA (torch_specinv/methods.py:273-412) for n_fft = 1024 / hop = 256 (the shape of BASELINE.json's cfg3),
// n_fft = 512 / hop = 128 and n_fft = 2048 / hop = 512, look_ahead <= 3, onesided fp32, as ONE persistent kernel built
// from the register FFT pipeline of gl_warp_core.cuh (16 or 8 complex values per lane, one warp -- two for 2048 --
// per frame).
//
// A signal is owned by LA+1 warps, one per ACTIVE frame; a frame stays in its warp's registers for its whole
// life (LA+1 outer steps x max_iter inner iterations), together with its momentum spectrum (tensor memory) and
// its magnitude row (tensor memory, fetched once when the frame is born).  Per inner iteration (methods.py:365-398)
// every warp
//   * publishes its synthesis-windowed frame u = frame * w * c in shared memory (rows of 32 lanes),
//   * rebuilds ITS frame of the overlap-add y: a hop is a quarter of a lane's sample pairs, so the contributions of the
//     other frames are the same lane's rows shifted by 4 per frame; the kept frames' part is constant over the
//     inner iterations and waits in tensor memory,
//   * windows it (asym_window1/2 for the newest frame when asked), runs the forward FFT, the momentum update
//     q = S - lr * pre and the magnitude projection on the FFT outputs in registers, and the inverse FFT.
// One named barrier per inner iteration (the u exchange, double buffered); the four FFT exchanges stay inside the
// warp.  After max_iter iterations the oldest frame is committed: it joins the kept ring and is overlap-added
// (window w, 1/envelope, centre trimming) into the output (methods.py:401-408).  HBM traffic: the magnitudes once,
// the signal once.
#include "specinv_common.cuh"
#include "gl_warp_core.cuh"
#include "sm100_ptx.cuh"

namespace specinv {
namespace rfast {

using namespace wfast;

constexpr int KEEP = 3, NAMAX = 4;            // kept frames (n_fft = 4 hop), at most LA + 1 = 4 active frames

struct RArgs {
    const float* mag; const float* mag_nyq;
    float* x_out;
    const float2* tw; const float2* twr;
    const float* wa; const float* ws; const float* inv_env;   // inv_env: samples [x0, x0 + x_len)
    const float* asym1; const float* asym2;   // analysis windows of the newest frame (already x forward scale)
    float coef;                               // c = hop / (w . w)
    float lr;                                 // alpha / (1 + alpha)
    int B, T, P, LA, max_iter, asymmetric;
    int frame0, n_rows, final;                // magnitude window and whether T is the total (RtisiWindow)
    long long x0, x_len;                      // output window: x_out column c of a signal is sample x0 + c
    int step_begin, step_end;                 // outer steps [step_begin, step_end) of the T + LA steps of a run
    float* state;                             // per-signal sliding state in / out (specinv_rtisi.cu: rtisi_state_elems)
    size_t state_elems;
};

// TMEM columns per lane: constant tables (identical in the four sub-partitions), then per-warp state
constexpr int TC_WA = 0, TC_WSC = 32, TC_TW1 = 64, TC_TW2 = 96, TC_TWR = 128, TC_AS1 = 144, TC_AS2 = 176;
// conjugates of the three twiddle tables (fft_regs.cuh: cmul2t), then the per-warp state
constexpr int TC_TW1C = 208, TC_TW2C = 240, TC_TWRC = 272, TC_WARP = 288;
constexpr bool HC = true;
// per warp (VV = values per lane): momentum spectrum `pre` 2 VV words, kept part of y 2 VV, magnitude row VV
constexpr int TMEM_COLS = 512;
// float2 of shared memory per signal: u of the active frames (double buffered), u of the kept frames, the output
// carry (one frame = VV rows of 32 lanes = M float2 each), and the two FFT exchange buffers of every warp
constexpr int sig_f2(int m) { return 2 * NAMAX * m + KEEP * m + m + NAMAX * 2 * m; }

// Named barrier over the `na` active frame groups of a signal (na * LANES threads; immediate thread counts).
template <int LANES>
__device__ __forceinline__ void sig_sync(int bar_id, int na) {
    switch (na) {
        case 1: asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "n"(LANES) : "memory"); break;
        case 2: asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "n"(2 * LANES) : "memory"); break;
        case 3: asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "n"(3 * LANES) : "memory"); break;
        default: asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "n"(4 * LANES) : "memory"); break;
    }
}

// Synchronise the warps that share a frame (named barrier) or just the warp.
template <int LANES>
__device__ __forceinline__ void frame_sync(int bar_id) {
    if constexpr (LANES == 32) __syncwarp();
    else asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "n"(LANES) : "memory");
}

// LANES lanes (LANES / 32 warps) per frame and VV complex values per lane: <32, 16> n_fft = 1024, <32, 8> n_fft = 512,
// <64, 16> n_fft = 2048; SIGS signals per CTA (SIGS x 4 frame slots)
template <int LANES, int VV, int SIGS>
__global__ void __launch_bounds__(SIGS * NAMAX * LANES, 1) rtisi_fast_kernel(const RArgs a) {
    using C = Cfg<LANES, VV>;
    constexpr int V = VV;                          // shadows wfast::V
    constexpr int M = C::M, HOP = C::HOP, RC = C::RC, HP = VV / 4;
    constexpr int ROWS = M;                        // float2 per frame: VV rows of LANES lanes
    constexpr int SIG_F2 = sig_f2(M);
    constexpr int G = LANES / 32;                  // warps per frame
    constexpr int WARPS = SIGS * NAMAX * G;
    constexpr int TC_PRE = 0, TC_YK = 2 * V, TC_MAG = 4 * V, TC_PER_WARP = 5 * V;
    static_assert(TC_WARP + ((WARPS + 3) / 4) * TC_PER_WARP <= TMEM_COLS, "TMEM columns");
    static_assert(1 + SIGS + SIGS * NAMAX <= 16 || G == 1, "named barriers");
    // bin offsets of the lane's VV bins (gl_warp_core.cuh: slot j -> bins l + 64 j and M - l - 64 j; lane 0 special)
    struct Bins {
        int pl, ph, ql, qh, q0;
        __device__ __forceinline__ int operator()(int e) const {
            const int j = e >> 1;
            return (e & 1) ? (j == 0 ? q0 : (j >= RC / 2 ? qh : ql) - 2 * LANES * j) : (j >= RC / 2 ? ph : pl) + 2 * LANES * j;
        }
    };
    extern __shared__ __align__(16) float2 sm[];
    __shared__ unsigned s_tmem_base;
    // compute-sanitizer's synccheck (12.9) reports "Missing init, barrier at shared address 0x0" for a kernel that
    // uses tcgen05.alloc but owns no mbarrier; this initialised, otherwise unused one keeps the tool usable here
    __shared__ __align__(8) unsigned long long s_tool_bar;
    __shared__ float2 s_ws[ROWS];                  // synthesis window pairs [row][lane] (commit only)
    const int tid = threadIdx.x, warp = tid >> 5;
    const int sig = warp / (NAMAX * G);            // signal slot inside the CTA
    const int wf = warp % (NAMAX * G);             // warp inside the signal
    const int p = wf / G;                          // physical frame slot of this warp's frame group
    const int l = 32 * (wf % G) + (tid & 31);      // lane inside the frame group, 0 .. LANES-1 (wf % G == warp % G)
    const int NA = a.LA + 1;
    const int fbar = 1 + SIGS + sig * NAMAX + p;   // named barrier of the frame group (G > 1)
    if (threadIdx.x == 0) mbar_init((unsigned)__cvta_generic_to_shared(&s_tool_bar), 1);
    if (warp == 0) tmem_alloc(&s_tmem_base, TMEM_COLS);
    for (int i = tid; i < ROWS; i += WARPS * 32) {
        const int row = i / LANES, ll = i % LANES;
        s_ws[i] = f2(a.ws[2 * LANES * row + 2 * ll], a.ws[2 * LANES * row + 2 * ll + 1]);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const unsigned tlane = s_tmem_base + ((unsigned)(32 * (warp & 3)) << 16);
    if (warp < 4) {
        float t[32];
        auto window_pairs = [&](const float* w, float scale, unsigned col) {
#pragma unroll
            for (int i = 0; i < V; ++i) { t[2 * i] = scale * w[2 * LANES * i + 2 * l]; t[2 * i + 1] = scale * w[2 * LANES * i + 2 * l + 1]; }
            tmem_stw<2 * V>(tlane + col, t);
        };
        window_pairs(a.wa, 0.5f, TC_WA);
        window_pairs(a.ws, a.coef, TC_WSC);
#pragma unroll
        for (int i = 0; i < V; ++i) {
            const float2 w = a.tw[((l + LANES * (i / C::R1)) * (i % C::R1)) & (M - 1)];
            t[2 * i] = w.x; t[2 * i + 1] = w.y;
        }
        tmem_stw<2 * V>(tlane + TC_TW1, t);
#pragma unroll
        for (int kb = 0; kb < C::R2; ++kb) {
            const float2 w = a.tw[(C::R1 * (l & (C::RC - 1)) * kb) & (M - 1)];
            t[2 * kb] = w.x; t[2 * kb + 1] = w.y;
        }
        tmem_stw<2 * C::R2>(tlane + TC_TW2, t);
#pragma unroll
        for (int j = 0; j < RC; ++j) {
            const int k = slot_bin_rt<LANES, VV>(l, j);
            float2 w;
            if (k <= M / 2) w = a.twr[k];
            else { w = a.twr[M - k]; w.x = -w.x; }
            t[2 * j] = w.x; t[2 * j + 1] = w.y;
        }
        tmem_stw<2 * RC>(tlane + TC_TWR, t);
#pragma unroll
        for (int j = 0; j < RC; ++j) t[2 * j + 1] = -t[2 * j + 1];
        tmem_stw<2 * RC>(tlane + TC_TWRC, t);
#pragma unroll
        for (int i = 0; i < V; ++i) {
            const float2 w = a.tw[((l + LANES * (i / C::R1)) * (i % C::R1)) & (M - 1)];
            t[2 * i] = w.x; t[2 * i + 1] = -w.y;
        }
        tmem_stw<2 * V>(tlane + TC_TW1C, t);
#pragma unroll
        for (int kb = 0; kb < C::R2; ++kb) {
            const float2 w = a.tw[(C::R1 * (l & (C::RC - 1)) * kb) & (M - 1)];
            t[2 * kb] = w.x; t[2 * kb + 1] = -w.y;
        }
        tmem_stw<2 * C::R2>(tlane + TC_TW2C, t);
        if (a.asymmetric) {
            window_pairs(a.asym1, 0.5f, TC_AS1);
            window_pairs(a.asym2, 0.5f, TC_AS2);
        }
        tmem_wait_st();
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    const int b = blockIdx.x * SIGS + sig;
    if (b < a.B && p < NA) {
        const unsigned twarp = tlane + TC_WARP + TC_PER_WARP * (warp >> 2);
        float2* base = sm + sig * SIG_F2;
        float2* U = base;                              // [2][NAMAX][ROWS]
        float2* Uk = U + 2 * NAMAX * ROWS;             // [KEEP][ROWS]
        float2* carry = Uk + KEEP * ROWS;              // [ROWS]
        float2* e1 = carry + ROWS + p * 2 * M;
        float2* e2 = e1 + M;
        const int bar_id = 1 + sig;
        const int hi_adj = l == 0 ? -(RC - 1) * LANES : 0;
        const Bins bin{l, l + hi_adj, M - l, M - l - hi_adj, l == 0 ? M / 2 : M - l};
        float* xo = a.x_out + (long long)b * a.x_len - a.x0;     // indexed by absolute sample

        // ---- everything zero (methods.py:353-358)
        float2 v[V];
#pragma unroll
        for (int i = 0; i < V; ++i) v[i] = f2(0.f, 0.f);
        {
            float z[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) z[i] = 0.f;
            tmem_stw<2 * V>(twarp + TC_PRE, z);
            tmem_stw<V>(twarp + TC_MAG, z);            // frames that precede the spectrogram have zero magnitude (:339)
        }
        float2 pre_nyq = f2(0.f, 0.f);
        for (int i = p * LANES + l; i < KEEP * ROWS + ROWS; i += LANES * NA) Uk[i] = f2(0.f, 0.f);  // kept frames and carry
        sig_sync<LANES>(bar_id, NA);
        int kslot = 0;                                 // kept ring: logical kept frame f (0 = oldest) = slot (kslot + f) % KEEP
        float mag_nyq = 0.f;

        // canonical state of this signal (natural sample / bin order, logical frame order)
        constexpr int N = 2 * M, F = M + 1;
        float* st_frames = a.state ? a.state + (size_t)b * a.state_elems : nullptr;
        float* st_pre = st_frames + (size_t)NA * N;
        float* st_kept = st_pre + 2 * (size_t)NA * F;
        float* st_carry = st_kept + (size_t)KEEP * N;
        if (a.step_begin > 0) {
            // ---- resume before outer step step_begin: this warp's frame, its momentum spectrum and magnitude row
            int la0 = (p - a.step_begin) % NA; if (la0 < 0) la0 += NA;
            const float2* fr = reinterpret_cast<const float2*>(st_frames + (size_t)la0 * N);
#pragma unroll
            for (int r = 0; r < V; ++r) v[r] = fr[r * LANES + l];                  // pair LANES r + l
            {
                float pre[2 * V];
                const float2* pr = reinterpret_cast<const float2*>(st_pre + 2 * (size_t)la0 * F);
#pragma unroll
                for (int e = 0; e < V; ++e) { const float2 q = pr[bin(e)]; pre[2 * e] = q.x; pre[2 * e + 1] = q.y; }
                tmem_stw<2 * V>(twarp + TC_PRE, pre);
                pre_nyq = l == 0 ? pr[M] : f2(0.f, 0.f);
            }
            if (la0 != a.LA) {            // (the newest frame fetches its row when the step starts)
                const int t_frame = a.step_begin + la0 - a.LA;
                float mg[V];
                const bool inside = t_frame >= 0 && t_frame < a.T;
                const float* mrow = a.mag + ((long long)b * a.n_rows + (inside ? t_frame - a.frame0 : 0)) * M;
#pragma unroll
                for (int e = 0; e < V; ++e) mg[e] = inside ? __ldg(mrow + bin(e)) : 0.f;
                mag_nyq = (inside && l == 0) ? __ldg(a.mag_nyq + (long long)b * a.n_rows + t_frame - a.frame0) : 0.f;
                tmem_stw<V>(twarp + TC_MAG, mg);
            }
            const float2* kp = reinterpret_cast<const float2*>(st_kept);
            for (int i = p * LANES + l; i < KEEP * ROWS; i += LANES * NA) Uk[i] = kp[i];
            const float2* cp = reinterpret_cast<const float2*>(st_carry);
            for (int i = p * LANES + l; i < ROWS; i += LANES * NA) carry[i] = cp[i];
            tmem_wait_st();
            sig_sync<LANES>(bar_id, NA);
        }

        for (int i = a.step_begin; i < a.step_end; ++i) {
            int la = (p - i) % NA; if (la < 0) la += NA;          // logical index of this warp's frame
            const int t_frame = i + la - a.LA;                    // spectrogram frame it reconstructs
            const bool newest = la == a.LA;
            if (newest) {
                // a new frame is born in this warp: fetch its magnitude row (zero outside the spectrogram, :339)
                float mg[V];
                const bool inside = t_frame >= 0 && t_frame < a.T;
                const float* mrow = a.mag + ((long long)b * a.n_rows + (inside ? t_frame - a.frame0 : 0)) * M;
#pragma unroll
                for (int e = 0; e < V; ++e) mg[e] = inside ? __ldg(mrow + bin(e)) : 0.f;
                mag_nyq = (inside && l == 0) ? __ldg(a.mag_nyq + (long long)b * a.n_rows + t_frame - a.frame0) : 0.f;
                tmem_stw<V>(twarp + TC_MAG, mg);
                if (i == 0) {
                    // zero-phase start: the newest frame = irfft(first magnitude frame + 0j) (:353-358)
                    struct IO0 {
                        const float* mg; float mn;
                        __device__ __forceinline__ float2 s0(int e) const { return f2(e < 0 ? mn : mg[e], 0.f); }
                    } io0{mg, mag_nyq};
                    float2 A[RC], Bv[RC], twr[RC];
                    tmem_ldw<2 * RC>(tlane + TC_TWR, reinterpret_cast<float*>(twr));
                    spectrum_pairs<VV>(l, A, Bv, twr, io0);
                    inv_pass3<LANES, VV>(l, A, Bv, e2);
                    frame_sync<LANES>(fbar);
                    float2 tw2[C::R2];
                    tmem_ldw<2 * C::R2>(tlane + TC_TW2, reinterpret_cast<float*>(tw2));
                    inv_pass2<LANES, VV>(l, e2, tw2, e1);
                    frame_sync<LANES>(fbar);
                    float2 tw1[V];
                    tmem_ldw<2 * V>(tlane + TC_TW1, reinterpret_cast<float*>(tw1));
                    inv_pass1<LANES, VV>(l, e1, tw1, v);
                    frame_sync<LANES>(fbar);
                }
            }
            // ---- part of this frame's y that comes from the kept frames: constant over the inner iterations.
            // kept frame f (0 = oldest) starts (KEEP - f) hops before active frame 0: row i' of this frame is row
            // i' + HP (la + KEEP - f) of the kept frame (HP = rows per hop).
            {
                float2 yk[V];
#pragma unroll
                for (int r = 0; r < V; ++r) yk[r] = f2(0.f, 0.f);
#pragma unroll
                for (int f = 0; f < KEEP; ++f) {
                    const int shift = HP * (la + KEEP - f);          // warp-uniform
                    const float2* src = Uk + ((kslot + f) % KEEP) * ROWS + l;
#pragma unroll
                    for (int r = 0; r < V - HP; ++r)                // a kept frame is at least one hop older
                        if (r + shift < V) yk[r] = yk[r] + src[(r + shift) * LANES];
                }
                tmem_wait_st();
                tmem_stw<2 * V>(twarp + TC_YK, reinterpret_cast<const float*>(yk));
                tmem_wait_st();
            }

            for (int j = 0; j < a.max_iter; ++j) {
                // ---- publish u = frame * w * c (:365-368), double buffered over j
                float2* Ub = U + (j & 1) * NAMAX * ROWS;
                float2 y[V];
                {
                    float2 w[V];
                    tmem_ldw<2 * V>(tlane + TC_WSC, reinterpret_cast<float*>(w));
#pragma unroll
                    for (int r = 0; r < V; ++r) {
                        y[r] = pmul(v[r], w[r]);
                        Ub[p * ROWS + r * LANES + l] = y[r];
                    }
                }
                sig_sync<LANES>(bar_id, NA);
                // ---- this frame of the overlap-add: own u + kept part + the other active frames, shifted by HP
                // rows per frame of distance (row r of this frame = row r - HP d of the frame d positions later)
                {
                    float2 yk[V];
                    tmem_ldw<2 * V>(twarp + TC_YK, reinterpret_cast<float*>(yk));
#pragma unroll
                    for (int r = 0; r < V; ++r) y[r] = y[r] + yk[r];
                }
#pragma unroll
                for (int d = -3; d <= 3; ++d) {
                    if (d == 0) continue;
                    const int lo = la + d;                          // logical index of the other frame (warp-uniform)
                    if (lo < 0 || lo > a.LA) continue;
                    int po = (lo + i) % NA;                         // its physical slot
                    const float2* src = Ub + po * ROWS + l;
#pragma unroll
                    for (int r = 0; r < V; ++r)
                        if (r - HP * d >= 0 && r - HP * d < V) y[r] = y[r] + src[(r - HP * d) * LANES];
                }
                // ---- analysis window (:371-385)
                {
                    float2 w[V];
                    const unsigned wcol = (a.asymmetric && newest) ? (j ? TC_AS2 : TC_AS1) : TC_WA;
                    tmem_ldw<2 * V>(tlane + wcol, reinterpret_cast<float*>(w));
#pragma unroll
                    for (int r = 0; r < V; ++r) y[r] = pmul(y[r], w[r]);
                }
                // momentum state and magnitudes of this frame's bins (element e of gl_warp_core.cuh)
                struct IO {
                    float2* pre; const float* mg; float2 pn; float mn;
                    __device__ __forceinline__ float2 s0(int e) const { return e < 0 ? pn : pre[e]; }
                    __device__ __forceinline__ float2 s1(int) const { return f2(0.f, 0.f); }
                    __device__ __forceinline__ float mag(int e) const { return e < 0 ? mn : mg[e]; }
                    __device__ __forceinline__ void put(int e, float2 q, float2) { if (e < 0) pn = q; else pre[e] = q; }
                };
                const bool mom = j > 0 || (i > 0 && !newest);
                {
                    float2 tw1[V], tw1c[V];
                    tmem_ldw<2 * V>(tlane + TC_TW1, reinterpret_cast<float*>(tw1));
                    tmem_ldw<2 * V>(tlane + TC_TW1C, reinterpret_cast<float*>(tw1c));
                    fwd_pass1<LANES, VV, HC>(l, y, tw1, e1, tw1c);
                }
                frame_sync<LANES>(fbar);
                {
                    float2 tw2[C::R2], tw2c[C::R2];
                    tmem_ldw<2 * C::R2>(tlane + TC_TW2, reinterpret_cast<float*>(tw2));
                    tmem_ldw<2 * C::R2>(tlane + TC_TW2C, reinterpret_cast<float*>(tw2c));
                    fwd_pass2<LANES, VV, HC>(l, e1, tw2, e2, tw2c);
                }
                frame_sync<LANES>(fbar);
                float2 A[RC], Bv[RC];
                fwd_pass3<LANES, VV>(l, e2, A, Bv);
                // ---- momentum (:387-392), pre <- S, projection (:394-396)
                {
                    float2 pre[V];
                    float mg[V];
                    tmem_wait_st();
                    tmem_ldw<2 * V>(twarp + TC_PRE, reinterpret_cast<float*>(pre));
                    tmem_ldw<V>(twarp + TC_MAG, mg);
                    IO io{pre, mg, pre_nyq, mag_nyq};
                    float2 twr[RC], twrc[RC];
                    tmem_ldw<2 * RC>(tlane + TC_TWR, reinterpret_cast<float*>(twr));
                    tmem_ldw<2 * RC>(tlane + TC_TWRC, reinterpret_cast<float*>(twrc));
                    float ds = 0.f, es = 0.f;
                    pointwise<OP_GL, false, VV, HC>(l, A, Bv, twr, io, mom ? a.lr : 0.f, 0.f, ds, es, twrc);
                    pre_nyq = io.pn;
                    tmem_stw<2 * V>(twarp + TC_PRE, reinterpret_cast<const float*>(pre));
                }
                frame_sync<LANES>(fbar);
                inv_pass3<LANES, VV>(l, A, Bv, e2);
                frame_sync<LANES>(fbar);
                {
                    float2 tw2[C::R2], tw2c[C::R2];
                    tmem_ldw<2 * C::R2>(tlane + TC_TW2, reinterpret_cast<float*>(tw2));
                    tmem_ldw<2 * C::R2>(tlane + TC_TW2C, reinterpret_cast<float*>(tw2c));
                    inv_pass2<LANES, VV, HC>(l, e2, tw2, e1, tw2c);
                }
                frame_sync<LANES>(fbar);
                {
                    float2 tw1[V], tw1c[V];
                    tmem_ldw<2 * V>(tlane + TC_TW1, reinterpret_cast<float*>(tw1));
                    tmem_ldw<2 * V>(tlane + TC_TW1C, reinterpret_cast<float*>(tw1c));
                    inv_pass1<LANES, VV, HC>(l, e1, tw1, v, tw1c);
                }
                frame_sync<LANES>(fbar);
            }

            // ---- commit the oldest active frame (:401-404) and fuse the final overlap-add (:406-408)
            if (la == 0) {
                const int t = i - a.LA;                             // index of the committed frame in the output
                if (t >= 0) {
                    float2 c[V];
#pragma unroll
                    for (int r = 0; r < V; ++r) {
                        const float2 w = s_ws[r * LANES + l];
                        c[r] = pfma(v[r], w, carry[r * LANES + l]);
                    }
                    const bool last = a.final && t == a.T - 1;      // the last frame flushes the whole carry
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        if (k == 0 || last) {
                            const long long m0 = (long long)(t + k) * HOP - a.P;
                            if (m0 >= a.x0 && m0 + HOP <= a.x0 + a.x_len) {
#pragma unroll
                                for (int r = 0; r < HP; ++r) {
                                    const float2 ie = __ldg(reinterpret_cast<const float2*>(a.inv_env + (m0 - a.x0) + 2 * LANES * r + 2 * l));
                                    const float2 val = c[HP * k + r];
                                    *reinterpret_cast<float2*>(xo + m0 + 2 * LANES * r + 2 * l) = pmul(val, ie);
                                }
                            }
                        }
                    }
#pragma unroll
                    for (int r = 0; r < V; ++r) carry[r * LANES + l] = r + HP < V ? c[r + HP] : f2(0.f, 0.f);
                }
                // the committed frame replaces the oldest kept frame (stored as u = frame * w * c)
                {
                    float2 w[V];
                    tmem_ldw<2 * V>(tlane + TC_WSC, reinterpret_cast<float*>(w));
                    float2* dst = Uk + kslot * ROWS + l;
#pragma unroll
                    for (int r = 0; r < V; ++r) dst[r * LANES] = pmul(v[r], w[r]);
                }
                // this warp's frame slot becomes the newest (all-zero) active frame of the next step
#pragma unroll
                for (int r = 0; r < V; ++r) v[r] = f2(0.f, 0.f);
            }
            kslot = (kslot + 1) % KEEP;
            sig_sync<LANES>(bar_id, NA);              // the kept ring and the carry are in place for the next step
        }
        if (a.step_begin == a.step_end && p == 0) {
            // a final launch with no step left (look_ahead = 0, frame T-1 committed by an earlier launch): release
            // the carry that commit shifted by one hop -- the blocks k = 1 .. 3 its flush would have written
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const long long m0 = (long long)(a.T + k) * HOP - a.P;
                if (m0 >= a.x0 && m0 + HOP <= a.x0 + a.x_len) {
#pragma unroll
                    for (int r = 0; r < HP; ++r) {
                        const float2 ie = __ldg(reinterpret_cast<const float2*>(a.inv_env + (m0 - a.x0) + 2 * LANES * r + 2 * l));
                        *reinterpret_cast<float2*>(xo + m0 + 2 * LANES * r + 2 * l) = pmul(carry[(HP * k + r) * LANES + l], ie);
                    }
                }
            }
        }
        if (a.state && !(a.final && a.step_end == a.T + a.LA)) {
            // ---- save the state before outer step step_end
            int la1 = (p - a.step_end) % NA; if (la1 < 0) la1 += NA;
            float2* fr = reinterpret_cast<float2*>(st_frames + (size_t)la1 * N);
#pragma unroll
            for (int r = 0; r < V; ++r) fr[r * LANES + l] = v[r];
            {
                float pre[2 * V];
                tmem_wait_st();
                tmem_ldw<2 * V>(twarp + TC_PRE, pre);
                float2* pr = reinterpret_cast<float2*>(st_pre + 2 * (size_t)la1 * F);
                const bool keep = la1 != a.LA;        // the newest frame's momentum is never used: saved as zero
#pragma unroll
                for (int e = 0; e < V; ++e) pr[bin(e)] = keep ? f2(pre[2 * e], pre[2 * e + 1]) : f2(0.f, 0.f);
                if (l == 0) pr[M] = keep ? pre_nyq : f2(0.f, 0.f);
            }
            float2* kp = reinterpret_cast<float2*>(st_kept);
            for (int i = p * LANES + l; i < KEEP * ROWS; i += LANES * NA) {
                const int f = i / ROWS, r = i - f * ROWS;
                kp[i] = Uk[((kslot + f) % KEEP) * ROWS + r];
            }
            float2* cp = reinterpret_cast<float2*>(st_carry);
            for (int i = p * LANES + l; i < ROWS; i += LANES * NA) cp[i] = carry[i];
        }
        tmem_wait_st();
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) tmem_dealloc(s_tmem_base, TMEM_COLS);
}

template <int LANES, int VV, int SIGS>
static int launch(const RArgs& a, cudaStream_t st) {
    const size_t smem = (size_t)SIGS * sig_f2(Cfg<LANES, VV>::M) * sizeof(float2);
    cudaError_t e = cudaFuncSetAttribute(rtisi_fast_kernel<LANES, VV, SIGS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    rtisi_fast_kernel<LANES, VV, SIGS><<<(a.B + SIGS - 1) / SIGS, SIGS * NAMAX * LANES, smem, st>>>(a);
    return (int)cudaGetLastError();
}

}  // namespace rfast

// Returns SPECINV_ERR_UNSUPPORTED when the shape is not the one this kernel is specialised for.
int rtisi_fast(const specinv_desc* d, const Dims& dm, const void* plan, const void* mag_main, const void* mag_nyq,
               void* x_out, const RtisiWindow& win, const void* asym1, const void* asym2, int look_ahead, int asymmetric,
               int max_iter, double alpha, double synth_coeff, int step_begin, int step_end, void* state, cudaStream_t st) {
    if (d->dtype != SPECINV_F32 || !d->onesided || d->hop * 4 != d->n_fft ||
        (d->n_fft != 2048 && d->n_fft != 1024 && d->n_fft != 512))
        return SPECINV_ERR_UNSUPPORTED;
    const int LA = look_ahead < 0 ? dm.K : look_ahead;
    if (LA > 3 || dm.K != rfast::KEEP) return SPECINV_ERR_UNSUPPORTED;
    rfast::RArgs a{};
    const PlanLayout pl = plan_layout(dm, d->dtype);
    const char* p = (const char*)plan;
    a.tw = (const float2*)(p + pl.tw); a.twr = (const float2*)(p + pl.twr);
    a.wa = (const float*)(p + pl.wa); a.ws = (const float*)(p + pl.ws); a.inv_env = (const float*)win.inv_env;
    a.asym1 = (const float*)asym1; a.asym2 = (const float*)asym2;
    a.mag = (const float*)mag_main; a.mag_nyq = (const float*)mag_nyq; a.x_out = (float*)x_out;
    a.coef = (float)synth_coeff; a.lr = (float)(alpha / (1.0 + alpha));
    a.B = dm.B; a.T = dm.T; a.P = dm.P; a.LA = LA; a.max_iter = max_iter; a.asymmetric = asymmetric;
    a.frame0 = win.frame0; a.n_rows = win.n_rows; a.final = win.final; a.x0 = win.x0; a.x_len = win.x_len;
    a.step_begin = step_begin; a.step_end = step_end; a.state = (float*)state;
    a.state_elems = (size_t)(LA + 1) * dm.N + 2 * (size_t)(LA + 1) * (dm.M + 1) + (size_t)dm.K * dm.N + dm.N;
    // Signals per CTA: as few as still fit the batch into one wave of CTAs (the kernel is latency-bound, so a signal
    // runs fastest when its warps share an SM with as few others as possible).
    int sms = 0, dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
        return SPECINV_ERR_NO_DEVICE;
    if (d->n_fft == 2048) return rfast::launch<64, 16, 1>(a, st);       // two warps per frame, one signal per CTA
    // n_fft = 1024 on one warp per frame: two warps at 8 values per lane measured slower (62.6 ms against 57.2 ms at
    // cfg3, DESIGN.md section 3.3)
    if (d->n_fft == 1024) return dm.B <= sms ? rfast::launch<32, 16, 1>(a, st) : rfast::launch<32, 16, 2>(a, st);
    return dm.B <= sms ? rfast::launch<32, 8, 1>(a, st) : dm.B <= 2 * sms ? rfast::launch<32, 8, 2>(a, st)
                                                                          : rfast::launch<32, 8, 4>(a, st);
}

}  // namespace specinv
