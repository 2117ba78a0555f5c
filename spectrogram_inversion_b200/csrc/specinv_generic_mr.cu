// Generic fused tile kernels on the mixed-radix FFT of mixed_radix.cuh: STFT, ISTFT, one Griffin-Lim iteration, one
// ADMM iteration for ANY even n_fft whose half M = n_fft / 2 factors into 2, 3, 5, 7, 11, 13 (400 = torchaudio's
// default, 600, 1000, 1536 ...; the reference infers n_fft from the bin count, methods.py:65-68), every hop, fp32 /
// fp64, every torch.stft option the reference forwards.
//
// Same tile structure as specinv_generic.cu (a CTA owns consecutive frames of one signal plus K recomputed halo
// frames, frames stay in shared memory, gather overlap-add, no atomics), but the transforms are run by TEAMS: the
// tile's frames are dealt to teams of 1 .. 16 warps, and a team takes its frames through
//     forward passes -> point-wise update / projection on the (k, M-k) pairs -> inverse passes
// on its own, synchronising only itself (__syncwarp, or a named barrier for multi-warp teams).  The CTA meets twice:
// after the frames are loaded and before the overlap-add.  Warps of different teams drift apart, so the global-memory
// latency of one team's point-wise stage (state / magnitude rows) hides behind the others' butterflies, and two CTAs
// per SM overlap the load / store phases.
//
// Replaces, per iteration, torch.stft + ~8 point-wise kernels + fft.irfft + conv_transpose1d with a dense
// diag(window) weight of the reference (methods.py:241-248, :464-477, :127-132).

#include "specinv_common.cuh"
#include "generic_tile.cuh"
#include "generic_fft.cuh"
#include "mixed_radix.cuh"

namespace specinv {

struct MrLaunch {
    int team_warps;        // warps per team (power of two)
    int frames_cap;        // frames the shared-memory tile holds (owned + halo)
    int Mp;                // padded complex elements per frame
    unsigned magic_M;      // ceil(2^32 / M)
    unsigned magic_npair;  // ceil(2^32 / (M/2 + 1))
    unsigned magic_np1;    // ceil(2^32 / (M/2)): the pairs k = 1 .. M/2
    unsigned magic_hop;    // ceil(2^32 / hop), or 0: divide (hop == 1, or tile positions * hop would overflow 32 bits)
};

template <typename T, int OP>
__global__ void __launch_bounds__(sizeof(T) == 8 ? 256 : 512, 2) mr_tile_kernel(const TileArgs a, const mr::Plan mp, const MrLaunch ml) {
    using C = cx_t<T>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    C* wb = reinterpret_cast<C*>(smem_raw);
    unsigned short* perm = reinterpret_cast<unsigned short*>(wb + (size_t)ml.frames_cap * ml.Mp);

    const Dims& dm = a.dm;
    const int M = dm.M, N = dm.N, hop = dm.hop, Mp = ml.Mp;
    const int b = blockIdx.y;
    const int t0 = blockIdx.x * a.tile_frames;
    const int t1 = min(dm.T, t0 + a.tile_frames);
    const int f0 = (OP == OP_STFT) ? t0 : max(0, t0 - dm.K);
    const int nfr = t1 - f0;
    const int tid = threadIdx.x, NT = blockDim.x;

    const C* __restrict__ tw = (const C*)a.tw;
    const C* __restrict__ twr = (const C*)a.twr;
    const T* __restrict__ wa = (const T*)a.wa;
    const T* __restrict__ ws = (const T*)a.ws;

    // padded position of bin k after the forward passes
    for (int k = tid; k < M; k += NT) perm[k] = (unsigned short)mr::padidx(mr::mr_position(mp, k));

    // ---- A: frame + analysis window: z[n] = x[2n] w[2n] + i x[2n+1] w[2n+1] ----------------------------------
    if constexpr (OP != OP_ISTFT) {
        const T* __restrict__ x = (const T*)a.x_in + (long long)b * dm.L;
        const long long base = (long long)f0 * hop;
        const bool interior = base >= dm.P && base + (long long)(nfr - 1) * hop + N <= dm.P + dm.L;
        const int total = nfr * M;
        // interior tile, even hop, aligned rows: a sample pair and its window pair are one vector load each
        const bool vec = interior && (hop & 1) == 0 && (((uintptr_t)(x + (base - dm.P))) & (2 * sizeof(T) - 1)) == 0;
        if (vec) {
            const C* __restrict__ x2 = reinterpret_cast<const C*>(x + (base - dm.P));
            const C* __restrict__ wa2 = reinterpret_cast<const C*>(wa);
            const int hop2 = hop >> 1;
#pragma unroll 4
            for (int idx = tid; idx < total; idx += NT) {
                const int f = mr::fdiv(idx, ml.magic_M), n = idx - f * M;
                const C v = __ldg(x2 + (size_t)f * hop2 + n), w = __ldg(wa2 + n);
                wb[f * Mp + mr::padidx(n)] = mk<T>(v.x * w.x, v.y * w.y);
            }
        } else
#pragma unroll 4
        for (int idx = tid; idx < total; idx += NT) {
            const int f = mr::fdiv(idx, ml.magic_M), n = idx - f * M;
            const long long pp = base + (long long)f * hop + 2 * n;
            T v0, v1;
            if (interior) {
                v0 = __ldg(x + (pp - dm.P)); v1 = __ldg(x + (pp - dm.P + 1));
            } else {
                const long long i0 = pad_index(pp, dm.P, dm.L, dm.pad_mode);
                const long long i1 = pad_index(pp + 1, dm.P, dm.L, dm.pad_mode);
                v0 = i0 >= 0 ? __ldg(x + i0) : T(0);
                v1 = i1 >= 0 ? __ldg(x + i1) : T(0);
            }
            wb[f * Mp + mr::padidx(n)] = mk<T>(v0 * __ldg(wa + 2 * n), v1 * __ldg(wa + 2 * n + 1));
        }
    }
    __syncthreads();

    // ---- the team's frames ------------------------------------------------------------------------------------
    const int G = ml.team_warps;
    const int team = (tid >> 5) / G, nteams = (NT >> 5) / G;
    const int tnt = G * 32, ttid = tid - team * tnt;
    const int per = (nfr + nteams - 1) / nteams;
    const int fa = min(nfr, team * per), nf = min(nfr, fa + per) - fa;
    C* tb = wb + (size_t)fa * Mp;
    auto team_sync = [&]() {
        if (G == 1) __syncwarp();
        else asm volatile("bar.sync %0, %1;" ::"r"(team + 1), "r"(tnt) : "memory");
    };

    // ---- B: forward passes (natural -> digit-reversed) ---------------------------------------------------------
    if constexpr (OP != OP_ISTFT) {
        for (int s = 0; s < mp.nst; ++s) {
            mr::pass<T, false>(tb, nf, Mp, mp, s, tw, ttid, tnt);
            team_sync();
        }
    }

    // ---- C: real-FFT post-process, point-wise update, inverse pre-process (pairs k, M-k) ------------------------
    // Two pairs per thread and trip: the global loads of both (state rows, magnitudes: up to 10 per pair) are issued
    // before any arithmetic, so a thread keeps ~20 loads in flight instead of stalling pair after pair (fp32).
    T dsum = T(0), esum = T(0);
    const bool want_sums = a.sums != nullptr;
    {
        const int npair = M / 2 + 1;
        const int total = nf * npair;
        struct Pair { int k, pA, pB; bool owned; long long fr; C* v; };
        auto locate = [&](int idx) {
            Pair p;
            const int f = mr::fdiv(idx, ml.magic_npair);
            p.k = idx - f * npair;
            const int t = f0 + fa + f;
            p.owned = t >= t0;
            p.fr = (long long)b * dm.T + t;
            p.v = tb + (size_t)f * Mp;
            const int kB = M - p.k;
            p.pA = perm[p.k]; p.pB = perm[kB == M ? 0 : kB];
            return p;
        };
        auto finish = [&](const Pair& p, C hA, C hB, C w) {
            if constexpr (OP != OP_STFT) {
                if (p.k == 0) { hA.y = T(0); hB.y = T(0); }  // C2R ignores Im(DC), Im(Nyquist)
                C zA, zB;
                irfft_pre_pair<T>(hA, hB, w, zA, zB);
                p.v[p.pA] = zA;
                if (M - p.k != p.k && p.k != 0) p.v[p.pB] = zB;
            }
        };
        if (dm.onesided) {
            // pairs k = 1 .. M/2: never the Nyquist bin (BinIO<T, false>: one row offset per frame, no select between the
            // main and the Nyquist arrays); the (0, M) pair of every frame follows
            constexpr bool TWO = sizeof(T) == 4;        // fp64: one pair (two would spill the 64-register budget)
            const int np1 = npair - 1, total1 = nf * np1;
            const unsigned magic_np1 = ml.magic_np1;
            auto locate1 = [&](int idx) {
                Pair p;
                const int f = mr::fdiv(idx, magic_np1);
                p.k = idx - f * np1 + 1;
                const int t = f0 + fa + f;
                p.owned = t >= t0;
                p.fr = (long long)b * dm.T + t;
                p.v = tb + (size_t)f * Mp;
                p.pA = perm[p.k]; p.pB = perm[M - p.k];
                return p;
            };
            using IO1 = BinIO<T, false>;
            for (int idx = ttid; idx < total1; idx += TWO ? 2 * tnt : tnt) {
                const bool two = TWO && idx + tnt < total1;
                const Pair p0 = locate1(idx), p1 = locate1(two ? idx + tnt : idx);
                const IO1 io0(a, p0.fr), io1(a, p1.fr);
                const BinIn<T> a0 = bin_load<T, OP>(a, io0, p0.k), b0 = bin_load<T, OP>(a, io0, M - p0.k);
                const BinIn<T> a1 = bin_load<T, OP>(a, io1, p1.k), b1 = bin_load<T, OP>(a, io1, M - p1.k);
                const C w0 = __ldg(twr + p0.k), w1 = __ldg(twr + p1.k);
                {
                    C sA = mk<T>(T(0), T(0)), sB = sA;
                    if constexpr (OP != OP_ISTFT) rfft_post_pair<T>(p0.v[p0.pA], p0.v[p0.pB], w0, sA, sB);
                    const C hA = bin_apply<T, OP>(a, io0, p0.k, sA, a0, p0.owned, want_sums, dsum, esum);
                    const C hB = (M - p0.k != p0.k) ? bin_apply<T, OP>(a, io0, M - p0.k, sB, b0, p0.owned, want_sums, dsum, esum) : hA;
                    finish(p0, hA, hB, w0);
                }
                if (two) {
                    C sA = mk<T>(T(0), T(0)), sB = sA;
                    if constexpr (OP != OP_ISTFT) rfft_post_pair<T>(p1.v[p1.pA], p1.v[p1.pB], w1, sA, sB);
                    const C hA = bin_apply<T, OP>(a, io1, p1.k, sA, a1, p1.owned, want_sums, dsum, esum);
                    const C hB = (M - p1.k != p1.k) ? bin_apply<T, OP>(a, io1, M - p1.k, sB, b1, p1.owned, want_sums, dsum, esum) : hA;
                    finish(p1, hA, hB, w1);
                }
            }
            for (int f = ttid; f < nf; f += tnt) {      // DC and Nyquist: both read Z[0]
                const Pair p = locate(f * npair);
                const BinIO<T> io(a, p.fr);
                const BinIn<T> iA = bin_load<T, OP>(a, io, 0), iB = bin_load<T, OP>(a, io, M);
                const C w = __ldg(twr);
                C sA = mk<T>(T(0), T(0)), sB = sA;
                if constexpr (OP != OP_ISTFT) rfft_post_pair<T>(p.v[p.pA], p.v[p.pB], w, sA, sB);
                const C hA = bin_apply<T, OP>(a, io, 0, sA, iA, p.owned, want_sums, dsum, esum);
                const C hB = bin_apply<T, OP>(a, io, M, sB, iB, p.owned, want_sums, dsum, esum);
                finish(p, hA, hB, w);
            }
        } else {
            // two-sided: bins kA, kB and their mirrors N-kA, N-kB (= conj of the real-input STFT);
            // ifft(...).real (methods.py:145-146) == irfft of the Hermitian part (p[k]+conj p[N-k])/2
            for (int idx = ttid; idx < total; idx += tnt) {
                const Pair p = locate(idx);
                const int kA = p.k, kB = M - p.k;
                const BinIO<T> io(a, p.fr);
                const BinIn<T> iA = bin_load<T, OP>(a, io, kA), iB = bin_load<T, OP>(a, io, kB);
                const BinIn<T> jA = bin_load<T, OP>(a, io, kA != 0 ? N - kA : kA), jB = bin_load<T, OP>(a, io, kB != M ? N - kB : kB);
                const C w = __ldg(twr + p.k);
                C sA = mk<T>(T(0), T(0)), sB = sA;
                if constexpr (OP != OP_ISTFT) rfft_post_pair<T>(p.v[p.pA], p.v[p.pB], w, sA, sB);
                C hA = bin_apply<T, OP>(a, io, kA, sA, iA, p.owned, want_sums, dsum, esum), hB;
                if (kA != 0) {
                    C m = bin_apply<T, OP>(a, io, N - kA, mk<T>(sA.x, -sA.y), jA, p.owned, want_sums, dsum, esum);
                    hA = mk<T>(T(0.5) * (hA.x + m.x), T(0.5) * (hA.y - m.y));
                }
                if (kB != kA) {
                    hB = bin_apply<T, OP>(a, io, kB, sB, iB, p.owned, want_sums, dsum, esum);
                    if (kB != M) {
                        C m = bin_apply<T, OP>(a, io, N - kB, mk<T>(sB.x, -sB.y), jB, p.owned, want_sums, dsum, esum);
                        hB = mk<T>(T(0.5) * (hB.x + m.x), T(0.5) * (hB.y - m.y));
                    }
                } else {
                    hB = hA;
                }
                finish(p, hA, hB, w);
            }
        }
    }

    if constexpr (OP == OP_GL || OP == OP_GLR || OP == OP_ADMM) {
        if (want_sums) {   // fused metric epilogue: warp reduce, one double atomic pair per warp
            double d = (double)dsum, e = (double)esum;
            for (int o = 16; o > 0; o >>= 1) {
                d += __shfl_xor_sync(0xffffffffu, d, o);
                e += __shfl_xor_sync(0xffffffffu, e, o);
            }
            if ((tid & 31) == 0 && nf > 0) { atomicAdd(a.sums, d); atomicAdd(a.sums + 1, e); }
        }
    }
    if constexpr (OP == OP_STFT) return;
    team_sync();

    // ---- D: inverse passes (digit-reversed -> natural) -----------------------------------------------------------
    for (int s = mp.nst - 1; s >= 0; --s) {
        mr::pass<T, true>(tb, nf, Mp, mp, s, tw, ttid, tnt, s == 0 ? ws : (const T*)nullptr);   // last pass: x synthesis window
        team_sync();
    }
    __syncthreads();

    // ---- E: overlap-add of the owned output range (gather over the windowed frames), times 1/envelope -----------
    {
        const long long o0 = (long long)t0 * hop;
        const long long o1 = (t1 == dm.T) ? dm.Lp : (long long)t1 * hop;
        const int span = (int)(o1 - o0);
        const int lead = (t0 - f0) * hop;           // tile-local position of o0 (frame f0 starts at 0)
        T* xo = (T*)a.x_out + (long long)b * dm.L;
        const T* __restrict__ ienv = (const T*)a.inv_env;
        auto newest = [&](int u, int& fl, int& off) {   // newest frame of the tile that covers position u, offset in it
            fl = ml.magic_hop ? (int)__umulhi((unsigned)u, ml.magic_hop) : u / hop;
            off = u - fl * hop;
            if (fl > nfr - 1) { off += (fl - (nfr - 1)) * hop; fl = nfr - 1; }
        };
        if ((hop & 1) == 0) {
            // even hop: two consecutive samples sit in ONE complex element of every frame that covers them
            for (int i = 2 * tid; i < span; i += 2 * NT) {
                const long long m = o0 + i - dm.P;
                if (m + 1 < 0 || m >= dm.L) continue;
                const bool ok0 = m >= 0, ok1 = m + 1 < dm.L;
                const T ie0 = ok0 ? __ldg(ienv + m) : T(0), ie1 = ok1 ? __ldg(ienv + m + 1) : T(0);
                int fl, off;
                newest(lead + i, fl, off);
                C acc = mk<T>(T(0), T(0));
                for (; fl >= 0 && off < N; --fl, off += hop) {
                    const C v = wb[fl * Mp + mr::padidx(off >> 1)];
                    acc.x += v.x; acc.y += v.y;
                }
                if (ok0) xo[m] = acc.x * ie0;
                if (ok1) xo[m + 1] = acc.y * ie1;
            }
        } else {
            const T* wbf = reinterpret_cast<const T*>(wb);
            for (int i = tid; i < span; i += NT) {
                const long long m = o0 + i - dm.P;
                if (m < 0 || m >= dm.L) continue;
                const T ie = __ldg(ienv + m);
                int fl, off;
                newest(lead + i, fl, off);
                T acc = T(0);
                for (; fl >= 0 && off < N; --fl, off += hop)
                    acc += wbf[2 * (fl * Mp + mr::padidx(off >> 1)) + (off & 1)];
                xo[m] = acc * ie;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int mr_smem_optin() {
    static int cached = -1;
    if (cached < 0) {
        int dev = 0, v = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess) return 0;
        cached = v;
    }
    return cached;
}

template <typename T, int OP>
static int launch_mr(TileArgs& a, const mr::Plan& mp, cudaStream_t st) {
    const Dims& dm = a.dm;
    const int Mp = mr::padded_len(dm.M);
    const size_t frame_bytes = (size_t)Mp * 2 * sizeof(T);
    const size_t perm_bytes = ((size_t)dm.M * 2 + 15) / 16 * 16;
    const int halo = (OP == OP_STFT) ? 0 : dm.K;
    const int optin = mr_smem_optin();
    if (optin <= 0) return SPECINV_ERR_NO_DEVICE;
    const size_t big = (size_t)optin - 1024 - perm_bytes;
    // Two CTAs of 16 warps per SM (1024 threads at 64 registers), each with half of the SM's shared memory (228 KB,
    // 1 KB reserved per CTA).  Four CTAs of 8 warps with a quarter each measured no better (within +-6 %, and 1.29 vs
    // 0.75 ms at 1536/384, where the smaller tile pays more halo frames).
    const int ctas = 2;
    size_t budget = (size_t)(228 * 1024 / ctas - 1024) - 256 - perm_bytes;
    if (budget > big) budget = big;
    int cap = (int)(budget / frame_bytes);
    if (cap - halo < (halo > 1 ? 2 * halo : 2)) cap = (int)(big / frame_bytes);   // poor owned / halo ratio: one fat CTA
    if (cap - halo < 1) return SPECINV_ERR_UNSUPPORTED;    // hop too small for this n_fft: the halo does not fit
    if (cap - halo > dm.T) cap = dm.T + halo;
    // small problems: prefer enough tiles to cover the 148 SMs twice
    while (cap - halo > 4 * (halo > 0 ? halo : 1) && (long long)dm.B * ((dm.T + cap - halo - 1) / (cap - halo)) < 2 * 148)
        cap = halo + (cap - halo + 1) / 2;
    // teams: the CTA's warps dealt to 16, 8, 4, 2 or 1 teams; the tile holds a multiple of the team count (even load),
    // and a bigger team pays ~3 % per doubling in barriers
    // fp64: 8 warps per CTA (two CTAs per SM at up to 128 registers: the double-precision butterflies of radix 8 / 11 /
    // 13 do not fit 64 registers without spilling)
    const int warps = (sizeof(T) == 8 ? 16 : 32) / ctas;
    int best_teams = 1, best_nfr = cap; double best_score = -1.0;
    for (int teams = warps; teams >= 1; teams >>= 1) {
        int nfr = cap / teams * teams;
        if (nfr - halo < 1) continue;
        int lg = 0; for (int g = warps / teams; g > 1; g >>= 1) ++lg;
        const double score = (double)(nfr - halo) / nfr * (1.0 - 0.03 * lg);
        if (score > best_score) { best_score = score; best_teams = teams; best_nfr = nfr; }
    }
    MrLaunch ml;
    ml.team_warps = warps / best_teams;
    ml.frames_cap = best_nfr;
    ml.Mp = Mp;
    ml.magic_M = mr::magic_of(dm.M);
    ml.magic_npair = mr::magic_of(dm.M / 2 + 1);
    ml.magic_np1 = mr::magic_of(dm.M / 2);
    ml.magic_hop = ((long long)(best_nfr + 1) * dm.hop + dm.N) * (long long)dm.hop < (1LL << 32) ? mr::magic_of(dm.hop) : 0u;
    a.tile_frames = best_nfr - halo;
    a.Mp = Mp;
    const size_t smem = (size_t)best_nfr * frame_bytes + perm_bytes;
    cudaError_t e = cudaFuncSetAttribute(mr_tile_kernel<T, OP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    dim3 grid((dm.T + a.tile_frames - 1) / a.tile_frames, dm.B);
    if (grid.y > 65535) return SPECINV_ERR_UNSUPPORTED;
    mr_tile_kernel<T, OP><<<grid, warps * 32, smem, st>>>(a, mp, ml);
    return (int)cudaGetLastError();
}

template <typename T>
static int launch_mr_op(int op, TileArgs& a, const mr::Plan& mp, cudaStream_t st) {
    switch (op) {
        case OP_STFT:  return launch_mr<T, OP_STFT>(a, mp, st);
        case OP_ISTFT: return launch_mr<T, OP_ISTFT>(a, mp, st);
        case OP_GL:    return launch_mr<T, OP_GL>(a, mp, st);
        case OP_GLR:   return launch_mr<T, OP_GLR>(a, mp, st);
        case OP_ADMM:  return launch_mr<T, OP_ADMM>(a, mp, st);
        default:       return SPECINV_ERR_INVALID;
    }
}

int mr_tile_launch(int dtype, int op, TileArgs& a, cudaStream_t st) {
    const Dims& dm = a.dm;
    if (dm.M > 4096 || (dm.N & 1)) return SPECINV_ERR_UNSUPPORTED;   // positions are 16-bit; the N/2-point trick needs an even N
    mr::Plan mp;
    // the plan's root table: W_M^j (M entries) for a power of two, W_N^j (N entries) otherwise (specinv_common.cuh)
    if (!mr::make_plan(dm.M, dm.pow2 ? dm.M : dm.N, &mp, dtype == SPECINV_F32)) return SPECINV_ERR_UNSUPPORTED;
    return dtype == SPECINV_F64 ? launch_mr_op<double>(op, a, mp, st) : launch_mr_op<float>(op, a, mp, st);
}

}  // namespace specinv
