// Streamed-frame generic kernels: STFT, ISTFT, one Griffin-Lim iteration (with or without momentum state, both
// recurrences), one ADMM iteration, for the shapes the tile kernels (specinv_generic.cu, specinv_generic_mr.cu) cannot
// hold: frames too large for the K = (n_fft - 1) / hop halo frames plus one owned frame to sit in shared memory at
// once, and every n_fft above 8192 (up to 32768 in fp32, 16384 in fp64).  Any even n_fft whose half factors into
// 2 .. 13, any hop, every torch.stft option the reference forwards.
//
// A CTA owns a long contiguous range of frames [t0, t1) of one signal and the output samples [t0 * hop, t1 * hop) of
// the padded signal (the last range: up to Lp).  It takes its K halo frames and then its owned frames through shared
// memory in ascending order, `nbuf` frames per step:
//     frame + window -> forward passes -> point-wise update / projection -> inverse passes (x synthesis window)
//     -> overlap-add into the carry
// The carry holds the samples that are still receiving frames.  After the step that adds frame f, no later frame
// touches a sample before (f + 1) * hop, so those samples are final: they are multiplied by 1/envelope and stored.
// Every sample is accumulated by exactly one CTA, in ascending frame order, without atomics: runs are deterministic.
// The carry is a ring of (nbuf - 1) * hop + n_fft samples in shared memory when it fits next to the frames, otherwise
// the CTA's own samples of x_out (written only by this CTA, L2-resident while they are open).
//
// State rows and metric sums are written for owned frames only, as in the tile kernels.

#include "specinv_common.cuh"
#include "generic_tile.cuh"
#include "generic_fft.cuh"
#include "mixed_radix.cuh"

namespace specinv {

struct StreamLaunch {
    int nbuf;         // frames per step in shared memory
    int Mp;           // padded complex elements per frame
    int range;        // owned frames per CTA
    int ring;         // samples of the shared-memory carry ring, or 0: the carry lives in x_out
};

template <typename T, int OP>
__global__ void __launch_bounds__(sizeof(T) == 8 ? 384 : 512, 1)
stream_tile_kernel(const TileArgs a, const mr::Plan mp, const StreamLaunch sl) {
    using C = cx_t<T>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const Dims& dm = a.dm;
    const int M = dm.M, N = dm.N, hop = dm.hop, Mp = sl.Mp;
    C* wb = reinterpret_cast<C*>(smem_raw);
    unsigned short* perm = reinterpret_cast<unsigned short*>(wb + (size_t)sl.nbuf * Mp);
    T* ring = reinterpret_cast<T*>(perm + ((M + 7) & ~7));

    const int b = blockIdx.y;
    const int t0 = blockIdx.x * sl.range;
    const int t1 = min(dm.T, t0 + sl.range);
    const int f0 = (OP == OP_STFT) ? t0 : max(0, t0 - dm.K);
    const int tid = threadIdx.x, NT = blockDim.x;

    const C* __restrict__ tw = (const C*)a.tw;
    const C* __restrict__ twr = (const C*)a.twr;
    const T* __restrict__ wa = (const T*)a.wa;
    const T* __restrict__ ws = (const T*)a.ws;
    const T* __restrict__ ienv = (const T*)a.inv_env;
    T* xo = (T*)a.x_out + (long long)b * dm.L;

    // padded position of bin k after the forward passes
    for (int k = tid; k < M; k += NT) perm[k] = (unsigned short)mr::padidx(mr::mr_position(mp, k));
    __syncthreads();

    // output samples this CTA finishes, as positions in the padded signal, clipped to the samples that exist
    const long long o0 = max((long long)t0 * hop, (long long)dm.P);
    const long long o1 = min((t1 == dm.T) ? dm.Lp : (long long)t1 * hop, (long long)dm.P + dm.L);

    T dsum = T(0), esum = T(0);
    const bool want_sums = a.sums != nullptr;
    const int npair = M / 2 + 1;

    for (int g = f0; g < t1; g += sl.nbuf) {
        const int nf = min(sl.nbuf, t1 - g);

        // ---- A: frame + analysis window: z[n] = x[2n] w[2n] + i x[2n+1] w[2n+1], then the forward passes -------------
        if constexpr (OP != OP_ISTFT) {
            const T* __restrict__ x = (const T*)a.x_in + (long long)b * dm.L;
            for (int f = 0; f < nf; ++f) {
                const long long base = (long long)(g + f) * hop;
                C* v = wb + (size_t)f * Mp;
                for (int n = tid; n < M; n += NT) {
                    const long long i0 = pad_index(base + 2 * n, dm.P, dm.L, dm.pad_mode);
                    const long long i1 = pad_index(base + 2 * n + 1, dm.P, dm.L, dm.pad_mode);
                    const T v0 = i0 >= 0 ? __ldg(x + i0) : T(0), v1 = i1 >= 0 ? __ldg(x + i1) : T(0);
                    v[mr::padidx(n)] = mk<T>(v0 * __ldg(wa + 2 * n), v1 * __ldg(wa + 2 * n + 1));
                }
            }
            __syncthreads();
            for (int s = 0; s < mp.nst; ++s) {
                mr::pass<T, false>(wb, nf, Mp, mp, s, tw, tid, NT);
                __syncthreads();
            }
        }

        // ---- C: real-FFT post-process, point-wise update, inverse pre-process (pairs k, M-k) ------------------------
        for (int idx = tid; idx < nf * npair; idx += NT) {
            const int f = idx / npair, k = idx - f * npair;
            const int t = g + f;
            const bool owned = t >= t0;
            C* v = wb + (size_t)f * Mp;
            const int kA = k, kB = M - k;
            const int pA = perm[kA], pB = perm[kB == M ? 0 : kB];
            const C w = __ldg(twr + k);
            C sA = mk<T>(T(0), T(0)), sB = sA;
            if constexpr (OP != OP_ISTFT) rfft_post_pair<T>(v[pA], v[pB], w, sA, sB);
            const BinIO<T> io(a, (long long)b * dm.T + t);
            C hA, hB;
            if (dm.onesided) {
                hA = bin_update<T, OP>(a, io, kA, sA, owned, want_sums, dsum, esum);
                hB = (kB != kA) ? bin_update<T, OP>(a, io, kB, sB, owned, want_sums, dsum, esum) : hA;
            } else {
                // two-sided: bins kA, kB and their mirrors N-kA, N-kB (= conj of the real-input STFT);
                // ifft(...).real (methods.py:145-146) == irfft of the Hermitian part (p[k]+conj p[N-k])/2
                hA = bin_update<T, OP>(a, io, kA, sA, owned, want_sums, dsum, esum);
                if (kA != 0) {
                    const C m = bin_update<T, OP>(a, io, N - kA, mk<T>(sA.x, -sA.y), owned, want_sums, dsum, esum);
                    hA = mk<T>(T(0.5) * (hA.x + m.x), T(0.5) * (hA.y - m.y));
                }
                if (kB != kA) {
                    hB = bin_update<T, OP>(a, io, kB, sB, owned, want_sums, dsum, esum);
                    if (kB != M) {
                        const C m = bin_update<T, OP>(a, io, N - kB, mk<T>(sB.x, -sB.y), owned, want_sums, dsum, esum);
                        hB = mk<T>(T(0.5) * (hB.x + m.x), T(0.5) * (hB.y - m.y));
                    }
                } else {
                    hB = hA;
                }
            }
            if constexpr (OP != OP_STFT) {
                if (k == 0) { hA.y = T(0); hB.y = T(0); }  // C2R ignores Im(DC), Im(Nyquist)
                C zA, zB;
                irfft_pre_pair<T>(hA, hB, w, zA, zB);
                v[pA] = zA;
                if (kB != kA && k != 0) v[pB] = zB;
            }
        }
        __syncthreads();
        if constexpr (OP == OP_STFT) continue;

        // ---- D: inverse passes (digit-reversed -> natural); the last one applies the synthesis window ---------------
        for (int s = mp.nst - 1; s >= 0; --s) {
            mr::pass<T, true>(wb, nf, Mp, mp, s, tw, tid, NT, s == 0 ? ws : (const T*)nullptr);
            __syncthreads();
        }

        // ---- E: overlap-add of frames g .. g+nf-1 into the carry, in ascending frame order ---------------------------
        {
            const long long gb = (long long)g * hop;                 // u = pp - gb: position relative to frame g
            const long long lo = max(gb, o0), hi = min(gb + (long long)(nf - 1) * hop + N, o1);
            const int rbase = sl.ring ? (int)(gb % sl.ring) : 0;
            const T* wbf = reinterpret_cast<const T*>(wb);
            for (long long pp = lo + tid; pp < hi; pp += NT) {
                const int u = (int)(pp - gb);
                const int fh = min(u / hop, nf - 1);                  // newest frame of the step that covers pp
                const int fl = u >= N ? (u - N) / hop + 1 : 0;        // oldest
                // the first frame that touches pp: no earlier frame covers it (frame f0 - 1 never covers an output
                // sample of the range: (K + 1) * hop >= n_fft); the last one: no later frame does, or it is frame T-1
                const bool first = u + hop >= N || g == 0;
                const bool last = u / hop <= nf - 1 || g + nf == dm.T;
                int slot = rbase + u;
                if (slot >= sl.ring) slot -= sl.ring;
                const long long m = pp - dm.P;
                T acc = first ? T(0) : (sl.ring ? ring[slot] : xo[m]);
                for (int f = fl; f <= fh; ++f) {
                    const int off = u - f * hop;
                    acc += wbf[2 * (f * Mp + mr::padidx(off >> 1)) + (off & 1)];
                }
                if (last) xo[m] = acc * __ldg(ienv + m);
                else if (sl.ring) ring[slot] = acc;
                else xo[m] = acc;
            }
        }
        __syncthreads();
    }

    if constexpr (OP == OP_GL || OP == OP_GLR || OP == OP_ADMM) {
        if (want_sums) {   // fused metric epilogue: block reduce, one double atomic pair per CTA
            __shared__ double red[2][32];
            double d = (double)dsum, e = (double)esum;
            for (int o = 16; o > 0; o >>= 1) {
                d += __shfl_xor_sync(0xffffffffu, d, o);
                e += __shfl_xor_sync(0xffffffffu, e, o);
            }
            if ((tid & 31) == 0) { red[0][tid >> 5] = d; red[1][tid >> 5] = e; }
            __syncthreads();
            if (tid == 0) {
                double dd = 0, ee = 0;
                for (int i = 0; i < (NT >> 5); ++i) { dd += red[0][i]; ee += red[1][i]; }
                atomicAdd(a.sums, dd);
                atomicAdd(a.sums + 1, ee);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int stream_smem_optin() {
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
static int launch_stream(TileArgs& a, const mr::Plan& mp, cudaStream_t st) {
    const Dims& dm = a.dm;
    const int Mp = mr::padded_len(dm.M);
    const size_t frame_bytes = (size_t)Mp * 2 * sizeof(T);
    const size_t perm_bytes = (size_t)((dm.M + 7) & ~7) * 2;
    const int halo = (OP == OP_STFT) ? 0 : dm.K;
    const int optin = stream_smem_optin();
    if (optin <= 0) return SPECINV_ERR_NO_DEVICE;
    // One CTA per SM (16 warps in fp32, 12 in fp64: the radix-16 / radix-13 passes and the point-wise stage need more
    // than the 64 / 128 registers of two CTAs per SM without spilling).  The opt-in limit minus the 512 B reduction
    // array holds the frames, the position table and the ring.
    const long long budget = (long long)optin - 512 - (long long)perm_bytes;
    // frames per step: nbuf frames and, with the carry in shared memory, a ring of (nbuf - 1) * hop + N samples
    auto fit = [&](bool carry) -> int {
        const long long per = (long long)frame_bytes + (carry ? (long long)dm.hop * sizeof(T) : 0);
        const long long fixed = carry ? (long long)(dm.N - dm.hop) * sizeof(T) : 0;
        return budget - fixed >= per ? (int)((budget - fixed) / per) : 0;
    };
    const bool carry = OP != OP_STFT;
    bool carry_smem = carry;
    int nbuf = fit(carry);
    if (nbuf < 1 && carry) { carry_smem = false; nbuf = fit(false); }   // the carry moves to x_out
    if (nbuf < 1) return SPECINV_ERR_UNSUPPORTED;
    // ranges: at most one wave over the 148 SMs (a CTA's range is one serial chain of steps), each range at least
    // 4 K owned frames (K halo frames are recomputed per range), never more frames than the signal has
    const int want = dm.B < 148 ? 148 / dm.B : 1;
    int range = (dm.T + want - 1) / want;
    const int min_range = 4 * (halo > 0 ? halo : 1);
    if (range < min_range) range = min_range;
    if (range > dm.T) range = dm.T;
    if (nbuf > 8) nbuf = 8;
    if (nbuf > range + halo) nbuf = range + halo;
    const int ring = carry_smem ? (nbuf - 1) * dm.hop + dm.N : 0;
    StreamLaunch sl;
    sl.nbuf = nbuf; sl.Mp = Mp; sl.range = range; sl.ring = ring;
    a.tile_frames = range;
    a.Mp = Mp;
    const size_t smem = (size_t)nbuf * frame_bytes + perm_bytes + (size_t)ring * sizeof(T);
    cudaError_t e = cudaFuncSetAttribute(stream_tile_kernel<T, OP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    dim3 grid((dm.T + range - 1) / range, dm.B);
    if (grid.y > 65535) return SPECINV_ERR_UNSUPPORTED;
    stream_tile_kernel<T, OP><<<grid, sizeof(T) == 8 ? 384 : 512, smem, st>>>(a, mp, sl);
    return (int)cudaGetLastError();
}

template <typename T>
static int launch_stream_op(int op, TileArgs& a, const mr::Plan& mp, cudaStream_t st) {
    switch (op) {
        case OP_STFT:  return launch_stream<T, OP_STFT>(a, mp, st);
        case OP_ISTFT: return launch_stream<T, OP_ISTFT>(a, mp, st);
        case OP_GL:    return launch_stream<T, OP_GL>(a, mp, st);
        case OP_GLR:   return launch_stream<T, OP_GLR>(a, mp, st);
        case OP_ADMM:  return launch_stream<T, OP_ADMM>(a, mp, st);
        default:       return SPECINV_ERR_INVALID;
    }
}

int stream_tile_launch(int dtype, int op, TileArgs& a, cudaStream_t st) {
    const Dims& dm = a.dm;
    if (dm.N & 1) return SPECINV_ERR_UNSUPPORTED;                   // the N/2-point trick needs an even N
    if (dm.N > (dtype == SPECINV_F64 ? 16384 : 32768)) return SPECINV_ERR_UNSUPPORTED;   // one frame must fit
    if (mr::padidx(dm.M - 1) > 0xffff) return SPECINV_ERR_UNSUPPORTED;   // 16-bit position table
    mr::Plan mp;
    // the plan's root table: W_M^j (M entries) for a power of two, W_N^j (N entries) otherwise (specinv_common.cuh)
    if (!mr::make_plan(dm.M, dm.pow2 ? dm.M : dm.N, &mp, dtype == SPECINV_F32)) return SPECINV_ERR_UNSUPPORTED;
    return dtype == SPECINV_F64 ? launch_stream_op<double>(op, a, mp, st) : launch_stream_op<float>(op, a, mp, st);
}

}  // namespace specinv
