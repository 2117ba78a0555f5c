// specinv_mel_inverse: torchaudio's InverseMelScale as one GEMM with relu epilogue,
//   out[b, f, t] = relu(sum_j P[f, j] * mel[b, j, t]),   P = pinv(fb^T) (n_stft x n_mels, host float64, see
// torchaudio_compat.py).  Register-blocked FFMA (packed FP32x2 in fp32, DFMA in fp64), no tensor cores: TF32 would
// miss the 1e-5 * max|ref| accuracy torchaudio's fp32 lstsq gives.
//
// Tiling: a CTA computes a BF x BT = 128 x 64 tile of out for one signal, looping over n_mels in BK = 16 slices
// staged in shared memory (so any n_mels works); each of the 256 threads holds an 8 (rows) x 4 (frames) block of
// accumulators.  A thread's frames are tx + 16 c, so every store instruction of a warp writes 16 consecutive frames of
// two rows.  Rows of P outside [f_lo, f_hi) are zero (bins no filter covers: DC, everything above f_max); CTAs with
// blockIdx.y >= the number of covered row tiles write zeros there without reading P or mel.
#include "specinv_common.cuh"
#include "fft_regs.cuh"

namespace specinv {
namespace mel {

constexpr int BF = 128, BT = 64, BK = 16, THREADS = 256;
constexpr int RM = 8, RN = 4;            // per-thread rows x frames
constexpr int AS_LD = BF + 4;            // padded row of the P slice: spreads the transposing stores over the banks
static_assert(BF == 16 * RM && BT == 16 * RN && THREADS == 256, "16 x 16 threads cover the tile");
static_assert(BF * BK % THREADS == 0 && BK * BT % THREADS == 0, "tile loads are whole rounds of the CTA");

// torch.relu: NaN stays NaN
template <typename T> __device__ __forceinline__ T relu(T v) { return v < T(0) ? T(0) : v; }

template <typename T> struct Acc {
    T v[RM][RN];
    __device__ __forceinline__ void zero() {
#pragma unroll
        for (int i = 0; i < RM; ++i)
#pragma unroll
            for (int c = 0; c < RN; ++c) v[i][c] = T(0);
    }
    __device__ __forceinline__ void fma(const T (&a)[RM], const T (&b)[RN]) {
#pragma unroll
        for (int i = 0; i < RM; ++i)
#pragma unroll
            for (int c = 0; c < RN; ++c) v[i][c] = fma_(a[i], b[c], v[i][c]);
    }
    static __device__ __forceinline__ T fma_(T a, T b, T c) { return ::fma(a, b, c); }
};

// fp32: the 4 frames of a row as two FP32x2 pairs, one FFMA2 per pair
template <> struct Acc<float> {
    float2 v[RM][RN / 2];
    __device__ __forceinline__ void zero() {
#pragma unroll
        for (int i = 0; i < RM; ++i)
#pragma unroll
            for (int c = 0; c < RN / 2; ++c) v[i][c] = f2(0.f, 0.f);
    }
    __device__ __forceinline__ void fma(const float (&a)[RM], const float (&b)[RN]) {
#pragma unroll
        for (int i = 0; i < RM; ++i)
#pragma unroll
            for (int c = 0; c < RN / 2; ++c) v[i][c] = pfma(f2(a[i], a[i]), f2(b[2 * c], b[2 * c + 1]), v[i][c]);
    }
    __device__ __forceinline__ float get(int i, int c) const { return (c & 1) ? v[i][c >> 1].y : v[i][c >> 1].x; }
};

template <typename T> __device__ __forceinline__ T acc_get(const Acc<T>& a, int i, int c) { return a.v[i][c]; }
template <> __device__ __forceinline__ float acc_get(const Acc<float>& a, int i, int c) { return a.get(i, c); }

// grid: x = batch * t_tiles, y = covered row tiles + zero row tiles
template <typename T>
__global__ void __launch_bounds__(THREADS)
mel_inverse_kernel(const T* __restrict__ P, const T* __restrict__ mel, T* __restrict__ out, int F, int M, int f_lo,
                   int f_hi, long long T_, int t_tiles, int y_cov) {
    __shared__ __align__(16) T As[BK][AS_LD];    // As[k][f] = P[f0 + f][k0 + k]
    __shared__ __align__(16) T Bs[BK][BT];       // Bs[k][t] = mel[b][k0 + k][t0 + t]
    const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
    const long long b = blockIdx.x / t_tiles;
    const long long t0 = (long long)(blockIdx.x % t_tiles) * BT;
    T* outb = out + b * F * T_;

    if ((int)blockIdx.y >= y_cov) {                  // rows no filter covers: [0, f_lo) then [f_hi, F)
        const int r0 = ((int)blockIdx.y - y_cov) * BF, n_zero = f_lo + (F - f_hi);
#pragma unroll
        for (int i = 0; i < RM; ++i) {
            const int r = r0 + ty * RM + i;
            const int f = r < f_lo ? r : f_hi + (r - f_lo);
#pragma unroll
            for (int c = 0; c < RN; ++c) {
                const long long t = t0 + tx + 16 * c;
                if (r < n_zero && t < T_) outb[(long long)f * T_ + t] = T(0);
            }
        }
        return;
    }

    const int f0 = f_lo + (int)blockIdx.y * BF;
    const T* melb = mel + b * M * T_;
    Acc<T> acc;
    acc.zero();
    for (int k0 = 0; k0 < M; k0 += BK) {
#pragma unroll
        for (int j = 0; j < BF * BK / THREADS; ++j) {     // 16 consecutive k of a row of P per half warp
            const int e = tid + j * THREADS, f = e / BK, k = e % BK, gf = f0 + f, gk = k0 + k;
            As[k][f] = (gf < f_hi && gk < M) ? P[(long long)gf * M + gk] : T(0);
        }
#pragma unroll
        for (int j = 0; j < BK * BT / THREADS; ++j) {     // 64 consecutive frames of a mel row per two warps
            const int e = tid + j * THREADS, k = e / BT, t = e % BT, gk = k0 + k;
            const long long gt = t0 + t;
            Bs[k][t] = (gk < M && gt < T_) ? melb[(long long)gk * T_ + gt] : T(0);
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            T a[RM], bv[RN];
#pragma unroll
            for (int i = 0; i < RM; ++i) a[i] = As[k][ty * RM + i];
#pragma unroll
            for (int c = 0; c < RN; ++c) bv[c] = Bs[k][tx + 16 * c];
            acc.fma(a, bv);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < RM; ++i) {
        const int f = f0 + ty * RM + i;
#pragma unroll
        for (int c = 0; c < RN; ++c) {
            const long long t = t0 + tx + 16 * c;
            if (f < f_hi && t < T_) outb[(long long)f * T_ + t] = relu(acc_get(acc, i, c));
        }
    }
}

}  // namespace mel
}  // namespace specinv

extern "C" int specinv_mel_inverse(int dtype, const void* P, int n_stft, int n_mels, int f_lo, int f_hi,
                                   const void* mel, void* out, int batch, int64_t n_frames, void* stream) {
    using namespace specinv::mel;
    if (dtype != SPECINV_F32 && dtype != SPECINV_F64) return SPECINV_ERR_INVALID;
    if (n_stft < 1 || n_mels < 1 || batch < 1 || n_frames < 0) return SPECINV_ERR_INVALID;
    if (f_lo < 0 || f_lo > f_hi || f_hi > n_stft) return SPECINV_ERR_INVALID;
    if (n_frames == 0) return SPECINV_OK;
    if (!out || (f_hi > f_lo && (!P || !mel))) return SPECINV_ERR_INVALID;
    const long long t_tiles = (n_frames + BT - 1) / BT;
    const int y_cov = (f_hi - f_lo + BF - 1) / BF, y_zero = (n_stft - (f_hi - f_lo) + BF - 1) / BF;
    if ((long long)batch * t_tiles > 0x7fffffffLL || y_cov + y_zero > 65535) return SPECINV_ERR_UNSUPPORTED;
    const dim3 grid((unsigned)(batch * t_tiles), (unsigned)(y_cov + y_zero));
    cudaStream_t st = (cudaStream_t)stream;
    if (dtype == SPECINV_F64)
        mel_inverse_kernel<double><<<grid, THREADS, 0, st>>>((const double*)P, (const double*)mel, (double*)out, n_stft,
                                                             n_mels, f_lo, f_hi, n_frames, (int)t_tiles, y_cov);
    else
        mel_inverse_kernel<float><<<grid, THREADS, 0, st>>>((const float*)P, (const float*)mel, (float*)out, n_stft,
                                                            n_mels, f_lo, f_hi, n_frames, (int)t_tiles, y_cov);
    return (int)cudaGetLastError();
}
