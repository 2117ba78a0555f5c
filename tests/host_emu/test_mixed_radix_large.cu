// Host-side check of the mixed-radix plan and passes (csrc/mixed_radix.cuh) at the transform lengths of the streamed
// kernel (csrc/specinv_generic_stream.cu): M = 6000, 8192 and 16384 (n_fft up to 32768).  One CTA's threads are
// emulated one after the other, pass by pass; the result is compared with a double-precision DFT (table-driven) at
// the digit-reversed positions, the 16-bit position table is checked, and the inverse passes must bring the frame back
// (times M).
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "../../spectrogram_inversion_b200/csrc/mixed_radix.cuh"
using namespace specinv;

template <typename T, typename C>
double run(int M, int tw_n, int nt) {
    mr::Plan p;
    if (!mr::make_plan(M, tw_n, &p, sizeof(T) == 4)) { printf("M=%d: no plan\n", M); return 1e9; }
    const int nf = 2, Mp = mr::padded_len(M);
    if (mr::padidx(M - 1) > 0xffff || mr::padidx(M - 1) >= Mp) { printf("M=%d: positions overflow\n", M); return 1e9; }
    std::vector<C> tw(tw_n), wb((size_t)nf * Mp);
    for (int j = 0; j < tw_n; ++j) { tw[j].x = (T)cos(2 * M_PI * j / tw_n); tw[j].y = (T)(-sin(2 * M_PI * j / tw_n)); }
    std::vector<double> cs(M), sn(M);
    for (int j = 0; j < M; ++j) { cs[j] = cos(2 * M_PI * j / M); sn[j] = -sin(2 * M_PI * j / M); }
    std::vector<double> re((size_t)nf * M), im((size_t)nf * M);
    for (int f = 0; f < nf; ++f)
        for (int n = 0; n < M; ++n) {
            re[f * M + n] = (double)rand() / RAND_MAX - 0.5; im[f * M + n] = (double)rand() / RAND_MAX - 0.5;
            wb[f * Mp + mr::padidx(n)].x = (T)re[f * M + n]; wb[f * Mp + mr::padidx(n)].y = (T)im[f * M + n];
        }
    for (int s = 0; s < p.nst; ++s)
        for (int tid = 0; tid < nt; ++tid) mr::pass<T, false>(wb.data(), nf, Mp, p, s, tw.data(), tid, nt);
    double err = 0;
    std::vector<char> seen(M, 0);
    for (int f = 0; f < nf; ++f)
        for (int k = 0; k < M; ++k) {
            double sr = 0, si = 0;
            long long j = 0;                              // (k n) mod M
            for (int n = 0; n < M; ++n) {
                sr += re[f * M + n] * cs[j] - im[f * M + n] * sn[j];
                si += re[f * M + n] * sn[j] + im[f * M + n] * cs[j];
                j += k; if (j >= M) j -= M;
            }
            const int pos = mr::mr_position(p, k);
            if (pos < 0 || pos >= M) return 1e9;
            if (f == 0) { if (seen[pos]) return 1e9; seen[pos] = 1; }
            const C v = wb[f * Mp + mr::padidx(pos)];
            err = fmax(err, fmax(fabs(v.x - sr), fabs(v.y - si)) / sqrt((double)M));
        }
    for (int s = p.nst - 1; s >= 0; --s)
        for (int tid = 0; tid < nt; ++tid) mr::pass<T, true>(wb.data(), nf, Mp, p, s, tw.data(), tid, nt);
    for (int f = 0; f < nf; ++f)
        for (int n = 0; n < M; ++n) {
            const C v = wb[f * Mp + mr::padidx(n)];
            err = fmax(err, fmax(fabs(v.x / M - re[f * M + n]), fabs(v.y / M - im[f * M + n])));
        }
    return err;
}

int main() {
    // the streamed kernel's root table: W_M for a power of two, W_N (N = 2 M entries) otherwise
    const int Ms[] = {6000, 8192, 16384};
    double ef = 0, ed = 0;
    for (int M : Ms) {
        const int tw_n = (M & (M - 1)) ? 2 * M : M;
        const double a = run<float, float2>(M, tw_n, 512), b = run<double, double2>(M, tw_n, 384);
        printf("M=%5d tw_n=%5d  fp32 %.2e  fp64 %.2e\n", M, tw_n, a, b);
        ef = fmax(ef, a); ed = fmax(ed, b);
    }
    printf("max err fp32 %.3e fp64 %.3e\n", ef, ed);
    return (ef < 1e-6 && ed < 4e-14) ? 0 : 1;     // the float64 reference DFT itself errs ~1e-14 at M = 16384
}
