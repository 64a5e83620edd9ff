// ms_fir_long.cuh -- device side of the FIR stage's route for long impulse responses (ir_len > 8192 taps; EXTENSION: the
// reference cuts every IR to 8192 taps, main_v2.py:443): uniformly partitioned overlap-save.
//
// With partitions of P taps and 2P-point transforms, output block j (samples [jP, jP + P)) is the last P samples of
//     IFFT( sum_p H_p . X_{j-p} ),   H_p = FFT(ir[pP, pP + P)),  X_m = FFT(u[(m - 1) P, (m + 1) P))
// Blocks m and m + Jh of a render (Jh = ceil(J / 2)) share one complex transform Z_m = X_m + i X_{m+Jh}: H_p is the
// spectrum of a real signal, so  sum_p H_p Z_{s-p} = Y_s + i Y_{s+Jh}  holds on Z directly (no Hermitian unpacking),
// provided the entries s - p < 0 exist as "head" entries Z_{-q} = i X_{Jh-q}.  The transforms are FftEngine jobs
// (ols_forward / ols_inverse, ms_fft_host.h); this file holds the frequency-domain multiply-accumulate between them.

#define FL_T 8                 // output entries per thread: T accumulators and a sliding window of T input entries
#define FL_NTHR 256

// One MAC task: output entries [s0, s0 + cnt) of one render, every bin.  Entries are N complex values apart; Z and Y
// point at entry 0, head entries lie below it.  Entry e of Z holds data only if e >= -z_head and e is in
// [a_lo, a_hi) U [b_lo, b_hi) (the entries whose input blocks touch the input's support); all others are zero.
struct FirMacTask {
    const cpx* H;              // partition 0 of the IR spectra (already / N)
    const cpx* Z;
    cpx* Y;                    // receives swap(Y_s): the inverse is then a forward transform (ols_inverse)
    int N, K, s0, cnt;
    int z_head, a_lo, a_hi, b_lo, b_hi, _pad;
};
// Exact zeros of a long render's output outside the blocks the inverse writes: [0, n0) and [n1, out_n).
struct FirZeroJob { real* out; int n0, n1, out_n, _pad; };

MS_DEV bool fir_long_live(const FirMacTask& t, int e) {
    return e >= -t.z_head && ((e >= t.a_lo && e < t.a_hi) || (e >= t.b_lo && e < t.b_hi));
}
MS_DEV cpx fir_cmac(cpx acc, cpx h, cpx z) {
    return mk(acc.x + h.x * z.x - h.y * z.y, acc.y + h.x * z.y + h.y * z.x);
}
// A thread owns one bin of a task's cnt output entries.  Per partition step it loads H_p (shared by every task of the
// IR: L2-resident) and one new Z entry, and does FL_T complex multiply-adds -- two loads per 4 FL_T FMAs.
MS_DEV void fir_long_mac_body(const FirMacTask* MS_RESTRICT tasks, const Ctx& c) {
    const FirMacTask t = tasks[c.by];
    const int k = c.bx * c.nthr + c.tid;
    if (k >= t.N) return;
    const long long N = t.N;
    cpx acc[FL_T], w[FL_T];                   // w[u] = Z_{s0 + u - p} at partition step p
#pragma unroll
    for (int u = 0; u < FL_T; ++u) {
        acc[u] = c_zero();
        w[u] = (u < t.cnt && fir_long_live(t, t.s0 + u)) ? __ldg(&t.Z[(long long)(t.s0 + u) * N + k]) : c_zero();
    }
    for (int p = 0; p < t.K; ++p) {
        const cpx h = __ldg(&t.H[(long long)p * N + k]);
#pragma unroll
        for (int u = 0; u < FL_T; ++u) acc[u] = fir_cmac(acc[u], h, w[u]);
#pragma unroll
        for (int u = FL_T - 1; u > 0; --u) w[u] = w[u - 1];
        const int e = t.s0 - p - 1;
        w[0] = (p + 1 < t.K && fir_long_live(t, e)) ? __ldg(&t.Z[(long long)e * N + k]) : c_zero();
    }
#pragma unroll
    for (int u = 0; u < FL_T; ++u)
        if (u < t.cnt) t.Y[(long long)(t.s0 + u) * N + k] = c_swap(acc[u]);
}
MS_DEV void fir_long_zero_body(const FirZeroJob* MS_RESTRICT jobs, int nbx, const Ctx& c) {
    const FirZeroJob j = jobs[c.by];
    const int stride = nbx * c.nthr;
    for (int i = c.bx * c.nthr + c.tid; i < j.n0; i += stride) j.out[i] = (real)0;
    for (int i = j.n1 + c.bx * c.nthr + c.tid; i < j.out_n; i += stride) j.out[i] = (real)0;
}
