// ms_fft_kernels.cuh -- batched, variable-length spectral jobs on pairs of real signals.
//
// One "job" = two real signals a, b of the same length n packed as z = a + i b (b may be absent).
// Everything the render path does in the frequency domain is linear with real coefficients, so the
// pair never has to be separated: a real-symmetric mask acts on Z = A + iB directly and the
// spectral stretch (a two-point gather, reference main_v2.py:117-128) acts on the upper half through
// mirrored indices (see spec_value()).
//
// Transform lengths:  n with only factors 2,3,5 -> direct mixed-radix;  any other n -> Bluestein
// (chirp-z) on a power-of-two length M >= 2n-1.  A transform of executed length M = F1*F2 runs
//   F1 == 1 : one kernel, whole vector in shared memory                      (rows kernel, G = 1)
//   F1  > 1 : columns kernel (T adjacent columns, length-F1 FFTs, twiddle W_M^{k1 n2})
//             then rows kernel (G adjacent rows, length-F2 FFTs).
// Rows kernel modes:  NAT  -> scatter to natural order k = k1 + F1 k2 through the tile transpose
//                     CONV -> multiply by the Bluestein filter spectrum, swap, FFT again, twiddle,
//                             leave in place; a final columns kernel (no twiddle) finishes the
//                             inverse and applies the output chirp.
//                     RAW  -> leave the [k1][k2] spectrum in place (used to build filter spectra).

enum { LD_WORK = 0, LD_CPX, LD_PAIR, LD_PAIR_CHIRP, LD_SPEC, LD_SPEC_CHIRP, LD_BW, LD_OLS, LD_REALPAD };
enum { ST_WORK = 0, ST_CPX, ST_Z, ST_Z_CHIRP, ST_PAIR, ST_PAIR_CHIRP, ST_OLS, ST_HMUL };
enum { MODE_NAT = 0, MODE_CONV, MODE_RAW };
enum { OP_NONE = 0, OP_GRAIN = 1, OP_TILT = 2, OP_ROT = 3 };

// Raised-cosine / brick-wall edges in Hz, evaluated at f = k * df in float64 exactly the way
// numpy's rfftfreq-based masks do (reference main_v2.py:47-58, 67-100).
struct BandEdge {
    double lo_f0, lo_f1;   // rising skirt  [f0, f1]; lo_mode 0: none, 1: brick (zero f < lo_f1), 2: cosine
    double hi_f0, hi_f1;   // falling skirt [f0, f1]; hi_mode 0: none, 1: brick (zero f > hi_f0), 2: cosine
    int lo_mode, hi_mode;
    int zero;              // band contributes nothing (hi <= 0)
    int _pad;
};

struct SpecOp {             // same layout as ms_spec_op (include/microsound_b200.h); asserted in ms_fft_api.inl
    int kind;              // OP_*
    int n_bands;           // 0: no multiband stage; else 3
    int lp_on;             // low-pass stage present
    int stretch_on;        // spectral stretch present
    double df;             // bin spacing in Hz: 1.0 / (n * (1.0 / sr))
    double factor;         // stretch factor
    double alpha;          // OP_TILT: shape = max(k,1)^alpha ;  OP_ROT: theta (0.9 * width)
    double warp_exp;       // OP_GRAIN: 1 / power of fft_warp_power (0: none)
    BandEdge lp;           // low-pass described as a band with only a falling skirt
    BandEdge mb[3];
};


struct FftJob {
    int n, M, F1, F2;
    int T, G;                    // column-tile width, row-group height
    RadixPlan p1, p2;
    const cpx* tw1;           // w_F1^i
    const cpx* tw2;           // w_F2^i
    const cpx* twM_hi;        // W_M^(1024 i)
    const cpx* twM_lo;        // W_M^i, i < 1024
    const cpx* ch_hi;         // W_2n^(1024 i)   (Bluestein chirp), null for direct
    const cpx* ch_lo;         // W_2n^i, i < 1024
    const cpx* bspec;         // FFT_M(conj chirp, wrapped)/M in [k1][k2] layout
    // columns pass by in-tile Bluestein (F1 has a prime factor > 5): length-F1 DFT as a length-B1 circular
    // convolution held entirely in shared memory.  B1 == 0: plain mixed-radix columns.
    int B1, _padb;
    RadixPlan pb;                // radices of B1
    const cpx* twb;              // w_B1^i
    const cpx* b1_chirp;         // exp(-i pi j^2 / F1), j < F1
    const cpx* b1_spec;          // FFT_B1(conj chirp, wrapped) / B1, natural order
    const real* in_a; const real* in_b;
    real* out_a; real* out_b;
    const cpx* cin; cpx* cout;   // LD_CPX / ST_CPX
    cpx* Z;                   // natural-order spectrum, n entries
    cpx* work;                // M entries
    real out_scale;
    int ols_n;                   // overlap-save: signal length (LD_OLS / ST_OLS)
    long long p0_a, p0_b;        // overlap-save: first input sample position of block a / b (may be negative)
    int ols_skip;                // overlap-save: taps - 1 (leading outputs of a block that are discarded)
    int live_lo, live_hi;        // overlap-save: outputs outside [live_lo, live_hi) are exactly zero (input support + taps)
    int _pad;
    SpecOp op[2];                // per packed signal (a, b)
};

// ---- twiddles ------------------------------------------------------------------------------------
MS_DEV cpx tw2level(const cpx* MS_RESTRICT hi, const cpx* MS_RESTRICT lo, unsigned e) {
    return c_mul(__ldg(&hi[e >> 10]), __ldg(&lo[e & 1023u]));
}
// W_M^e from sincospi (e < M): used where every lane needs its own exponent -- a table lookup at a per-lane address costs
// the L1 data pipe up to 32 sectors a request, and that pipe (not DRAM, not FP64) is what bounds the FFT kernels.
MS_DEV cpx tw_direct(unsigned e, int M) {
    real sn, cs;
    r_sincospi((real)(2.0 * ((double)e / (double)M)), &sn, &cs);
    return mk(cs, -sn);
}
// chirp c[j] = exp(-i pi j^2 / n) = W_{2n}^(j^2 mod 2n)
MS_DEV cpx chirp(const FftJob& J, int j) {
    const long long jj = (long long)j * (long long)j;
    const long long m2 = 2ll * J.n;
    long long q = (long long)((double)jj / (double)m2);
    long long r = jj - q * m2;
    if (r < 0) r += m2;
    if (r >= m2) r -= m2;
    return tw2level(J.ch_hi, J.ch_lo, (unsigned)r);
}

// ---- spectral operators --------------------------------------------------------------------------
MS_DEV real edge_weight(const BandEdge& b, double f) {
    if (b.zero) return (real)0.;
    real w = (real)1.;
    if (b.lo_mode == 1) { if (f < b.lo_f1) return (real)0.; }
    else if (b.lo_mode == 2) {
        if (f < b.lo_f0) return (real)0.;
        if (f <= b.lo_f1) {
            double t = (f - b.lo_f0) / fmax(1e-12, b.lo_f1 - b.lo_f0);
            w *= (real)0.5 * ((real)1. - r_cospi((real)t));
        }
    }
    if (b.hi_mode == 1) { if (f > b.hi_f0) return (real)0.; }
    else if (b.hi_mode == 2) {
        if (f > b.hi_f1) return (real)0.;
        if (f >= b.hi_f0) {
            double t = (f - b.hi_f0) / fmax(1e-12, b.hi_f1 - b.hi_f0);
            w *= (real)0.5 * ((real)1. + r_cospi((real)t));
        }
    }
    return w;
}
MS_DEV real lp_weight(const SpecOp& op, int kk) { return op.lp_on ? edge_weight(op.lp, (double)kk * op.df) : (real)1.; }
MS_DEV real mb_weight(const SpecOp& op, int kk) {
    if (op.n_bands == 0) return (real)1.;
    const double f = (double)kk * op.df;
    real w = (real)0.;
    for (int b = 0; b < op.n_bands; ++b) w += edge_weight(op.mb[b], f);
    return w;
}
// One packed signal's spectrum out of Z = A + iB:  A[i] = (Z[i] + conj Z[n-i]) / 2,
// B[i] = (Z[i] - conj Z[n-i]) / (2i)   (0 <= i <= n/2).
MS_DEV cpx split_bin(const cpx* MS_RESTRICT Z, int n, int i, int sel, int paired) {
    const cpx p = __ldg(&Z[i]);
    if (!paired) return p;                    // b absent: Z is already A
    const cpx q = __ldg(&Z[i == 0 ? 0 : n - i]);
    if (sel == 0) return mk((real)0.5 * (p.x + q.x), (real)0.5 * (p.y - q.y));
    return mk((real)0.5 * (p.y + q.y), (real)0.5 * (q.x - p.x));
}
// low-passed spectrum at integer bin i, then the optional power warp (fft_warp_power, main_v2.py:103-115): bin i of
// the warped spectrum is the low-passed one interpolated at (i / kmax) ** (1 / power) * kmax (zero beyond the last bin).
MS_DEV cpx lp_bin(const SpecOp& op, const cpx* MS_RESTRICT Z, int n, int i, int sel, int paired) {
    return c_scale(split_bin(Z, n, i, sel, paired), lp_weight(op, i));
}
MS_DEV cpx warp_bin_on(const SpecOp& op, const cpx* MS_RESTRICT Z, int n, int i, int sel, int paired) {
    const int kmax = n >> 1;
    const double km = kmax < 1 ? 1.0 : (double)kmax;
    const double pos = pow((double)i / km, op.warp_exp) * km;
    if (pos > (double)kmax) return c_zero();
    int i0 = (int)pos;
    real fr = (real)(pos - (double)i0);
    if (i0 >= kmax) { i0 = kmax; fr = (real)0.; }
    cpx y = lp_bin(op, Z, n, i0, sel, paired);
    if (fr != (real)0.) {
        const cpx v1 = lp_bin(op, Z, n, i0 + 1, sel, paired);
        y = mk(y.x + (v1.x - y.x) * fr, y.y + (v1.y - y.y) * fr);
    }
    return y;
}
// low-pass -> [power warp] -> stretch (two-point gather at kk / factor, zero beyond the last bin) -> multiband weights
template <int WARP>
MS_DEV cpx grain_value(const SpecOp& op, const cpx* MS_RESTRICT Z, int n, int kk, int sel, int paired) {
    const int kmax = n >> 1;
    cpx y;
    if (!op.stretch_on) {
        y = WARP ? warp_bin_on(op, Z, n, kk, sel, paired) : lp_bin(op, Z, n, kk, sel, paired);
    } else {
        const double pos = (double)kk / fmax(1e-12, op.factor);
        if (pos > (double)kmax) return c_zero();
        int i0 = (int)pos;
        real fr = (real)(pos - (double)i0);
        if (i0 >= kmax) { i0 = kmax; fr = (real)0.; }
        y = WARP ? warp_bin_on(op, Z, n, i0, sel, paired) : lp_bin(op, Z, n, i0, sel, paired);
        if (fr != (real)0.) {
            cpx v1 = WARP ? warp_bin_on(op, Z, n, i0 + 1, sel, paired) : lp_bin(op, Z, n, i0 + 1, sel, paired);
            y = mk(y.x + (v1.x - y.x) * fr, y.y + (v1.y - y.y) * fr);
        }
    }
    return c_scale(y, mb_weight(op, kk));
}
// (the warped variant lives out of line as a whole, so the common path compiles exactly as it did without it)
MS_DEV_NOINLINE cpx grain_value_warped(const SpecOp& op, const cpx* MS_RESTRICT Z, int n, int kk, int sel, int paired) {
    return grain_value<1>(op, Z, n, kk, sel, paired);
}
MS_DEV cpx warp_bin(const SpecOp& op, const cpx* MS_RESTRICT Z, int n, int i, int sel, int paired) {      // partial-lock kernel
    if (op.warp_exp == 0.0) return lp_bin(op, Z, n, i, sel, paired);
    return warp_bin_on(op, Z, n, i, sel, paired);
}
// What irfft() would be handed for one signal at folded bin kk (0 <= kk <= n/2):
// low-pass -> stretch (two-point gather at kk/factor, zero beyond the last bin) -> multiband weights,
// or the tilt / rotation multipliers.
MS_DEV cpx op_value(const SpecOp& op, const cpx* MS_RESTRICT Z, int n, int kk, int sel, int paired) {
    const int kmax = n >> 1;
    if (op.kind == OP_NONE) return split_bin(Z, n, kk, sel, paired);
    if (op.kind == OP_TILT) {
        real s = (real)pow((double)(kk < 1 ? 1 : kk), op.alpha);
        return c_scale(split_bin(Z, n, kk, sel, paired), s);
    }
    if (op.kind == OP_ROT) {   // exp(i theta sin(2 pi kk / kmax))
        if (kk == 0) return split_bin(Z, n, kk, sel, paired);
        real sn, cs, rs, rc;
        r_sincospi((real)2.0 * (real)((double)kk / (double)(kmax < 1 ? 1 : kmax)), &sn, &cs);
        r_sincos((real)op.alpha * sn, &rs, &rc);
        return c_mul(split_bin(Z, n, kk, sel, paired), mk(rc, rs));
    }
    if (op.warp_exp != 0.0) return grain_value_warped(op, Z, n, kk, sel, paired);
    return grain_value<0>(op, Z, n, kk, sel, paired);
}
// Y[k] for natural k in [0, n): both packed signals at once, Hermitian-extended the way irfft does
// (imaginary part of DC and, for even n, of the Nyquist bin is dropped).
MS_DEV cpx spec_value(const FftJob& J, const cpx* MS_RESTRICT Z, int k) {
    const int n = J.n, kmax = n >> 1;
    const int upper = k > kmax;
    const int kk = upper ? n - k : k;
    const int paired = J.in_b != nullptr;
    cpx ya = op_value(J.op[0], Z, n, kk, 0, paired);
    cpx yb = paired ? op_value(J.op[1], Z, n, kk, 1, paired) : c_zero();
    if (kk == 0 || (!(n & 1) && kk == kmax)) { ya.y = (real)0.; yb.y = (real)0.; }
    if (upper) { ya.y = -ya.y; yb.y = -yb.y; }
    return mk(ya.x - yb.y, ya.y + yb.x);
}

// ---- load / store functors -----------------------------------------------------------------------
template <int LD>
MS_DEV cpx job_load(const FftJob& J, int idx) {
    if (LD == LD_WORK) return J.work[idx];
    if (LD == LD_CPX) return idx < J.n ? __ldg(&J.cin[idx]) : c_zero();
    if (LD == LD_PAIR || LD == LD_PAIR_CHIRP) {
        if (idx >= J.n) return c_zero();
        cpx v = mk(__ldg(&J.in_a[idx]), J.in_b ? __ldg(&J.in_b[idx]) : (real)0.);
        if (LD == LD_PAIR_CHIRP) v = c_mul(v, chirp(J, idx));
        return v;
    }
    if (LD == LD_SPEC) {            // inverse direct: feed swap(Y)
        if (idx >= J.n) return c_zero();
        return c_swap(spec_value(J, J.Z, idx));
    }
    if (LD == LD_SPEC_CHIRP) {      // inverse Bluestein: conj(Y) * chirp
        if (idx >= J.n) return c_zero();
        return c_mul(c_conj(spec_value(J, J.Z, idx)), chirp(J, idx));
    }
    if (LD == LD_OLS) {             // two blocks of one signal as re / im; zero outside [0, ols_n)
        const long long pa = J.p0_a + idx, pb = J.p0_b + idx;
        const real a = (pa >= 0 && pa < J.ols_n) ? __ldg(&J.in_a[pa]) : (real)0.;
        const real b = (J.in_b && pb >= 0 && pb < J.ols_n) ? __ldg(&J.in_b[pb]) : (real)0.;
        return mk(a, b);
    }
    if (LD == LD_REALPAD) {         // real taps, zero padded, pre-scaled by 1/M
        return idx < J.n ? mk(__ldg(&J.in_a[idx]) * J.out_scale, (real)0.) : c_zero();
    }
    if (LD == LD_BW) {              // wrapped conjugate chirp, scaled by 1/M
        int d;
        if (idx < J.n) d = idx; else if (idx > J.M - J.n) d = J.M - idx; else return c_zero();
        return c_scale(c_conj(chirp(J, d)), (real)1.0 / (real)J.M);
    }
    return c_zero();
}
template <int ST>
MS_DEV void job_store(const FftJob& J, int idx, cpx v) {
    if (ST == ST_WORK) { J.work[idx] = v; return; }
    if (ST == ST_HMUL) {            // filter spectrum: IR spectrum (at cin, already / B) times (1 + reflection-cloud spectrum)
        J.work[idx] = c_mul(__ldg(&J.cin[idx]), mk(v.x + (real)1.0, v.y));
        return;
    }
    if (ST == ST_OLS) {             // valid part of the circular convolution; un-swap the inverse half
        if (idx < J.ols_skip) return;
        const long long qa = J.p0_a + idx, qb = J.p0_b + idx;
        if (qa < J.ols_n) J.out_a[qa] = (qa >= J.live_lo && qa < J.live_hi) ? v.y : (real)0;
        if (J.out_b && qb < J.ols_n) J.out_b[qb] = (qb >= J.live_lo && qb < J.live_hi) ? v.x : (real)0;
        return;
    }
    if (idx >= J.n) return;
    if (ST == ST_CPX) { J.cout[idx] = c_scale(v, J.out_scale); return; }
    if (ST == ST_Z) { J.Z[idx] = v; return; }
    if (ST == ST_Z_CHIRP) { J.Z[idx] = c_mul(c_swap(v), chirp(J, idx)); return; }     // un-swap the inverse half of the convolution
    if (ST == ST_PAIR) {            // y = swap(FFT(swap(Y))) / n
        J.out_a[idx] = v.y * J.out_scale;
        if (J.out_b) J.out_b[idx] = v.x * J.out_scale;
        return;
    }
    if (ST == ST_PAIR_CHIRP) {      // r = chirp * conv ; y = conj(r) / n
        cpx r = c_mul(c_swap(v), chirp(J, idx));
        J.out_a[idx] = r.x * J.out_scale;
        if (J.out_b) J.out_b[idx] = -r.y * J.out_scale;
        return;
    }
}

// Load functors that are plain memory loads: the tile-fill loops issue them in batches of four BEFORE the first dependent
// shared-memory store (ncu on B200: with load and store in one loop body every STS waited out its own LDG -- the compiler
// cannot hoist a global load over a store through a pointer it cannot prove disjoint).
template <int LD> struct LdPlain { static constexpr bool v = (LD == LD_WORK || LD == LD_CPX || LD == LD_PAIR || LD == LD_OLS || LD == LD_REALPAD); };

// The job descriptor (geometry, radix plans, table pointers, spectral operators: ~1 KB) is staged in shared
// memory by the CTA: every later field access is a shared-memory load instead of a global one.
#define MS_JOB_SMEM ((sizeof(FftJob) + 15) / 16 * 16)
MS_DEV const FftJob& stage_job(const FftJob* MS_RESTRICT jobs, const Ctx& c) {
    const unsigned* src = (const unsigned*)(jobs + c.by);
    unsigned* dst = (unsigned*)c.smem;
    for (int i = c.tid; i < (int)(sizeof(FftJob) / 4); i += c.nthr) dst[i] = src[i];
    c.sync();
    return *(const FftJob*)c.smem;
}

// ---- spectral operator pass ---------------------------------------------------------------------------
// swap(Y[k]) for every natural k in [0, n) into `work`, in front of a plain-load inverse (two-pass lengths).  A thread owns
// folded bins kk and writes both k = kk and k = n - kk: consecutive threads gather at consecutive bins (the stretch /
// warp gathers of a warp fall into a few sectors), where the columns tile of the inverse would gather F1 rows F2 apart.
#define SPECOP_NTHR 256
#define SPECOP_PER 4
MS_DEV void spec_op_body(const FftJob* MS_RESTRICT jobs, const Ctx& c) {
    const FftJob& J = stage_job(jobs, c);
    const int n = J.n, kmax = n >> 1;
    const int kk0 = c.bx * (SPECOP_NTHR * SPECOP_PER) + c.tid;
    if (c.bx * (SPECOP_NTHR * SPECOP_PER) > kmax) return;
    const int paired = J.in_b != nullptr;
#pragma unroll 2
    for (int u = 0; u < SPECOP_PER; ++u) {
        const int kk = kk0 + u * SPECOP_NTHR;
        if (kk > kmax) break;
        cpx ya = op_value(J.op[0], J.Z, n, kk, 0, paired);
        cpx yb = paired ? op_value(J.op[1], J.Z, n, kk, 1, paired) : c_zero();
        if (kk == 0 || (!(n & 1) && kk == kmax)) { ya.y = (real)0.; yb.y = (real)0.; }
        J.work[kk] = mk(ya.y + yb.x, ya.x - yb.y);                                  // swap(Y[kk])
        if (kk != 0 && kk != n - kk) J.work[n - kk] = mk(yb.x - ya.y, ya.x + yb.y);   // swap(Y[n - kk]): both spectra conjugated
    }
}

// ---- columns kernel --------------------------------------------------------------------------------
// SB != 0: in-tile Bluestein with static convolution length B1 = SB and T = MS_SB_TILE / SB full columns, in place
#define MS_SB_TILE 2048
template <int LD, int ST, int TWID, int SB>
MS_DEV void fft_cols_bluestein_static(const FftJob& J, const Ctx& c) {
    static_assert(!SB || LdPlain<LD>::v, "static Bluestein columns: plain loads only");   // (SB = 0: never called)
    constexpr int T = MS_SB_TILE / (SB ? SB : 1);
    const int F1 = J.F1, F2 = J.F2;
    const int col0 = c.bx * T;
    if (col0 >= F2) return;
    cpx* s = (cpx*)(c.smem + MS_JOB_SMEM);
    TileGeom g; g.cnt = T; g.vs = 1; g.es = T; g.colmajor = 1;
    constexpr int all = MS_SB_TILE;
    for (int e0 = c.tid; e0 < all; e0 += 4 * c.nthr) {
        cpx ld[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int e = e0 + u * c.nthr, i = e / T, v = e - i * T;
            ld[u] = (e < all && i < F1) ? job_load<LD>(J, i * F2 + col0 + v) : c_zero();
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int e = e0 + u * c.nthr, i = e / T, v = e - i * T;
            if (e < all) s[tile_addr(g, v, i)] = i < F1 ? c_mul(ld[u], __ldg(&J.b1_chirp[i])) : c_zero();
        }
    }
    c.sync();
    tile_fft_pow2<1, SB ? SB : 128, T>(s, g, J.twb, c);
#pragma unroll 2
    for (int e = c.tid; e < all; e += c.nthr) {
        const int i = e / T, v = e - i * T;
        const int a = tile_addr(g, v, i);
        s[a] = c_swap(c_mul(s[a], __ldg(&J.b1_spec[i])));
    }
    c.sync();
    tile_fft_pow2<1, SB ? SB : 128, T>(s, g, J.twb, c);
    const int total = F1 * T;
    // a thread keeps its column (256 threads, T | 256) and walks k1 in steps of 256 / T: W_M^(k1 col) starts from sincospi and
    // is stepped by W_M^(col 256 / T) (T distinct values per warp: a cheap lookup)
    cpx tw = mk((real)1., (real)0.), tstep = tw;
    if (TWID) {
        const unsigned col = (unsigned)(col0 + c.tid % T);
        tw = tw_direct((unsigned)(c.tid / T) * col, J.M);
        tstep = tw2level(J.twM_hi, J.twM_lo, (unsigned)(((long long)col * (c.nthr / T)) % J.M));
    }
#pragma unroll 2
    for (int e = c.tid; e < total; e += c.nthr) {
        const int k1 = e / T, v = e - k1 * T;
        cpx val = c_mul(c_swap(s[tile_addr(g, v, k1)]), __ldg(&J.b1_chirp[k1]));
        if (TWID) { val = c_mul(val, tw); tw = c_mul(tw, tstep); }
        job_store<ST>(J, k1 * F2 + col0 + v, val);
    }
}
// B1 = 256 with WARP-LOCAL transforms (warp_fft256, ms_fft_core.cuh): eight adjacent columns per CTA, one warp per column.
// The tile is transposed through shared memory on the way in (chirp applied) and on the way out; between them the two
// 256-point transforms of the Bluestein convolution chain through registers (filter product in between) with
// __syncwarp only -- no block barrier inside the transforms and a third of the shared-memory round trips of the
// block-wide form above (measured on the FIR stage: 15.3 -> 9.3 ms with the same building block).
#define WB_RS ((ms_pad(256) + 1) | 1)
template <int LD, int ST, int TWID>
MS_DEV void fft_cols_bluestein_warp256(const FftJob& J, const Ctx& c) {
    const int F1 = J.F1, F2 = J.F2;
    const int col0 = c.bx * 8;
    if (col0 >= F2) return;
    cpx* s = (cpx*)(c.smem + MS_JOB_SMEM);
    const int lane = c.tid & 31, warp = c.tid >> 5;
    // rows 0 .. 127 may hold data (F1 <= 128), rows 128 .. 255 are the zero padding of the convolution
    static_assert(LdPlain<LD>::v, "warp-local Bluestein columns: plain loads only");
    cpx ld[4];                                                  // all loads in flight before the first store
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int e = c.tid + 256 * i, row = e >> 3, v = e & 7;
        ld[i] = row < F1 ? job_load<LD>(J, row * F2 + col0 + v) : c_zero();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int e = c.tid + 256 * i, row = e >> 3, v = e & 7;
        s[v * WB_RS + ms_pad(row)] = row < F1 ? c_mul(ld[i], __ldg(&J.b1_chirp[row])) : c_zero();
    }
    c.sync();
    cpx v[8];
    cpx* sw = s + warp * WB_RS;
#pragma unroll
    for (int q = 0; q < 4; ++q) v[q] = sw[ms_pad(lane + 32 * q)];
#pragma unroll
    for (int q = 4; q < 8; ++q) v[q] = c_zero();                // (the zero padding of the convolution never goes through shared memory)
    c.syncwarp();
    warp_fft256(v, sw, J.twb, lane, c);
#pragma unroll
    for (int m = 0; m < 8; ++m) v[m] = c_swap(c_mul(v[m], __ldg(&J.b1_spec[lane + 32 * m])));
    c.syncwarp();
    warp_fft256(v, sw, J.twb, lane, c);
    c.syncwarp();
    const int col = col0 + warp;
    // W_M^(k1 col), k1 = lane + 32 m:  W^(lane col) from sincospi (a table lookup at a per-lane address costs the L1 data pipe
    // 32 sectors a request, and that pipe is what bounds this kernel), stepped by the warp-uniform W^(32 col)
    cpx tb = mk((real)1., (real)0.), ts = tb;
    if (TWID) {
        real sn, cs;
        r_sincospi((real)(2.0 * ((double)((unsigned)lane * (unsigned)col) / (double)J.M)), &sn, &cs);
        tb = mk(cs, -sn);
        ts = tw2level(J.twM_hi, J.twM_lo, (unsigned)(((long long)32 * col) % J.M));
    }
#pragma unroll
    for (int m = 0; m < 4; ++m) {                               // F1 <= 128: outputs k1 = lane + 32 m, m < 4
        const int k1 = lane + 32 * m;
        if (k1 < F1) {
            cpx val = c_mul(c_swap(v[m]), __ldg(&J.b1_chirp[k1]));
            if (TWID) val = c_mul(val, tb);
            sw[ms_pad(k1)] = val;
        }
        if (TWID) tb = c_mul(tb, ts);
    }
    c.sync();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int e = c.tid + 256 * i, k1 = e >> 3, vv = e & 7;
        if (k1 < F1) job_store<ST>(J, k1 * F2 + col0 + vv, s[vv * WB_RS + ms_pad(k1)]);
    }
}
// Plain columns of exactly 256 rows (smooth n with 256 | n): one warp-local transform per column, no convolution.
template <int LD, int ST, int TWID>
MS_DEV void fft_cols_warp_plain256(const FftJob& J, const Ctx& c) {
    const int F2 = J.F2;
    const int col0 = c.bx * 8;
    if (col0 >= F2) return;
    const int ncol = (F2 - col0) < 8 ? (F2 - col0) : 8;
    cpx* s = (cpx*)(c.smem + MS_JOB_SMEM);
    const int lane = c.tid & 31, warp = c.tid >> 5;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        cpx ld[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int e = c.tid + 256 * (4 * half + i);
            ld[i] = (e & 7) < ncol ? job_load<LD>(J, (e >> 3) * F2 + col0 + (e & 7)) : c_zero();
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int e = c.tid + 256 * (4 * half + i);
            s[(e & 7) * WB_RS + ms_pad(e >> 3)] = ld[i];
        }
    }
    c.sync();
    cpx v[8];
    cpx* sw = s + warp * WB_RS;
#pragma unroll
    for (int q = 0; q < 8; ++q) v[q] = sw[ms_pad(lane + 32 * q)];
    c.syncwarp();
    warp_fft256(v, sw, J.tw1, lane, c);
    c.syncwarp();
    const int col = col0 + warp;
    cpx tb = mk((real)1., (real)0.), ts = tb;
    if (TWID) {
        tb = tw_direct((unsigned)lane * (unsigned)col, J.M);
        ts = tw2level(J.twM_hi, J.twM_lo, (unsigned)(((long long)32 * col) % J.M));
    }
#pragma unroll
    for (int m = 0; m < 8; ++m) {
        sw[ms_pad(lane + 32 * m)] = TWID ? c_mul(v[m], tb) : v[m];
        if (TWID) tb = c_mul(tb, ts);
    }
    c.sync();
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int e = c.tid + 256 * i;
        if ((e & 7) < ncol) job_store<ST>(J, (e >> 3) * F2 + col0 + (e & 7), s[(e & 7) * WB_RS + ms_pad(e >> 3)]);
    }
}
template <int LD, int ST, int TWID>
MS_DEV void fft_cols_warp_plain_body(const FftJob* MS_RESTRICT jobs, const Ctx& c) {
    const FftJob& J = stage_job(jobs, c);
    fft_cols_warp_plain256<LD, ST, TWID>(J, c);
}
// B1 = 512 (F1 <= 256), same scheme with warp_fft512: eight columns per CTA, a lane holds sixteen values of its column.
#define WB5_RS ((ms_pad(512) + 1) | 1)
template <int LD, int ST, int TWID>
MS_DEV void fft_cols_bluestein_warp512(const FftJob& J, const Ctx& c) {
    const int F1 = J.F1, F2 = J.F2;
    const int col0 = c.bx * 8;
    if (col0 >= F2) return;
    cpx* s = (cpx*)(c.smem + MS_JOB_SMEM);
    const int lane = c.tid & 31, warp = c.tid >> 5;
    const int ncol = (F2 - col0) < 8 ? (F2 - col0) : 8;         // (the class guarantees 4 | F2 only: the last tile may hold four columns)
    // rows 0 .. 255 may hold data, rows 256 .. 511 are the zero padding of the convolution (never staged: zeros in registers)
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        cpx ld[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int e = c.tid + 256 * (4 * half + i), row = e >> 3, vv = e & 7;
            ld[i] = (row < F1 && vv < ncol) ? job_load<LD>(J, row * F2 + col0 + vv) : c_zero();
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int e = c.tid + 256 * (4 * half + i), row = e >> 3, vv = e & 7;
            s[vv * WB5_RS + ms_pad(row)] = row < F1 ? c_mul(ld[i], __ldg(&J.b1_chirp[row])) : c_zero();
        }
    }
    c.sync();
    cpx v[16];
    cpx* sw = s + warp * WB5_RS;
#pragma unroll
    for (int q = 0; q < 8; ++q) v[q] = sw[ms_pad(lane + 32 * q)];
#pragma unroll
    for (int q = 8; q < 16; ++q) v[q] = c_zero();
    c.syncwarp();
    warp_fft512(v, sw, J.twb, lane, c);
#pragma unroll
    for (int m = 0; m < 16; ++m) v[m] = c_swap(c_mul(v[m], __ldg(&J.b1_spec[lane + 32 * m])));
    c.syncwarp();
    warp_fft512(v, sw, J.twb, lane, c);
    c.syncwarp();
    const int col = col0 + warp;
    cpx tb = mk((real)1., (real)0.), ts = tb;
    if (TWID) {
        tb = tw_direct((unsigned)lane * (unsigned)col, J.M);
        ts = tw2level(J.twM_hi, J.twM_lo, (unsigned)(((long long)32 * col) % J.M));
    }
#pragma unroll
    for (int m = 0; m < 8; ++m) {                               // F1 <= 256: outputs k1 = lane + 32 m, m < 8
        const int k1 = lane + 32 * m;
        if (k1 < F1) {
            cpx val = c_mul(c_swap(v[m]), __ldg(&J.b1_chirp[k1]));
            if (TWID) val = c_mul(val, tb);
            sw[ms_pad(k1)] = val;
        }
        if (TWID) tb = c_mul(tb, ts);
    }
    c.sync();
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int e = c.tid + 256 * i, k1 = e >> 3, vv = e & 7;
        if (k1 < F1 && vv < ncol) job_store<ST>(J, k1 * F2 + col0 + vv, s[vv * WB5_RS + ms_pad(k1)]);
    }
}
template <int LD, int ST, int TWID>
MS_DEV void fft_cols_warp512_body(const FftJob* MS_RESTRICT jobs, const Ctx& c) {
    const FftJob& J = stage_job(jobs, c);
    fft_cols_bluestein_warp512<LD, ST, TWID>(J, c);
}
template <int LD, int ST, int TWID>
MS_DEV void fft_cols_warp_body(const FftJob* MS_RESTRICT jobs, const Ctx& c) {
    const FftJob& J = stage_job(jobs, c);
    fft_cols_bluestein_warp256<LD, ST, TWID>(J, c);
}

template <int LD, int ST, int TWID, int SB>
MS_DEV void fft_cols_body(const FftJob* MS_RESTRICT jobs, const Ctx& c) {
    const FftJob& J = stage_job(jobs, c);
    if (SB) { fft_cols_bluestein_static<LD, ST, TWID, SB>(J, c); return; }
    const int T = J.T, F1 = J.F1, F2 = J.F2;
    const int col0 = c.bx * T;
    if (col0 >= F2) return;
    const int cnt = (F2 - col0) < T ? (F2 - col0) : T;
    const int rows = J.B1 ? J.B1 : F1;                         // vector length held in the tile
    cpx* s = (cpx*)(c.smem + MS_JOB_SMEM);
    cpx* const sA = s;
    cpx* s2 = s + (ms_pad((rows - 1) * T + T - 1) + 2);
    TileGeom g; g.cnt = cnt; g.vs = 1; g.es = T; g.colmajor = 1;
    const int total = F1 * cnt;
    const unsigned mgc = ms_magic_dev(cnt);
    if (J.B1) {
        // length-F1 DFT of every column as chirp * IFFT_B1(FFT_B1(x * chirp) * spec)
        const int all = rows * cnt;
#pragma unroll 2
        for (int e = c.tid; e < all; e += c.nthr) {
            const int i = ms_fastdiv(e, mgc), v = e - i * cnt;
            cpx val = c_zero();
            if (i < F1) val = c_mul(job_load<LD>(J, i * F2 + col0 + v), __ldg(&J.b1_chirp[i]));
            s[tile_addr(g, v, i)] = val;
        }
        c.sync();
        s = tile_fft<1>(s, s2, g, J.pb, J.twb, c);
        for (int e = c.tid; e < all; e += c.nthr) {
            const int i = ms_fastdiv(e, mgc), v = e - i * cnt;
            const int a = tile_addr(g, v, i);
            s[a] = c_swap(c_mul(s[a], __ldg(&J.b1_spec[i])));
        }
        c.sync();
        cpx* other = (s == sA) ? s2 : sA;
        s = tile_fft<1>(s, other, g, J.pb, J.twb, c);
        for (int e = c.tid; e < total; e += c.nthr) {
            const int k1 = ms_fastdiv(e, mgc), v = e - k1 * cnt;
            cpx val = c_mul(c_swap(s[tile_addr(g, v, k1)]), __ldg(&J.b1_chirp[k1]));
            if (TWID) val = c_mul(val, tw2level(J.twM_hi, J.twM_lo, (unsigned)k1 * (unsigned)(col0 + v)));
            job_store<ST>(J, k1 * F2 + col0 + v, val);
        }
        return;
    }
    if (LdPlain<LD>::v) {
        for (int e0 = c.tid; e0 < total; e0 += 4 * c.nthr) {
            cpx ld[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int e = e0 + u * c.nthr, i = ms_fastdiv(e, mgc), v = e - i * cnt;
                ld[u] = e < total ? job_load<LD>(J, i * F2 + col0 + v) : c_zero();
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int e = e0 + u * c.nthr, i = ms_fastdiv(e, mgc), v = e - i * cnt;
                if (e < total) s[tile_addr(g, v, i)] = ld[u];
            }
        }
    } else {
#pragma unroll 4
        for (int e = c.tid; e < total; e += c.nthr) {
            const int i = ms_fastdiv(e, mgc), v = e - i * cnt;
            s[tile_addr(g, v, i)] = job_load<LD>(J, i * F2 + col0 + v);
        }
    }
    c.sync();
    s = tile_fft<1>(s, s2, g, J.p1, J.tw1, c);
    if (TWID && c.nthr % cnt == 0) {
        // the thread keeps its column: stepped twiddles as in the static Bluestein tiles
        const int k10 = ms_fastdiv(c.tid, mgc);
        const unsigned col = (unsigned)(col0 + c.tid - k10 * cnt);
        cpx tw = tw_direct((unsigned)k10 * col, J.M);
        const cpx tstep = tw2level(J.twM_hi, J.twM_lo, (unsigned)(((long long)col * (c.nthr / cnt)) % J.M));
#pragma unroll 4
        for (int e = c.tid; e < total; e += c.nthr) {
            const int k1 = ms_fastdiv(e, mgc), v = e - k1 * cnt;
            job_store<ST>(J, k1 * F2 + col0 + v, c_mul(s[tile_addr(g, v, k1)], tw));
            tw = c_mul(tw, tstep);
        }
        return;
    }
#pragma unroll 4
    for (int e = c.tid; e < total; e += c.nthr) {
        const int k1 = ms_fastdiv(e, mgc), v = e - k1 * cnt;
        cpx val = s[tile_addr(g, v, k1)];
        if (TWID) val = c_mul(val, tw2level(J.twM_hi, J.twM_lo, (unsigned)k1 * (unsigned)(col0 + v)));
        job_store<ST>(J, k1 * F2 + col0 + v, val);
    }
}

// ---- rows kernel -----------------------------------------------------------------------------------
template <int LD, int MODE, int ST>
MS_DEV void fft_rows_body(const FftJob* MS_RESTRICT jobs, const Ctx& c) {
    const FftJob& J = stage_job(jobs, c);
    const int G = J.G, F1 = J.F1, F2 = J.F2;
    const int row0 = c.bx * G;
    if (row0 >= F1) return;
    const int cnt = (F1 - row0) < G ? (F1 - row0) : G;
    cpx* s = (cpx*)(c.smem + MS_JOB_SMEM);
    cpx* const sA = s;
    TileGeom g; g.cnt = cnt; g.vs = (ms_pad(F2) + 1) | 1; g.es = 1; g.colmajor = 0;
    cpx* s2 = s + (G * g.vs + 2);
    const int total = F2 * cnt;
    const unsigned mgF = J.p2.mg_F, mgc = ms_magic_dev(cnt);
    if (LdPlain<LD>::v) {
        for (int e0 = c.tid; e0 < total; e0 += 4 * c.nthr) {
            cpx ld[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int e = e0 + u * c.nthr, r = ms_fastdiv(e, mgF), i = e - r * F2;
                ld[u] = e < total ? job_load<LD>(J, (row0 + r) * F2 + i) : c_zero();
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int e = e0 + u * c.nthr, r = ms_fastdiv(e, mgF), i = e - r * F2;
                if (e < total) s[tile_addr(g, r, i)] = ld[u];
            }
        }
    } else {
#pragma unroll 4
        for (int e = c.tid; e < total; e += c.nthr) {
            const int r = ms_fastdiv(e, mgF), i = e - r * F2;
            s[tile_addr(g, r, i)] = job_load<LD>(J, (row0 + r) * F2 + i);
        }
    }
    c.sync();
    s = tile_fft<0>(s, s2, g, J.p2, J.tw2, c);
    if (MODE == MODE_NAT) {
        for (int e = c.tid; e < total; e += c.nthr) {
            const int k2 = ms_fastdiv(e, mgc), r = e - k2 * cnt;
            job_store<ST>(J, (row0 + r) + F1 * k2, s[tile_addr(g, r, k2)]);
        }
    } else if (MODE == MODE_RAW) {
        for (int e = c.tid; e < total; e += c.nthr) {
            const int r = ms_fastdiv(e, mgF), i = e - r * F2;
            job_store<ST>(J, (row0 + r) * F2 + i, s[tile_addr(g, r, i)]);
        }
    } else {   // MODE_CONV
#pragma unroll 4
        for (int e = c.tid; e < total; e += c.nthr) {
            const int r = ms_fastdiv(e, mgF), i = e - r * F2;
            const int a = tile_addr(g, r, i);
            s[a] = c_swap(c_mul(s[a], __ldg(&J.bspec[(row0 + r) * F2 + i])));
        }
        c.sync();
        cpx* other = (s == sA) ? s2 : sA;
        s = tile_fft<0>(s, other, g, J.p2, J.tw2, c);
#pragma unroll 4
        for (int e = c.tid; e < total; e += c.nthr) {
            const int r = ms_fastdiv(e, mgF), i = e - r * F2;
            cpx val = s[tile_addr(g, r, i)];
            if (F1 > 1) val = c_mul(val, tw2level(J.twM_hi, J.twM_lo, (unsigned)(row0 + r) * (unsigned)i));
            job_store<ST>(J, (row0 + r) * F2 + i, val);
        }
    }
}

// out[j] = exp(-i pi j^2 / n), j < n
MS_DEV void gen_chirp_body(cpx* out, int n, const Ctx& c, int grid_threads, int gtid) {
    for (int j = gtid; j < n; j += grid_threads) {
        const long long e = ((long long)j * (long long)j) % (2ll * n);
        double sn, cs;
        r_sincospi((double)e / (double)n, &sn, &cs);
        out[j] = mk((real)cs, (real)(-sn));
    }
}

// ---- table generators (float64 angles, rounded once) -------------------------------------------------
// out[i] = exp(-2 pi i * ((i * mul) mod N) / N),  i < count
MS_DEV void gen_table_body(cpx* out, int count, long long mul, long long N, const Ctx& c, int grid_threads, int gtid) {
    for (int i = gtid; i < count; i += grid_threads) {
        long long e = ((long long)i * mul) % N;
        double sn, cs;
        r_sincospi(2.0 * (double)e / (double)N, &sn, &cs);
        out[i] = mk((real)cs, (real)(-sn));
    }
}
