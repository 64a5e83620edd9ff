// ms_fft_host.h -- host side of the spectral engine: geometry planning, twiddle / chirp / Bluestein
// filter caches, and the kernel sequences.  Compiled by nvcc into the product and by g++ into the
// block emulator used by the CPU tests (same source, see ms_rt.cuh).

// largest vector one CTA transforms in shared memory / largest tile a CTA holds (two ping-pong buffers)
static const int MS_SMALL_MAX = sizeof(real) == 4 ? 8192 : 4096;
static const int MS_TILE_MAX = sizeof(real) == 4 ? 8192 : 4096;

// ---- kernel structs ----------------------------------------------------------------------------------
#ifndef MS_FFT_MINB
#define MS_FFT_MINB 2
#endif
#ifndef MS_SQ_MINB
#define MS_SQ_MINB 5
#endif
#ifndef MS_SB_MINB
#define MS_SB_MINB 5
#endif
template <int LD, int ST, int TWID, int SQ = 0, int SB = 0> struct ColsK {
    static constexpr int MAXT = ((SQ && sizeof(real) == 8) || SB) ? 256 : 512;      // static tiles: 2048 elements, 256 threads
    static constexpr int MINB = SB ? MS_SB_MINB : (SQ && sizeof(real) == 8) ? MS_SQ_MINB : MS_FFT_MINB;   // 2 x 512: <= 64 registers
    static MS_DEV void run(const FftJob* jobs, const Ctx& c) { fft_cols_body<LD, ST, TWID, SQ, SB>(jobs, c); }
};
#ifndef MS_WB_MINB
#define MS_WB_MINB 4
#endif
template <int LD, int ST, int TWID> struct ColsWarpK {              // in-tile Bluestein, B1 = 256, warp-local transforms
    static constexpr int MAXT = 256;
    static constexpr int MINB = MS_WB_MINB;
    static MS_DEV void run(const FftJob* jobs, const Ctx& c) { fft_cols_warp_body<LD, ST, TWID>(jobs, c); }
};
template <int LD, int ST, int TWID> struct ColsWarpPlainK {         // plain columns of 256 rows, warp-local transform
    static constexpr int MAXT = 256;
    static constexpr int MINB = MS_WB_MINB;
    static MS_DEV void run(const FftJob* jobs, const Ctx& c) { fft_cols_warp_plain_body<LD, ST, TWID>(jobs, c); }
};
#ifndef MS_WB5_MINB
#define MS_WB5_MINB 2
#endif
template <int LD, int ST, int TWID> struct ColsWarp512K {           // in-tile Bluestein, B1 = 512, warp-local transforms (16 values per lane)
    static constexpr int MAXT = 256;
    static constexpr int MINB = MS_WB5_MINB;
    static MS_DEV void run(const FftJob* jobs, const Ctx& c) { fft_cols_warp512_body<LD, ST, TWID>(jobs, c); }
};
template <int LD, int MODE, int ST, int SQ = 0> struct RowsK {
    static constexpr int MAXT = (SQ && sizeof(real) == 8) ? 256 : 512;
    static constexpr int MINB = (SQ && sizeof(real) == 8) ? MS_SQ_MINB : MS_FFT_MINB;
    static MS_DEV void run(const FftJob* jobs, const Ctx& c) { fft_rows_body<LD, MODE, ST, SQ>(jobs, c); }
};
#ifndef MS_SPECOP_MINB
#define MS_SPECOP_MINB 6          // 40 registers (the cold operator branches spill): 1.98 -> 1.62 ms over the sweep; 7 and 8 were slower
#endif
struct SpecOpK {                                                    // spectral operators, elementwise, in front of the inverse
    static constexpr int MAXT = SPECOP_NTHR;
    static constexpr int MINB = MS_SPECOP_MINB;
    static MS_DEV void run(const FftJob* jobs, const Ctx& c) { spec_op_body(jobs, c); }
};
// tile width of the static 256 x 256 kernels: what plan_direct picks for 65536 points in this precision
static const int MS_SQ = (sizeof(real) == 4 ? 8192 : 4096) / 2 / 256;
struct GenChirpK {
    static constexpr int MAXT = 256;
    static constexpr int MINB = 1;
    static MS_DEV void run(cpx* out, int n, const Ctx& c) { gen_chirp_body(out, n, c, c.nthr * 64, c.bx * c.nthr + c.tid); }
};
struct GenTableK {
    static constexpr int MAXT = 256;
    static constexpr int MINB = 1;
    static MS_DEV void run(cpx* out, int count, long long mul, long long N, const Ctx& c) {
        gen_table_body(out, count, mul, N, c, c.nthr * 64, c.bx * c.nthr + c.tid);
    }
};

static inline bool ms_is_smooth(long long n) {
    if (n < 1) return false;
    while (n % 2 == 0) n /= 2;
    while (n % 3 == 0) n /= 3;
    while (n % 5 == 0) n /= 5;
    return n == 1;
}
static inline int ms_round32(int x) { return (x + 31) / 32 * 32; }
// Length of the circular convolution that carries a Bluestein transform.  Any 2-3-5-smooth M >= need would do,
// but measured on B200 (C5 sweep, f64) smooth lengths lose to the next power of two even at equal pass count
// (270 in five passes: grain stage 17.1 -> 22.5 ms; 320 = 8*8*5 in three: 22.7 ms): radix-8 passes over 2^k tiles
// are the cheapest per element here.  So: the next power of two.
static inline int ms_conv_len(int need) {
    int p2 = 1; while (p2 < need) p2 <<= 1;
    return p2;
}

struct LaunchShape { int ept, nthr; size_t smem; unsigned gx; };

static inline int cols_tile_elems(const FftJob& J) { return J.T * (J.B1 ? J.B1 : J.F1); }
static inline int rows_tile_elems(const FftJob& J) { return J.G * J.F2; }
static inline int cols_rows(const FftJob& J) { return J.B1 ? J.B1 : J.F1; }
static inline size_t cols_smem(const FftJob& J) { return MS_JOB_SMEM + 2 * sizeof(cpx) * (size_t)(ms_pad((cols_rows(J) - 1) * J.T + J.T - 1) + 2); }
static inline size_t rows_smem(const FftJob& J) { return MS_JOB_SMEM + 2 * sizeof(cpx) * (size_t)(J.G * ((ms_pad(J.F2) + 1) | 1) + 2); }

static inline void shape_for(int tile, LaunchShape* s) {
    s->ept = 0;
    s->nthr = std::min(512, std::max(64, ms_round32((tile + 7) / 8)));     // one radix-8 butterfly per thread per pass
}

class FftEngine {
public:
    static FftEngine& get() { static FftEngine e; return e; }

    // Fill geometry + table pointers of J for logical length n.  Returns 0 / -1.
    int prepare(FftJob& J, int n, ms_stream_t st) {
        std::lock_guard<std::mutex> lk(mu_);
        return prepare_locked(J, n, st);
    }

    // jobs_dev: device copy of `jobs` (same order).  Jobs must be sorted by job_class().
    // + 4 * static Bluestein id (1..4 for B1 = 128, 256, 512, 1024 with 2048-element tiles of full columns)
    static int sb_id(const FftJob& J) {
        if (!J.B1 && !J.ch_hi && J.F1 == 256 && J.T == 8 && (J.n & (J.n - 1))) return 5;   // plain warp-local columns
        if (!J.B1 || J.ch_hi || J.T * J.B1 != MS_SB_TILE || J.F2 % J.T) return 0;
        return J.B1 == 128 ? 1 : J.B1 == 256 ? 2 : J.B1 == 512 ? 3 : J.B1 == 1024 ? 4 : 0;
    }
    static int job_class(const FftJob& J) { return (J.ch_hi ? 2 : 0) + (J.F1 > 1 ? 1 : 0) + 4 * sb_id(J); }

    // [b, e) ranges of equal job_class() inside [lo, hi): what run() turns into one launch sequence each
    static std::vector<std::pair<size_t, size_t>> class_ranges(const std::vector<FftJob>& jobs, size_t lo = 0, size_t hi = (size_t)-1) {
        std::vector<std::pair<size_t, size_t>> out;
        const size_t end = std::min(hi, jobs.size());
        size_t b = lo;
        while (b < end) {
            const int cls = job_class(jobs[b]);
            size_t e = b;
            while (e < end && job_class(jobs[e]) == cls && e - b < 32768) ++e;
            out.emplace_back(b, e);
            b = e;
        }
        return out;
    }
    // forward: pair (in_a,in_b) -> Z ;  inverse: spec op on Z -> (out_a,out_b)
    // (all entry points take an optional [lo, hi) job range so callers can walk a batch in L2-sized groups)
    int forward(const std::vector<FftJob>& jobs, const FftJob* jobs_dev, ms_stream_t st, size_t lo = 0, size_t hi = (size_t)-1) { return run(jobs, jobs_dev, st, 0, lo, hi); }
    int inverse(const std::vector<FftJob>& jobs, const FftJob* jobs_dev, ms_stream_t st, size_t lo = 0, size_t hi = (size_t)-1) { return run(jobs, jobs_dev, st, 1, lo, hi); }
    // complex natural-order transform cin -> cout (direct lengths only; test entry)
    int c2c(const std::vector<FftJob>& jobs, const FftJob* jobs_dev, ms_stream_t st) { return run(jobs, jobs_dev, st, 2); }
    // filter spectrum: real taps at in_a (n of them) -> FFT_M / M in [k1][k2] layout at `work`
    int filter_spectrum(const std::vector<FftJob>& jobs, const FftJob* jobs_dev, ms_stream_t st, size_t lo = 0, size_t hi = (size_t)-1) { return run(jobs, jobs_dev, st, 3, lo, hi); }
    // combined filter spectrum: real reflection taps at in_a -> IR spectrum (cin) * (1 + FFT_M(taps)) at `work`
    int filter_compose(const std::vector<FftJob>& jobs, const FftJob* jobs_dev, ms_stream_t st, size_t lo = 0, size_t hi = (size_t)-1) { return run(jobs, jobs_dev, st, 5, lo, hi); }
    // overlap-save: two blocks per job, multiplied by `bspec`, valid outputs stored
    int overlap_save(const std::vector<FftJob>& jobs, const FftJob* jobs_dev, ms_stream_t st, size_t lo = 0, size_t hi = (size_t)-1) { return run(jobs, jobs_dev, st, 4, lo, hi); }
    // partitioned overlap-save (ms_fir_long.cuh), direct lengths only.  Forward: two blocks of real input as re / im (LD_OLS:
    // in_a / in_b at p0_a / p0_b, zero outside [0, ols_n)) -> natural-order spectrum * out_scale at `cout`.  Inverse: the
    // natural-order swap(Y) at `cin` -> its transform, i.e. swap(M * IFFT(Y)) -> valid outputs of both blocks (ST_OLS).
    int ols_forward(const std::vector<FftJob>& jobs, const FftJob* jobs_dev, ms_stream_t st) { return run(jobs, jobs_dev, st, 6); }
    int ols_inverse(const std::vector<FftJob>& jobs, const FftJob* jobs_dev, ms_stream_t st) { return run(jobs, jobs_dev, st, 7); }

private:
    std::mutex mu_;
    std::map<int, cpx*> wtab_;                                  // F -> w_F^i
    std::map<long long, std::pair<cpx*, cpx*>> two_level_;   // modulus N -> (hi, lo)
    std::map<int, cpx*> bspec_;                                 // n -> Bluestein filter spectrum
    std::map<int, FftJob> geom_;                                   // n -> prepared geometry template

    template <class K, class... A>
    static int L(unsigned gx, unsigned gy, int nthr, size_t smem, ms_stream_t st, A... a) {
        MsDim g; g.x = gx; g.y = gy;
        return ms_launch<K>(g, nthr, smem, st, a...);
    }

    int get_wtab(int F, ms_stream_t st, const cpx** out) {
        auto it = wtab_.find(F);
        if (it == wtab_.end()) {
            cpx* p = (cpx*)ms_dev_alloc(sizeof(cpx) * (size_t)F);
            if (!p) MS_FAIL("out of device memory for twiddle table F=%d", F);
            if (L<GenTableK>(64, 1, 256, 0, st, p, F, 1ll, (long long)F)) return -1;
            it = wtab_.emplace(F, p).first;
        }
        *out = it->second;
        return 0;
    }
    int get_two_level(long long N, ms_stream_t st, const cpx** hi, const cpx** lo) {
        auto it = two_level_.find(N);
        if (it == two_level_.end()) {
            int nhi = (int)((N + 1023) / 1024) + 1;
            cpx* ph = (cpx*)ms_dev_alloc(sizeof(cpx) * (size_t)nhi);
            cpx* pl = (cpx*)ms_dev_alloc(sizeof(cpx) * 1024);
            if (!ph || !pl) MS_FAIL("out of device memory for two-level table N=%lld", N);
            if (L<GenTableK>(64, 1, 256, 0, st, ph, nhi, 1024ll, N)) return -1;
            if (L<GenTableK>(64, 1, 256, 0, st, pl, 1024, 1ll, N)) return -1;
            it = two_level_.emplace(N, std::make_pair(ph, pl)).first;
        }
        *hi = it->second.first; *lo = it->second.second;
        return 0;
    }

    // Per-element cost of the in-tile Bluestein columns by convolution length (<= 128, 256, 512, 1024) and of one radix-2
    // level of the rows pass, relative to the warp-local 256 kernel.  Measured on B200 (C5 sweep, f64, per padded element):
    // 128: 1.4, 256: 1.0, 512 (warp-local): 1.45, 1024 (block-wide tile): 2.45 -- so a longer convolution has to buy a much
    // better padding ratio to be chosen (step 31.2 -> 30.8 ms against the analytic cost).  Development switch
    // MS_PLAN_W="c128,c256,c512,c1024,rows" overrides; MS_PLAN_W=0 selects the analytic cost.
    static const double* mixed_weights() {
        static double w[5] = {1.4, 1.0, 1.45, 2.45, 0.02}; static int init = 0;
        if (!init) {
            init = 1;
            const char* e = getenv("MS_PLAN_W");
            if (e && sscanf(e, "%lf,%lf,%lf,%lf,%lf", &w[0], &w[1], &w[2], &w[3], &w[4]) != 5) w[0] = -1;
        }
        return w;
    }
    static bool plan_direct(int n, FftJob& J) {
        if (!ms_is_smooth(n)) return false;
        J.M = n;
        if (n <= MS_SMALL_MAX) { J.F1 = 1; J.F2 = n; J.T = 1; J.G = 1; return true; }
        int best = 0; long long best_cost = -1;
        for (int f1 = 2; f1 <= 2048 && f1 < n; ++f1) {
            if (n % f1) continue;
            int f2 = n / f1;
            if (f2 > 2048 || f2 < 2) continue;
            long long cost = (long long)std::max(f1, f2) + ((f1 > 512 || f2 > 512) ? 100000 : 0)
                           + ((f1 > 1024 || f2 > 1024) ? 1000000 : 0);
            if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = f1; }
        }
        if (!best) return false;
        J.F1 = best; J.F2 = n / best;
        J.T = 16; J.G = 16;
        // smooth n with 256 | n (not a power of two: those belong to the FIR stage's static kernels): columns of exactly 256
        // rows run as one warp-local transform each -- a third of the generic tile's cost per element
        if ((n & (n - 1)) && n % 256 == 0 && n / 256 >= 16 && n / 256 <= MS_TILE_MAX / 4) {
            J.F1 = 256; J.F2 = n / 256; J.T = 8;
            while (J.G > 4 && J.G * J.F2 > MS_TILE_MAX / 2) J.G /= 2;
            while (J.G > 1 && J.G * J.F2 > MS_TILE_MAX) J.G /= 2;
            return true;
        }
        while (J.T > 4 && J.T * J.F1 > MS_TILE_MAX / 2) J.T /= 2;       // half tiles (<= 74 KB in f64): three CTAs per SM
        while (J.G > 4 && J.G * J.F2 > MS_TILE_MAX / 2) J.G /= 2;
        while (J.T > 1 && J.T * J.F1 > MS_TILE_MAX) J.T /= 2;
        while (J.G > 1 && J.G * J.F2 > MS_TILE_MAX) J.G /= 2;
        return true;
    }
    // n = F1 * F2 with F2 smooth (rows kernel) and F1 arbitrary, done in the columns kernel as an in-tile
    // Bluestein of length B1 = pow2 >= 2 F1 - 1.  Same global traffic as the direct two-pass transform.
    static bool plan_mixed(int n, FftJob& J) {
        const int tile_target = MS_TILE_MAX / 2;
        int best = 0; double best_cost = 0;
        for (int f2 = 16; f2 <= MS_TILE_MAX && f2 < n; ++f2) {
            if (n % f2 || !ms_is_smooth(f2)) continue;
            const int f1 = n / f2;
            if (f1 < 2 || ms_is_smooth(f1)) continue;
            const int b1 = ms_conv_len(2 * f1 - 1);
            if (b1 * 4 > MS_TILE_MAX) continue;
            const int T = std::max(1, std::min(16, tile_target / b1)), G = std::max(1, std::min(16, tile_target / f2));
            double lg2 = 0, lgb = 0;
            for (int t = f2; t > 1; t >>= 1) lg2 += 1;
            for (int t = b1; t > 1; t >>= 1) lgb += 1;
            double cost = lg2 + 2.0 * lgb * (double)b1 / (double)f1 + (T < 8 ? 16.0 / T : 0) + (G < 8 ? 16.0 / G : 0);
            if (mixed_weights()[0] > 0) {
                // measured form: padded elements per useful one times the per-element cost of that columns kernel
                const double* w = mixed_weights();
                const double cb = b1 <= 128 ? w[0] : b1 == 256 ? w[1] : b1 == 512 ? w[2] : b1 == 1024 ? w[3] : w[3] * (double)b1 / 1024.0;
                cost = w[4] * lg2 + cb * (double)b1 / (double)f1 + (T < 8 ? 16.0 / T : 0) + (G < 8 ? 16.0 / G : 0);
            }
            if (!best || cost < best_cost) { best = f2; best_cost = cost; }
        }
        if (!best) return false;
        J.M = n; J.F2 = best; J.F1 = n / best;
        const int b1 = ms_conv_len(2 * J.F1 - 1);
        J.B1 = b1;
        J.T = std::max(1, std::min(16, tile_target / b1));
        J.G = std::max(1, std::min(16, tile_target / J.F2));
        return true;
    }
    static bool plan_bluestein(int n, FftJob& J) {
        long long need = 2ll * n - 1, M = 1; int lg = 0;
        while (M < need) { M <<= 1; ++lg; }
        if (M > (1ll << 22)) return false;
        J.M = (int)M;
        if (M <= MS_SMALL_MAX) { J.M = ms_conv_len((int)need); J.F1 = 1; J.F2 = J.M; J.T = 1; J.G = 1; return true; }
        int l1 = std::min(lg / 2, 9);
        J.F1 = 1 << l1; J.F2 = (int)(M >> l1);
        if (J.F2 > MS_TILE_MAX) return false;
        J.T = 16;
        while (J.T > 1 && J.T * J.F1 > MS_TILE_MAX / 2) J.T /= 2;
        J.G = std::max(1, std::min(16, (MS_TILE_MAX / 2) / J.F2));
        return true;
    }

    int prepare_locked(FftJob& J, int n, ms_stream_t st) {
        if (n < 1) MS_FAIL("fft: bad length %d", n);
        auto it = geom_.find(n);
        if (it == geom_.end()) {
            FftJob g; memset(&g, 0, sizeof g);
            g.n = n;
            bool blu = false, mixed = false;
            if (!plan_direct(n, g)) {
                if (n > MS_SMALL_MAX / 2 && plan_mixed(n, g)) mixed = true;
                else { blu = true; if (!plan_bluestein(n, g)) MS_FAIL("fft: length %d unsupported", n); }
            }
            if (!ms_make_radix_plan(g.F2, &g.p2)) MS_FAIL("fft: cannot factor %d", g.F2);
            if (get_wtab(g.F2, st, &g.tw2)) return -1;
            if (mixed) {
                // borrow the small Bluestein plan of length F1: its filter spectrum (natural order) and radix plan
                FftJob sub; memset(&sub, 0, sizeof sub);
                if (prepare_locked(sub, g.F1, st)) return -1;
                if (!sub.ch_hi || sub.F1 != 1 || sub.M != g.B1) MS_FAIL("fft: internal: sub-plan of %d is not a small Bluestein", g.F1);
                g.pb = sub.p2; g.twb = sub.tw2; g.b1_spec = sub.bspec;
                cpx* ch = (cpx*)ms_dev_alloc(sizeof(cpx) * (size_t)g.F1);
                if (!ch) MS_FAIL("out of device memory for chirp table");
                if (L<GenChirpK>(64, 1, 256, 0, st, ch, g.F1)) return -1;
                g.b1_chirp = ch;
                if (get_two_level(g.M, st, &g.twM_hi, &g.twM_lo)) return -1;
            } else if (g.F1 > 1) {
                if (!ms_make_radix_plan(g.F1, &g.p1)) MS_FAIL("fft: cannot factor %d", g.F1);
                if (get_wtab(g.F1, st, &g.tw1)) return -1;
                if (get_two_level(g.M, st, &g.twM_hi, &g.twM_lo)) return -1;
            }
            if (blu) {
                if (get_two_level(2ll * n, st, &g.ch_hi, &g.ch_lo)) return -1;
                if (make_bspec(g, st)) return -1;
            }
            it = geom_.emplace(n, g).first;
        }
        const FftJob& g = it->second;
        J.n = g.n; J.M = g.M; J.F1 = g.F1; J.F2 = g.F2; J.T = g.T; J.G = g.G;
        J.p1 = g.p1; J.p2 = g.p2; J.tw1 = g.tw1; J.tw2 = g.tw2; J.twM_hi = g.twM_hi; J.twM_lo = g.twM_lo;
        J.ch_hi = g.ch_hi; J.ch_lo = g.ch_lo; J.bspec = g.bspec;
        J.B1 = g.B1; J.pb = g.pb; J.twb = g.twb; J.b1_chirp = g.b1_chirp; J.b1_spec = g.b1_spec;
        return 0;
    }

    int make_bspec(FftJob& g, ms_stream_t st) {
        cpx* spec = (cpx*)ms_dev_alloc(sizeof(cpx) * (size_t)g.M);
        FftJob* jd = (FftJob*)ms_dev_alloc(sizeof(FftJob));
        if (!spec || !jd) MS_FAIL("out of device memory for Bluestein spectrum n=%d M=%d", g.n, g.M);
        FftJob t = g; t.work = spec; t.bspec = nullptr;
        if (ms_h2d(jd, &t, sizeof t, st)) return -1;
        LaunchShape s;
        if (g.F1 == 1) {
            shape_for(rows_tile_elems(t), &s);
            if (launch_rows<LD_BW, MODE_RAW, ST_WORK>(s.ept, 1, 1, s.nthr, rows_smem(t), st, jd)) return -1;
        } else {
            shape_for(cols_tile_elems(t), &s);
            if (launch_cols<LD_BW, ST_WORK, 1>(s.ept, (t.F2 + t.T - 1) / t.T, 1, s.nthr, cols_smem(t), st, jd)) return -1;
            shape_for(rows_tile_elems(t), &s);
            if (launch_rows<LD_WORK, MODE_RAW, ST_WORK>(s.ept, (t.F1 + t.G - 1) / t.G, 1, s.nthr, rows_smem(t), st, jd)) return -1;
        }
#ifndef MS_HOST_EMUL
        MS_CUDA_OK(cudaStreamSynchronize(st));
#endif
        ms_dev_free(jd);
        g.bspec = spec;
        bspec_[g.n] = spec;
        return 0;
    }

    template <int LD, int ST, int TWID, int SQ = 0>
    static int launch_cols(int ept, unsigned gx, unsigned gy, int nthr, size_t smem, ms_stream_t st, const FftJob* jd) {
        return L<ColsK<LD, ST, TWID, SQ>>(gx, gy, nthr, smem, st, jd);
    }
    // in-tile Bluestein columns with static convolution length (sb = sb_id): 256 threads, one tile buffer
    template <int LD, int ST, int TWID>
    static int launch_cols_sb(int sb, unsigned gx, unsigned gy, ms_stream_t st, const FftJob* jd) {
        const size_t smem = MS_JOB_SMEM + sizeof(cpx) * (size_t)(MS_SB_TILE + MS_SB_TILE / 8 + 4);
        switch (sb) {
            case 1: return L<ColsK<LD, ST, TWID, 0, 128>>(gx, gy, 256, smem, st, jd);
            case 2:
                if (sb_warp()) return L<ColsWarpK<LD, ST, TWID>>(gx, gy, 256, MS_JOB_SMEM + sizeof(cpx) * (size_t)(8 * WB_RS), st, jd);
                return L<ColsK<LD, ST, TWID, 0, 256>>(gx, gy, 256, smem, st, jd);
            case 3:
                if (sb_warp() && LdPlain<LD>::v) return L<ColsWarp512K<LD, ST, TWID>>((gx + 1) / 2, gy, 256, MS_JOB_SMEM + sizeof(cpx) * (size_t)(8 * WB5_RS), st, jd);
                return L<ColsK<LD, ST, TWID, 0, 512>>(gx, gy, 256, smem, st, jd);
            case 5:
                if (LdPlain<LD>::v) return L<ColsWarpPlainK<LD, ST, TWID>>(gx, gy, 256, MS_JOB_SMEM + sizeof(cpx) * (size_t)(8 * WB_RS), st, jd);
                return -1;
            default: return L<ColsK<LD, ST, TWID, 0, 1024>>(gx, gy, 256, smem, st, jd);
        }
    }
    // development switch MS_SPEC_PASS=0: the operators inside the load functor of the inverse columns (round 1 form)
    static bool spec_pass() { static int v = -1; if (v < 0) { const char* e = getenv("MS_SPEC_PASS"); v = (e && e[0] == '0') ? 0 : 1; } return v != 0; }
    // development switch MS_SB_WARP=0: the block-wide B1 = 256 kernel instead of the warp-local one
    static bool sb_warp() { static int v = -1; if (v < 0) { const char* e = getenv("MS_SB_WARP"); v = (e && e[0] == '0') ? 0 : 1; } return v != 0; }
    template <int LD, int MODE, int ST, int SQ = 0>
    static int launch_rows(int ept, unsigned gx, unsigned gy, int nthr, size_t smem, ms_stream_t st, const FftJob* jd) {
        return L<RowsK<LD, MODE, ST, SQ>>(gx, gy, nthr, smem, st, jd);
    }
    // shared memory of the static kernels: the job + ONE tile (the static passes run in place)
    static size_t sq_smem(bool cols) {
        FftJob t; t.T = t.G = MS_SQ; t.F1 = t.F2 = 256; t.B1 = 0;
        return MS_JOB_SMEM + ((cols ? cols_smem(t) : rows_smem(t)) - MS_JOB_SMEM) / 2;
    }
    // every job of [b, e) is a plain 256 x 256 transform with the static tile width: the FIR stage's 65536-point blocks
    static bool all_square(const std::vector<FftJob>& jobs, size_t b, size_t e) {
        for (size_t i = b; i < e; ++i) {
            const FftJob& J = jobs[i];
            if (J.F1 != 256 || J.F2 != 256 || J.T != MS_SQ || J.G != MS_SQ || J.B1 || J.ch_hi) return false;
        }
        return e > b;
    }

    struct ClassShape { LaunchShape cols, rows; };
    static ClassShape class_shape(const std::vector<FftJob>& jobs, size_t b, size_t e) {
        ClassShape cs; int tc = 0, tr = 0; size_t sc = 0, sr = 0; unsigned gc = 0, gr = 0;
        for (size_t i = b; i < e; ++i) {
            const FftJob& J = jobs[i];
            tr = std::max(tr, rows_tile_elems(J)); sr = std::max(sr, rows_smem(J));
            gr = std::max(gr, (unsigned)((J.F1 + J.G - 1) / J.G));
            if (J.F1 > 1) {
                tc = std::max(tc, cols_tile_elems(J)); sc = std::max(sc, cols_smem(J));
                gc = std::max(gc, (unsigned)((J.F2 + J.T - 1) / J.T));
            }
        }
        shape_for(std::max(tc, 1), &cs.cols); cs.cols.smem = sc; cs.cols.gx = gc;
        shape_for(std::max(tr, 1), &cs.rows); cs.rows.smem = sr; cs.rows.gx = gr;
        return cs;
    }

    // what: 0 forward (pair -> Z), 1 inverse (spec(Z) -> pair), 2 c2c test path, 3 / 5 filter spectra, 4 overlap-save,
    // 6 / 7 forward / inverse of the partitioned overlap-save
    int run(const std::vector<FftJob>& jobs, const FftJob* jobs_dev, ms_stream_t st, int what, size_t lo = 0, size_t hi = (size_t)-1) {
        const size_t end = std::min(hi, jobs.size());
        size_t b = lo;
        while (b < end) {
            const int full_cls = job_class(jobs[b]);
            const int cls = full_cls & 3, sb = full_cls >> 2;
            size_t e = b;
            while (e < end && job_class(jobs[e]) == full_cls && e - b < 32768) ++e;
            const ClassShape cs = class_shape(jobs, b, e);
            const unsigned gy = (unsigned)(e - b);
            const FftJob* jd = jobs_dev + b;
            const LaunchShape &C = cs.cols, &R = cs.rows;
            int rc = 0;
            if (what == 3) {
                if (cls == 0) rc = launch_rows<LD_REALPAD, MODE_RAW, ST_WORK>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd);
                else if (cls == 1) {
                    rc = launch_cols<LD_REALPAD, ST_WORK, 1>(C.ept, C.gx, gy, C.nthr, C.smem, st, jd);
                    if (!rc) rc = launch_rows<LD_WORK, MODE_RAW, ST_WORK>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd);
                } else MS_FAIL("filter spectrum needs a direct length");
            } else if (what == 5) {
                if (cls == 0) rc = launch_rows<LD_REALPAD, MODE_RAW, ST_HMUL>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd);
                else if (cls == 1) {
                    // (summing the few non-zero input rows of the tap vector directly in the rows kernel, instead of
                    //  the columns pass, was measured SLOWER on B200: 7.8 ms vs 2.95 + 3.79 ms for the C5 sweep)
                    if (all_square(jobs, b, e)) {
                        rc = launch_cols<LD_REALPAD, ST_WORK, 1, MS_SQ>(C.ept, C.gx, gy, C.nthr, sq_smem(true), st, jd);
                        if (!rc) rc = launch_rows<LD_WORK, MODE_RAW, ST_HMUL, MS_SQ>(R.ept, R.gx, gy, R.nthr, sq_smem(false), st, jd);
                    } else {
                    rc = launch_cols<LD_REALPAD, ST_WORK, 1>(C.ept, C.gx, gy, C.nthr, C.smem, st, jd);
                    if (!rc) rc = launch_rows<LD_WORK, MODE_RAW, ST_HMUL>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd);
                    }
                } else MS_FAIL("filter spectrum needs a direct length");
            } else if (what == 4) {
                if (cls == 0) rc = launch_rows<LD_OLS, MODE_CONV, ST_OLS>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd);
                else if (cls == 1 && all_square(jobs, b, e)) {
                    rc = launch_cols<LD_OLS, ST_WORK, 1, MS_SQ>(C.ept, C.gx, gy, C.nthr, sq_smem(true), st, jd);
                    if (!rc) rc = launch_rows<LD_WORK, MODE_CONV, ST_WORK, MS_SQ>(R.ept, R.gx, gy, R.nthr, sq_smem(false), st, jd);
                    if (!rc) rc = launch_cols<LD_WORK, ST_OLS, 0, MS_SQ>(C.ept, C.gx, gy, C.nthr, sq_smem(true), st, jd);
                } else if (cls == 1) {
                    rc = launch_cols<LD_OLS, ST_WORK, 1>(C.ept, C.gx, gy, C.nthr, C.smem, st, jd);
                    if (!rc) rc = launch_rows<LD_WORK, MODE_CONV, ST_WORK>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd);
                    if (!rc) rc = launch_cols<LD_WORK, ST_OLS, 0>(C.ept, C.gx, gy, C.nthr, C.smem, st, jd);
                } else MS_FAIL("overlap-save needs a direct length");
            } else if (what == 6 || what == 7) {
                if (cls == 0) rc = what == 6 ? launch_rows<LD_OLS, MODE_NAT, ST_CPX>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd)
                                             : launch_rows<LD_CPX, MODE_NAT, ST_OLS>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd);
                else if (cls == 1) {
                    rc = what == 6 ? launch_cols<LD_OLS, ST_WORK, 1>(C.ept, C.gx, gy, C.nthr, C.smem, st, jd)
                                   : launch_cols<LD_CPX, ST_WORK, 1>(C.ept, C.gx, gy, C.nthr, C.smem, st, jd);
                    if (!rc) rc = what == 6 ? launch_rows<LD_WORK, MODE_NAT, ST_CPX>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd)
                                            : launch_rows<LD_WORK, MODE_NAT, ST_OLS>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd);
                } else MS_FAIL("partitioned overlap-save needs a direct length");
            } else if (what == 2) {
                if (cls == 0) rc = launch_rows<LD_CPX, MODE_NAT, ST_CPX>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd);
                else if (cls == 1) {
                    rc = launch_cols<LD_CPX, ST_WORK, 1>(C.ept, C.gx, gy, C.nthr, C.smem, st, jd);
                    if (!rc) rc = launch_rows<LD_WORK, MODE_NAT, ST_CPX>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd);
                } else MS_FAIL("c2c test path supports direct lengths only");
            } else if (cls == 0) {
                rc = what == 0 ? launch_rows<LD_PAIR, MODE_NAT, ST_Z>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd)
                               : launch_rows<LD_SPEC, MODE_NAT, ST_PAIR>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd);
            } else if (cls == 1) {
                if (what == 0) {
                    rc = sb ? launch_cols_sb<LD_PAIR, ST_WORK, 1>(sb, C.gx, gy, st, jd)
                            : launch_cols<LD_PAIR, ST_WORK, 1>(C.ept, C.gx, gy, C.nthr, C.smem, st, jd);
                    if (!rc) rc = launch_rows<LD_WORK, MODE_NAT, ST_Z>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd);
                } else if (spec_pass()) {
                    // operators in their own elementwise pass (Z -> work), then the inverse in place in `work`: a columns
                    // tile reads exactly the positions it writes back
                    int nmax = 0;
                    for (size_t i = b; i < e; ++i) nmax = std::max(nmax, jobs[i].n);
                    const unsigned gxo = (unsigned)((nmax / 2 + 1 + SPECOP_NTHR * SPECOP_PER - 1) / (SPECOP_NTHR * SPECOP_PER));
                    rc = L<SpecOpK>(gxo, gy, SPECOP_NTHR, MS_JOB_SMEM, st, jd);
                    if (!rc) rc = sb ? launch_cols_sb<LD_WORK, ST_WORK, 1>(sb, C.gx, gy, st, jd)
                                     : launch_cols<LD_WORK, ST_WORK, 1>(C.ept, C.gx, gy, C.nthr, C.smem, st, jd);
                    if (!rc) rc = launch_rows<LD_WORK, MODE_NAT, ST_PAIR>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd);
                } else {
                    rc = (sb && sb != 5) ? launch_cols_sb<LD_SPEC, ST_WORK, 1>(sb, C.gx, gy, st, jd)
                                         : launch_cols<LD_SPEC, ST_WORK, 1>(C.ept, C.gx, gy, C.nthr, C.smem, st, jd);
                    if (!rc) rc = launch_rows<LD_WORK, MODE_NAT, ST_PAIR>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd);
                }
            } else if (cls == 2) {
                rc = what == 0 ? launch_rows<LD_PAIR_CHIRP, MODE_CONV, ST_Z_CHIRP>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd)
                               : launch_rows<LD_SPEC_CHIRP, MODE_CONV, ST_PAIR_CHIRP>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd);
            } else {
                if (what == 0) rc = launch_cols<LD_PAIR_CHIRP, ST_WORK, 1>(C.ept, C.gx, gy, C.nthr, C.smem, st, jd);
                else rc = launch_cols<LD_SPEC_CHIRP, ST_WORK, 1>(C.ept, C.gx, gy, C.nthr, C.smem, st, jd);
                if (!rc) rc = launch_rows<LD_WORK, MODE_CONV, ST_WORK>(R.ept, R.gx, gy, R.nthr, R.smem, st, jd);
                if (!rc) {
                    if (what == 0) rc = launch_cols<LD_WORK, ST_Z_CHIRP, 0>(C.ept, C.gx, gy, C.nthr, C.smem, st, jd);
                    else rc = launch_cols<LD_WORK, ST_PAIR_CHIRP, 0>(C.ept, C.gx, gy, C.nthr, C.smem, st, jd);
                }
            }
            if (rc) return rc;
            b = e;
        }
        return 0;
    }
};
