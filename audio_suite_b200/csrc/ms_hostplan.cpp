// ms_hostplan.cpp -- native host planner (g++, no CUDA): the scalar half of render() (main_v2.py:589-646, 742-753,
// 760-781) and the job-table packing for the common family of renders -- the five gen_basic generators, Single or
// Poisson event fields, band-limit / power warp / stretch / multiband operators, reflection cloud, impulse response,
// stereo, soft clip -- i.e. what a preset sweep consists of.  Everything else stays with the Python planner
// (plan.py / tables.py), which is also the specification this file is tested against: tests/test_hostplan.py demands
// identical tables, bit for bit, on randomised parameter sets.
//
// Randomness is numpy's, restated: SeedSequence (numpy/random/bit_generator.pyx), PCG64 XSL-RR 128/64
// (numpy/random/src/pcg64), Generator.uniform / random / integers (Lemire, 32-bit halves buffered in the bit
// generator) / exponential (256-layer ziggurat, tables read out of numpy's libnpyrandom.a by
// oracle/extract_zig_tables.py).  Python's round() is half-to-even = nearbyint() in the default rounding mode; the
// floating-point expressions are written in the reference's operation order and the file is compiled with
// -ffp-contract=off so nothing is fused.  exp() of the reflection gains is left to numpy (np.exp and libm's exp differ
// in the last bit for ~5 % of arguments): the planner hands back delays and raw gains.
#include <stdint.h>
#include <string.h>
#include <math.h>
#include <vector>
#include <string>
#include <algorithm>
#include <atomic>
#include <thread>
#include <numeric>
#include "../../include/microsound_b200.h"
#include "ms_zig_exp_tables.h"

namespace {

typedef unsigned __int128 u128;

// ---- SeedSequence(entropy = non-negative int).generate_state(4, uint64) ---------------------------------------------
static const uint32_t SS_INIT_A = 0x43b0d7e5u, SS_MULT_A = 0x931e8875u, SS_INIT_B = 0x8b51f9ddu, SS_MULT_B = 0x58f38dedu;
static const uint32_t SS_MIX_L = 0xca01f9ddu, SS_MIX_R = 0x4973f715u;
static inline uint32_t ss_hashmix(uint32_t value, uint32_t& hc) {
    value ^= hc; hc *= SS_MULT_A; value *= hc; value ^= value >> 16; return value;
}
static inline uint32_t ss_mix(uint32_t x, uint32_t y) {
    uint32_t r = SS_MIX_L * x - SS_MIX_R * y; r ^= r >> 16; return r;
}
static void seed_sequence_state(uint64_t entropy, uint64_t out[4]) {
    uint32_t ent[2]; int ne = 1;
    ent[0] = (uint32_t)(entropy & 0xffffffffu); ent[1] = (uint32_t)(entropy >> 32);
    if (ent[1]) ne = 2;
    uint32_t pool[4], hc = SS_INIT_A;
    for (int i = 0; i < 4; ++i) pool[i] = ss_hashmix(i < ne ? ent[i] : 0u, hc);
    for (int s = 0; s < 4; ++s) for (int d = 0; d < 4; ++d) if (s != d) pool[d] = ss_mix(pool[d], ss_hashmix(pool[s], hc));
    uint32_t w[8], hb = SS_INIT_B;
    for (int i = 0; i < 8; ++i) {
        uint32_t v = pool[i & 3];
        v ^= hb; hb *= SS_MULT_B; v *= hb; v ^= v >> 16;
        w[i] = v;
    }
    for (int i = 0; i < 4; ++i) out[i] = (uint64_t)w[2 * i] | ((uint64_t)w[2 * i + 1] << 32);
}

// ---- PCG64 ----------------------------------------------------------------------------------------------------------
struct Pcg64 {
    u128 state, inc; int has32; uint32_t half;
    static u128 mult() { return ((u128)0x2360ED051FC65DA4ull << 64) | (u128)0x4385DF649FCCF645ull; }
    void seed(uint64_t entropy) {
        uint64_t v[4]; seed_sequence_state(entropy, v);
        const u128 initstate = ((u128)v[0] << 64) | v[1], initseq = ((u128)v[2] << 64) | v[3];
        state = 0; inc = (initseq << 1) | 1;
        step(); state += initstate; step();
        has32 = 0; half = 0;
    }
    void step() { state = state * mult() + inc; }
    uint64_t next64() {
        step();
        const uint64_t hi = (uint64_t)(state >> 64), lo = (uint64_t)state;
        const uint64_t x = hi ^ lo; const unsigned rot = (unsigned)(hi >> 58);
        return (x >> rot) | (x << ((64u - rot) & 63u));
    }
    uint32_t next32() {
        if (has32) { has32 = 0; return half; }
        const uint64_t n = next64();
        has32 = 1; half = (uint32_t)(n >> 32);
        return (uint32_t)(n & 0xffffffffu);
    }
    double next_double() { return (double)(next64() >> 11) * (1.0 / 9007199254740992.0); }
    double uniform(double lo, double hi) { return lo + (hi - lo) * next_double(); }       // Generator.uniform: low + (high - low) * U
    // Generator.integers(0, high) for 0 < high <= 2^32 (numpy: bounded_lemire_uint32 on rng = high - 1)
    uint64_t integers(uint64_t high) {
        const uint64_t rng = high - 1;
        if (rng == 0) return 0;
        if (rng == 0xFFFFFFFFull) return next32();
        const uint32_t rng_excl = (uint32_t)rng + 1u;
        uint64_t m = (uint64_t)next32() * rng_excl;
        uint32_t leftover = (uint32_t)m;
        if (leftover < rng_excl) {
            const uint32_t threshold = (0xFFFFFFFFu - (uint32_t)rng) % rng_excl;
            while (leftover < threshold) { m = (uint64_t)next32() * rng_excl; leftover = (uint32_t)m; }
        }
        return m >> 32;
    }
    double standard_exponential() {
        for (;;) {
            uint64_t ri = next64();
            ri >>= 3;
            const unsigned idx = (unsigned)(ri & 0xFF);
            ri >>= 8;
            double we; memcpy(&we, &MS_ZIG_WE_BITS[idx], 8);
            const double x = (double)ri * we;
            if (ri < MS_ZIG_KE[idx]) return x;
            if (idx == 0) return 7.69711747013104972 - log1p(-next_double());
            double f0, f1; memcpy(&f0, &MS_ZIG_FE_BITS[idx - 1], 8); memcpy(&f1, &MS_ZIG_FE_BITS[idx], 8);
            if ((f0 - f1) * next_double() + f1 < exp(-x)) return x;
        }
    }
};

// Python round(): half to even.  In the default rounding mode adding and subtracting 1.5 * 2^52 rounds |x| < 2^51 to the
// nearest integer, ties to even, exactly like nearbyint() -- without the libm call (this runs per reflection tap).
static inline double py_round(double x) {
    if (fabs(x) < 2251799813685248.0) { volatile double t = x + 6755399441055744.0; return t - 6755399441055744.0; }
    return nearbyint(x);
}
static inline double clampd(double v, double lo, double hi) { return v < lo ? lo : (v > hi ? hi : v); }

enum { F_base_sr, F_out_dur_s, F_time_unfold, F_peak, F_sat_drive, F_stereo_on, F_stereo_width, F_mode, F_micro_ms, F_seed,
       F_dust_density, F_noise_tilt, F_ring_hz, F_ring_decay_ms, F_multiband, F_partial_stretch, F_nl_warp_on, F_nl_warp_power,
       F_mb_b1, F_mb_b2, F_mb_b3, F_mb_u1, F_mb_u2, F_mb_u3, F_mb_roll, F_bandlimit_on, F_bandlimit_out_hz, F_bandlimit_roll_hz,
       F_event_process, F_grains_per_sec, F_max_grains, F_grain_amp_rand, F_grain_offset_on, F_grain_offset_max_ms,
       F_lane_density, F_lane_unfold, F_lane_cutoff, F_lane_stretch, F_er_cloud_on, F_er_taps, F_er_max_ms, F_space_ir_on, F_ir_id,
       F_ir_r_id, F_env_a, F_env_d, F_env_s, F_env_r, F_env_curve, F_bessel_id, F_export_sr, F_COUNT };
enum { MODE_GAUSS = 0, MODE_DUST = 1, MODE_NOISE = 2, MODE_SKEW = 3, MODE_RES = 4, MODE_PLAIN = 5 };

struct Lanes { const int64_t* ptr; const double* t; const double* v; };
static double eval_lane(const Lanes& L, int id, double t, double dflt) {          // eval_breakpoints, main_v2.py:469-482
    if (id < 0) return dflt;
    const int64_t a = L.ptr[id], b = L.ptr[id + 1];
    if (b <= a) return dflt;
    if (t <= L.t[a]) return L.v[a];
    if (t >= L.t[b - 1]) return L.v[b - 1];
    for (int64_t i = a; i + 1 < b; ++i) {
        const double t0 = L.t[i], v0 = L.v[i], t1 = L.t[i + 1], v1 = L.v[i + 1];
        if (t0 <= t && t <= t1) {
            const double den = t1 - t0, w = (t - t0) / (den > 1e-12 ? den : 1e-12);
            return (1 - w) * v0 + w * v1;
        }
    }
    return dflt;
}
static long long design_rate(long long base_sr, double unfold) {                   // main_v2.py:596-597, 645-646
    long long r = (long long)py_round((double)base_sr * unfold);
    if (r < base_sr) r = base_sr;
    if (r > 30000000ll) r = 30000000ll;
    return r;
}
static void zero_edge(ms_band_edge& e) { memset(&e, 0, sizeof e); }
static void lowpass_edge(ms_band_edge& e, double sr, double cutoff, double roll) {  // main_v2.py:43-58
    zero_edge(e);
    const double nyq = 0.5 * sr;
    const double fc = std::min(std::max(cutoff, 1.0), nyq);
    const double width = std::max(0.0, roll);
    if (width <= 0) { e.hi_mode = 1; e.hi_f0 = fc; e.hi_f1 = fc; }
    else { e.hi_mode = 2; e.hi_f0 = fc; e.hi_f1 = std::min(nyq, fc + width); }
}
static void bandpass_edge(ms_band_edge& e, double sr, double lo, double hi, double roll) {   // main_v2.py:64-100
    zero_edge(e);
    lo = std::max(0.0, lo);
    hi = std::max(lo, hi);
    const double nyq = 0.5 * sr;
    hi = std::min(hi, nyq);
    if (hi <= 0) { e.zero = 1; return; }
    const double width = std::max(0.0, roll);
    if (lo > 0) {
        if (width <= 0) { e.lo_mode = 1; e.lo_f0 = lo; e.lo_f1 = lo; }
        else { e.lo_mode = 2; e.lo_f0 = std::max(0.0, lo - width); e.lo_f1 = lo; }
    }
    if (hi < nyq) {
        if (width <= 0) { e.hi_mode = 1; e.hi_f0 = hi; e.hi_f1 = hi; }
        else { e.hi_mode = 2; e.hi_f0 = hi; e.hi_f1 = std::min(nyq, hi + width); }
    }
}

struct Item { int64_t n, src, dst; ms_spec_op op; };         // tables.SPEC_ITEM: exported as it is
static_assert(sizeof(Item) == 3 * sizeof(int64_t) + sizeof(ms_spec_op), "Item must have no padding");
struct Plan {
    std::vector<ms_synth_evt> sy1, sy2;
    std::vector<ms_ola_render> ola_r, env_reps;
    std::vector<ms_ola_evt> ola_e;
    std::vector<ms_fir_render> fir;
    std::vector<ms_post_render> post;
    std::vector<int32_t> tap_off, dust_pos;
    std::vector<double> tap_delay, tap_raw, dust_val;
    std::vector<Item> tilt, grain, rot;
    std::vector<int64_t> odd;                       // rows of 4: y_at, scratch, n, dr
    std::vector<int64_t> out_at, out_n, y_at, last, srs, ir_order;
    std::vector<ms_export_render> exp;              // renders with export_sr: resampler rows ...
    std::vector<int64_t> export_of, ratios, bank_at; // ... their render indices; distinct (up, down) in order of first use
    int64_t pool_n, mono_n, frames, h_total, max_h, max_out_n, env_n, n_ir, n_bank;
    int64_t alg[7];                                 // synth, tilt_spectral, grain_spectral, overlap_add, fir_in, fir_taps, post
    std::string error; int error_render;
};
struct EnvKey { int64_t n, a, d_end, sus_end, has_rel; double inv_a, inv_d, inv_r, S, curve; std::vector<int> members; };
static bool same_env(const EnvKey& k, const EnvKey& o) {
    return k.n == o.n && k.a == o.a && k.d_end == o.d_end && k.sus_end == o.sus_end && k.has_rel == o.has_rel &&
           k.inv_a == o.inv_a && k.inv_d == o.inv_d && k.inv_r == o.inv_r && k.S == o.S && k.curve == o.curve;
}

// per-render scalars that the second (sequential) pass needs
struct Scal {
    std::vector<int64_t> mono_at, fir_of, fir_r_of, st_dl, st_dr;      // fir_r_of: the right channel's row (space_ir_stereo), or -1
    std::vector<int64_t> ex_up, ex_down;                                 // export_sr as up / down in lowest terms (0: none)
    std::vector<int> stereo_on, bessel_id;
    std::vector<double> st_theta, drive, peak;
    void resize(size_t n) {
        ex_up.assign(n, 0); ex_down.assign(n, 0);
        mono_at.resize(n); fir_of.assign(n, -1); fir_r_of.assign(n, -1); st_dl.resize(n); st_dr.resize(n); stereo_on.resize(n); bessel_id.resize(n);
        st_theta.resize(n); drive.resize(n); peak.resize(n);
    }
};
// Renders [r0, r1) planned into P with every offset RELATIVE to the start of the range (pool, mono plane, event / tap / dust /
// FIR record indices, filter pool); `fir.ir` holds the impulse response ID (-2: the unit impulse) until append_part()
// resolves it.  Ranges are independent, so a slice is planned by several threads and appended in order.
static int plan_range(Plan& P, Scal& SC, const double* rows, int r0, int r1, const Lanes& L, const int64_t* ir_len) {
    const int R = r1 - r0;
    P.pool_n = P.mono_n = P.frames = P.h_total = P.max_h = P.max_out_n = P.env_n = P.n_ir = 0;
    memset(P.alg, 0, sizeof P.alg);
    P.error_render = -1;
    P.ola_r.resize(R);
    P.out_n.resize(R); P.last.assign(3 * (size_t)R, -1); P.srs.resize(2 * (size_t)R);
    SC.resize((size_t)R);
    std::vector<int64_t>& mono_at = SC.mono_at; std::vector<int64_t>& fir_of = SC.fir_of;
    std::vector<int>& stereo_on = SC.stereo_on; std::vector<int64_t>& st_dl = SC.st_dl; std::vector<int64_t>& st_dr = SC.st_dr;
    std::vector<double>& st_theta = SC.st_theta; std::vector<double>& drive = SC.drive; std::vector<double>& peak = SC.peak;
    std::vector<int>& bessel_id = SC.bessel_id;
    std::vector<double> times;
    std::vector<uint64_t> dbits; std::vector<int32_t> dlast; std::vector<double> dvals, er_dl, er_ga;
    for (int r = 0; r < R; ++r) {
        const double* p = rows + (size_t)(r0 + r) * F_COUNT;
        const long long base_sr = (long long)p[F_base_sr];
        const double out_dur = p[F_out_dur_s];
        long long out_n = (long long)py_round(out_dur * (double)base_sr);
        if (out_n < 1) out_n = 1;
        const double base_unfold = std::max(1.0, p[F_time_unfold]);
        const long long design_sr_base = design_rate(base_sr, base_unfold);
        const double rate = p[F_grains_per_sec];
        const long long seed = (long long)p[F_seed];
        const int process = (int)p[F_event_process];
        // ---- event times (main_v2.py:507-558): Single, or Poisson gaps
        times.clear();
        if (process == 0 || rate <= 0) times.push_back(0.0);
        else {
            Pcg64 g; g.seed((uint64_t)(seed + 9999));
            double t = 0.0;
            const double scale = 1.0 / rate;
            while (t < out_dur) { t += scale * g.standard_exponential(); if (t < out_dur) times.push_back(t); }
        }
        const long long max_grains = (long long)p[F_max_grains];
        if ((long long)times.size() > max_grains) times.resize((size_t)std::max(0ll, max_grains));
        Pcg64 rng; rng.seed((uint64_t)(seed + 123456));
        const double micro_ms = p[F_micro_ms], micro_s = micro_ms / 1000.0;
        const double spread = p[F_grain_amp_rand];
        const int mode = (int)p[F_mode];
        const int offset_on = p[F_grain_offset_on] != 0.0;
        const long long max_off = offset_on ? (long long)py_round((p[F_grain_offset_max_ms] / 1000.0) * (double)base_sr) : 0;
        // ---- ADSR segment lengths (main_v2.py:173-177)
        const long long a = std::max(0ll, (long long)py_round((double)base_sr * p[F_env_a] / 1000.0));
        const long long d = std::max(0ll, (long long)py_round((double)base_sr * p[F_env_d] / 1000.0));
        const long long rel = std::max(0ll, (long long)py_round((double)base_sr * p[F_env_r] / 1000.0));
        const double S = clampd(p[F_env_s], 0.0, 1.0), curve = std::max(1e-6, p[F_env_curve]);
        const long long n_out = out_n;
        if (a > n_out) { P.error = "adsr"; P.error_render = r0 + r; return -1; }
        const long long d_end = d > 0 ? std::min(n_out, a + d) : a;
        const long long sus_end = std::max(d_end, n_out - rel);
        const int64_t ev_begin = (int64_t)P.ola_e.size();
        int64_t max_len = 0, x_begin = n_out, x_end = 0;
        for (size_t i = 0; i < times.size(); ++i) {
            const double t0 = times[i];
            const double dens = eval_lane(L, (int)p[F_lane_density], t0, rate);
            double ufac = eval_lane(L, (int)p[F_lane_unfold], t0, base_unfold);
            const double cutoff_out = eval_lane(L, (int)p[F_lane_cutoff], t0, p[F_bandlimit_out_hz]);
            const double stretch = eval_lane(L, (int)p[F_lane_stretch], t0, p[F_partial_stretch]);
            double amp = 1.0;
            if (rate > 0) amp *= std::min(std::max(dens / std::max(1e-6, rate), 0.15), 4.0);
            amp *= rng.uniform(1.0 - spread, 1.0 + spread);
            ufac = std::max(1.0, ufac);
            const long long sr_evt = design_rate(base_sr, ufac);
            long long n = (long long)py_round((double)sr_evt * micro_ms / 1000.0);
            if (n < 16) n = 16;
            const long long start = (long long)py_round(t0 * (double)base_sr);
            long long offset = 0, length = 0; int placed = 0;
            if (start < n_out) {
                if (offset_on && max_off > 0) offset = (long long)rng.integers((uint64_t)std::max(1ll, std::min(max_off, n)));
                length = std::max(0ll, std::min(n_out - start, n - offset));
                placed = length > 0;
            }
            const double cutoff_gen = cutoff_out * ufac;
            // ---- grain operator (plan.grain_spec_op)
            ms_spec_op op; memset(&op, 0, sizeof op);
            op.kind = MS_OP_GRAIN;
            op.df = 1.0 / ((double)n * (1.0 / (double)sr_evt));
            op.factor = 1.0;
            if (p[F_bandlimit_on] != 0.0 && n >= 8) { op.lp_on = 1; lowpass_edge(op.lp, (double)sr_evt, cutoff_gen, p[F_bandlimit_roll_hz]); }
            if (p[F_nl_warp_on] != 0.0 && n >= 16) op.warp_exp = 1.0 / std::max(1e-6, p[F_nl_warp_power]);
            if (n >= 16 && !(fabs(stretch - 1.0) < 1e-9)) { op.stretch_on = 1; op.factor = stretch; }
            if (p[F_multiband] != 0.0 && n >= 8) {
                const double b1 = p[F_mb_b1], b2 = p[F_mb_b2], b3 = p[F_mb_b3], roll = p[F_mb_roll];
                const double lo[3] = {0.0, b1, b2}, hi[3] = {b1, b2, b3}, us[3] = {p[F_mb_u1], p[F_mb_u2], p[F_mb_u3]};
                op.n_bands = 3;
                for (int b = 0; b < 3; ++b) bandpass_edge(op.mb[b], (double)sr_evt, lo[b] * us[b], hi[b] * us[b], roll);
            }
            const int has_spec = op.lp_on || op.stretch_on || op.n_bands || op.warp_exp != 0.0;
            // ---- generator constants
            long long fade = std::max(8ll, (long long)(0.01 * (double)n)), sigma = 1, ker_len = 8;
            double f_over_sr = 0.0, ring_decay = 0.0, env_decay = 0.0;
            int64_t dust_b = 0, dust_c = 0;
            const int64_t e = (int64_t)P.sy1.size();
            const int64_t micro = P.pool_n;
            P.pool_n += n;
            P.alg[0] += n;
            int64_t out1 = micro, aux2 = 0; int mode2 = -1;
            if (mode == MODE_GAUSS) sigma = std::max(1ll, (long long)(0.0025 * (double)n));
            else if (mode == MODE_DUST) {
                // main_v2.py:240-244: indices and values from the event's stream; duplicates: last write wins
                Pcg64 g; g.seed((uint64_t)(seed + (long long)i));
                long long k = (long long)py_round(p[F_dust_density] * (double)n);
                if (k < 1) k = 1;
                // a bitmap of the positions hit + the last draw that hit each: ascending unique positions fall out of a scan
                const size_t words = (size_t)((n + 63) / 64);
                dbits.assign(words, 0ull);
                if (dlast.size() < (size_t)n) dlast.resize((size_t)n);
                for (long long j = 0; j < k; ++j) {
                    const uint64_t pos = g.integers((uint64_t)n);
                    dbits[pos >> 6] |= 1ull << (pos & 63);
                    dlast[pos] = (int32_t)j;
                }
                dvals.resize((size_t)k);
                for (long long j = 0; j < k; ++j) dvals[(size_t)j] = g.uniform(-1.0, 1.0);
                dust_b = (int64_t)P.dust_pos.size();
                for (size_t w = 0; w < words; ++w) {
                    uint64_t m = dbits[w];
                    while (m) {
                        const int b = __builtin_ctzll(m);
                        m &= m - 1;
                        const size_t pos = w * 64 + (size_t)b;
                        P.dust_pos.push_back((int32_t)pos);
                        P.dust_val.push_back(dvals[(size_t)dlast[pos]]);
                    }
                }
                dust_c = (int64_t)P.dust_pos.size() - dust_b;
                ker_len = std::max(8ll, (long long)(0.01 * (double)n));
            } else if (mode == MODE_NOISE || mode == MODE_SKEW) {
                const double T = std::max(1e-6, micro_s * (mode == MODE_NOISE ? 0.25 : 0.2));
                env_decay = 1.0 / (T * (double)sr_evt);
                const int64_t raw = P.pool_n, tilted = P.pool_n + n;
                P.pool_n += 2 * n;
                out1 = raw; mode2 = mode; aux2 = tilted;
                Item it; it.n = n; it.src = raw; it.dst = tilted; memset(&it.op, 0, sizeof it.op);
                it.op.kind = MS_OP_TILT;
                it.op.df = 1.0 / ((double)n * (1.0 / (double)sr_evt));
                it.op.alpha = log(pow(10.0, p[F_noise_tilt] / 20.0)) / log(2.0);      // math.log(10 ** (tilt / 20), 2.0)
                P.tilt.push_back(it);
                P.alg[1] += 2 * n;
            } else if (mode == MODE_RES) {
                f_over_sr = std::max(10.0, p[F_ring_hz]) / (double)sr_evt;
                ring_decay = 1.0 / (std::max(1e-6, p[F_ring_decay_ms] / 1000.0) * (double)sr_evt);
                env_decay = 1.0 / (std::max(1e-6, micro_s * 0.15) * (double)sr_evt);
            }
            Pcg64 evs; evs.seed((uint64_t)(seed + (long long)i));
            ms_synth_evt s1; memset(&s1, 0, sizeof s1);
            s1.s_hi = (uint64_t)(evs.state >> 64); s1.s_lo = (uint64_t)evs.state; s1.i_hi = (uint64_t)(evs.inc >> 64); s1.i_lo = (uint64_t)evs.inc;
            s1.n = (int32_t)n; s1.mode = mode; s1.fade = (int32_t)fade; s1.sigma = (int32_t)sigma; s1.out = out1;
            s1.f_over_sr = f_over_sr; s1.inv_fade = fade > 0 ? 1.0 / (double)fade : 0.0; s1.ring_decay = ring_decay; s1.env_decay = env_decay;
            s1.dust_begin = dust_b; s1.dust_count = (int32_t)dust_c; s1.ker_len = (int32_t)ker_len; s1.aux = 0;
            ms_synth_evt s2 = s1;
            s2.mode = mode2; s2.out = micro; s2.dust_begin = 0; s2.dust_count = 0; s2.aux = aux2;
            P.sy1.push_back(s1); P.sy2.push_back(s2);
            (void)e;
            int64_t g_at = micro;
            if (has_spec) {
                g_at = P.pool_n; P.pool_n += n;
                Item it; it.n = n; it.src = micro; it.dst = g_at; it.op = op;
                P.grain.push_back(it);
                P.alg[2] += 2 * n * ((op.lp_on ? 1 : 0) + (op.stretch_on ? 1 : 0) + (op.n_bands ? 1 : 0) + (op.warp_exp != 0.0 ? 1 : 0));
            }
            P.last[3 * (size_t)r + 0] = micro; P.last[3 * (size_t)r + 1] = g_at; P.last[3 * (size_t)r + 2] = n;
            if (placed) {
                ms_ola_evt oe; oe.grain = g_at + offset; oe.start = (int32_t)start; oe.len = (int32_t)length; oe.amp = amp;
                P.ola_e.push_back(oe);
                max_len = std::max<int64_t>(max_len, length);
                x_begin = std::min<int64_t>(x_begin, start);
                x_end = std::max<int64_t>(x_end, start + length);
                P.alg[3] += length;
            }
        }
        // ---- envelope description (tables.pack_chunk); sharing is decided over the whole slice (finish_plan)
        const int64_t has_rel = (rel > 0 && n_out > sus_end) ? 1 : 0;
        const double inv_a = a > 0 ? 1.0 / (double)a : 0.0, inv_d = d_end > a ? 1.0 / (double)(d_end - a) : 0.0;
        const double inv_r = n_out - sus_end > 1 ? 1.0 / (double)(n_out - sus_end - 1) : 0.0;
        ms_ola_render& orr = P.ola_r[r];
        memset(&orr, 0, sizeof orr);
        orr.out = P.mono_n; orr.out_n = (int32_t)n_out; orr.ev_begin = (int32_t)ev_begin; orr.ev_end = (int32_t)P.ola_e.size(); orr.max_len = (int32_t)max_len;
        orr.A = (int32_t)a; orr.D_end = (int32_t)d_end; orr.sus_end = (int32_t)sus_end; orr.has_release = (int32_t)has_rel;
        orr.inv_A = inv_a; orr.inv_D = inv_d; orr.inv_R = inv_r; orr.S = S; orr.curve = curve; orr.env = -1;
        P.alg[3] += n_out;
        // ---- reflection cloud (main_v2.py:410-417) + impulse response -> one FIR
        int64_t t_begin = (int64_t)P.tap_off.size(), max_tap = 0; int has_er = 0;
        if (p[F_er_cloud_on] != 0.0) {
            long long taps = (long long)p[F_er_taps];
            if (taps < 1) taps = 1;
            const double max_ms = p[F_er_max_ms];
            Pcg64 g; g.seed((uint64_t)(seed + 202));
            std::vector<double>& dl = er_dl; std::vector<double>& ga = er_ga;
            dl.resize((size_t)taps); ga.resize((size_t)taps);
            for (long long j = 0; j < taps; ++j) dl[(size_t)j] = g.uniform(0.3, max_ms) / 1000.0;
            for (long long j = 0; j < taps; ++j) ga[(size_t)j] = g.uniform(-1.0, 1.0);
            int64_t kept = 0;
            for (long long j = 0; j < taps; ++j) {
                const long long off = (long long)py_round(dl[(size_t)j] * (double)base_sr);
                if (off > 0 && off < n_out) {
                    P.tap_off.push_back((int32_t)off); P.tap_delay.push_back(dl[(size_t)j]); P.tap_raw.push_back(ga[(size_t)j]);
                    max_tap = std::max<int64_t>(max_tap, off); ++kept;
                }
            }
            has_er = kept > 0;
            if (kept > 4096) { P.error = "er_taps"; P.error_render = r0 + r; return -1; }
        }
        const int ir_id = p[F_space_ir_on] != 0.0 ? (int)p[F_ir_id] : -1;
        if (has_er || ir_id >= 0) {
            int64_t ir_at, irl;
            if (ir_id >= 0) {
                ir_at = ir_id; irl = ir_len[ir_id];
                P.alg[4] += 2 * n_out; P.alg[5] += irl;
            } else {
                ir_at = -2; irl = 1;
            }
            int64_t h_len = irl;
            if (has_er) { h_len = irl + max_tap; P.alg[4] += 2 * n_out; }
            if (x_begin == 0 && a > 0) x_begin = 1;           // env[0] = 0 ** curve = 0 (main_v2.py:181-182)
            ms_fir_render fr; memset(&fr, 0, sizeof fr);
            fr.ir = ir_at; fr.ir_len = (int32_t)irl; fr.h_len = (int32_t)h_len; fr.h = P.h_total; fr.tap_begin = (int32_t)t_begin;
            fr.tap_end = (int32_t)P.tap_off.size(); fr.x = P.mono_n; fr.y = 0; fr.out_n = (int32_t)n_out;
            fr.x_begin = (int32_t)std::min(x_begin, x_end); fr.x_end = (int32_t)x_end;
            fir_of[r] = (int64_t)P.fir.size();
            P.fir.push_back(fr);
            const int ir_r_id = ir_id >= 0 ? (int)p[F_ir_r_id] : -1;
            if (ir_r_id >= 0) {                               // space_ir_stereo: the right channel's row differs only in ir and y
                P.alg[4] += has_er ? 4 * n_out : 2 * n_out; P.alg[5] += ir_len[ir_r_id];
                fr.ir = ir_r_id;
                SC.fir_r_of[r] = (int64_t)P.fir.size();
                P.fir.push_back(fr);
            }
            P.h_total += h_len; P.max_h = std::max(P.max_h, h_len);
        }
        mono_at[r] = P.mono_n;
        P.mono_n += n_out;
        P.max_out_n = std::max<int64_t>(P.max_out_n, n_out);
        P.srs[2 * (size_t)r] = base_sr; P.srs[2 * (size_t)r + 1] = design_sr_base;
        // ---- stereo / clip scalars (main_v2.py:424-429, 780-781)
        stereo_on[r] = 0;
        if (p[F_stereo_on] != 0.0 && n_out >= 64) {
            const double w = clampd(p[F_stereo_width], 0.0, 1.0);
            stereo_on[r] = 1;
            st_dl[r] = (long long)py_round((1 + 7 * w) * 0.0005 * (double)base_sr);
            st_dr[r] = (long long)py_round((1 + 9 * w) * 0.0007 * (double)base_sr);
            st_theta[r] = w * 0.9;
        }
        drive[r] = p[F_sat_drive]; peak[r] = p[F_peak]; bessel_id[r] = (int)p[F_bessel_id];
        const long long ex_sr = (long long)p[F_export_sr];          // validated by plan.export_ratio; 0: none
        if (ex_sr > 0) { const long long g = std::gcd(base_sr, ex_sr); SC.ex_up[r] = ex_sr / g; SC.ex_down[r] = base_sr / g; }
        P.out_n[r] = n_out;
    }
    return 0;
}

template <class T> static void append(std::vector<T>& d, const std::vector<T>& s) { d.insert(d.end(), s.begin(), s.end()); }

// Appends the range plan `Q` (relative offsets) to the slice plan `P`; returns the number of renders appended.
static void append_part(Plan& P, Scal& S, const Plan& Q, const Scal& QS, std::vector<int64_t>& ir_at_of, int64_t& delta_at, const int64_t* ir_len) {
    const int64_t pool_b = P.pool_n, mono_b = P.mono_n, ev_b = (int64_t)P.ola_e.size(), fir_b = (int64_t)P.fir.size();
    const int64_t tap_b = (int64_t)P.tap_off.size(), dust_b = (int64_t)P.dust_pos.size(), h_b = P.h_total;
    const size_t R = Q.ola_r.size();
    for (size_t i = 0; i < Q.sy1.size(); ++i) {
        ms_synth_evt s1 = Q.sy1[i], s2 = Q.sy2[i];
        s1.out += pool_b; s2.out += pool_b;
        if (s1.mode == MODE_DUST) s1.dust_begin += dust_b;
        if (s2.mode != -1) s2.aux += pool_b;
        P.sy1.push_back(s1); P.sy2.push_back(s2);
    }
    for (ms_ola_evt e : Q.ola_e) { e.grain += pool_b; P.ola_e.push_back(e); }
    for (ms_ola_render o : Q.ola_r) { o.out += mono_b; o.ev_begin += (int32_t)ev_b; o.ev_end += (int32_t)ev_b; P.ola_r.push_back(o); }
    for (ms_fir_render f : Q.fir) {
        // impulse responses in order of first use; the unit impulse (reflections without an IR) is one more entry
        const int64_t id = f.ir;
        if (id >= 0) {
            size_t k = 0;
            for (; k < P.ir_order.size(); ++k) if (P.ir_order[k] == id) break;
            if (k == P.ir_order.size()) { P.ir_order.push_back(id); ir_at_of.push_back(P.n_ir); P.n_ir += ir_len[id]; }
            f.ir = ir_at_of[k];
        } else {
            if (delta_at < 0) { delta_at = P.n_ir; P.ir_order.push_back(-2); ir_at_of.push_back(P.n_ir); P.n_ir += 1; }
            f.ir = delta_at;
        }
        f.h += h_b; f.tap_begin += (int32_t)tap_b; f.tap_end += (int32_t)tap_b; f.x += mono_b;
        P.fir.push_back(f);
    }
    append(P.tap_off, Q.tap_off); append(P.tap_delay, Q.tap_delay); append(P.tap_raw, Q.tap_raw);
    append(P.dust_pos, Q.dust_pos); append(P.dust_val, Q.dust_val);
    for (Item it : Q.tilt) { it.src += pool_b; it.dst += pool_b; P.tilt.push_back(it); }
    for (Item it : Q.grain) { it.src += pool_b; it.dst += pool_b; P.grain.push_back(it); }
    for (size_t r = 0; r < R; ++r) {
        for (int k = 0; k < 2; ++k) { const int64_t v = Q.last[3 * r + k]; P.last.push_back(v < 0 ? v : v + pool_b); }
        P.last.push_back(Q.last[3 * r + 2]);
        S.mono_at.push_back(QS.mono_at[r] + mono_b);
        S.fir_of.push_back(QS.fir_of[r] < 0 ? -1 : QS.fir_of[r] + fir_b);
        S.fir_r_of.push_back(QS.fir_r_of[r] < 0 ? -1 : QS.fir_r_of[r] + fir_b);
    }
    append(P.out_n, Q.out_n); append(P.srs, Q.srs);
    append(S.stereo_on, QS.stereo_on); append(S.st_dl, QS.st_dl); append(S.st_dr, QS.st_dr); append(S.st_theta, QS.st_theta);
    append(S.drive, QS.drive); append(S.peak, QS.peak); append(S.bessel_id, QS.bessel_id);
    append(S.ex_up, QS.ex_up); append(S.ex_down, QS.ex_down);
    P.pool_n += Q.pool_n; P.mono_n += Q.mono_n; P.h_total += Q.h_total;
    P.max_h = std::max(P.max_h, Q.max_h); P.max_out_n = std::max(P.max_out_n, Q.max_out_n);
    for (int k = 0; k < 7; ++k) P.alg[k] += Q.alg[k];
}

// Output planes, post records, shared envelopes: the part of the plan that looks at the slice as a whole.
static void finish_plan(Plan& P, const Scal& S, const double* bessel, int n_coef) {
    const int R = (int)P.ola_r.size();
    P.post.resize(R); P.out_at.resize(R); P.y_at.resize(R);
    const std::vector<int64_t>& mono_at = S.mono_at; const std::vector<int64_t>& fir_of = S.fir_of;
    const std::vector<int>& stereo_on = S.stereo_on; const std::vector<int64_t>& st_dl = S.st_dl; const std::vector<int64_t>& st_dr = S.st_dr;
    const std::vector<double>& st_theta = S.st_theta; const std::vector<double>& drive = S.drive; const std::vector<double>& peak = S.peak;
    const std::vector<int>& bessel_id = S.bessel_id;
    // ---- second pass: output planes, post records
    const int64_t plane = P.mono_n;
    int64_t extra = 0;
    for (int r = 0; r < R; ++r) {
        const int64_t n = P.out_n[r];
        int64_t y = mono_at[r];
        if (fir_of[r] >= 0) { y = plane + mono_at[r]; P.fir[(size_t)fir_of[r]].y = y; }
        ms_post_render& po = P.post[r];
        memset(&po, 0, sizeof po);
        int mode = 0; int64_t dl = 0, dr = 0, rbuf = 0;
        if (S.fir_r_of[r] >= 0) {
            // space_ir_stereo: [yR | right] (even n), [yR | rolled copy | right] (odd n), [yR] (no stereo diffusion)
            const int64_t y_r = 2 * plane + extra;
            P.fir[(size_t)S.fir_r_of[r]].y = y_r;
            extra += n;
            if (!stereo_on[r]) {
                mode = 2; rbuf = y_r;
            } else if (n % 2 == 0) {
                mode = 3; rbuf = y_r + n; dl = st_dl[r]; dr = st_dr[r];
                const double* cf = bessel + (size_t)bessel_id[r] * n_coef;
                for (int k = 0; k < n_coef && k < 2 * MS_POST_K + 1; ++k) po.coef[k] = cf[k];
                extra += n;
            } else {
                mode = 2; rbuf = y_r + 2 * n; dl = st_dl[r]; dr = st_dr[r];
                P.odd.push_back(y_r); P.odd.push_back(y_r + n); P.odd.push_back(n); P.odd.push_back(dr);
                Item it; it.n = n; it.src = y_r + n; it.dst = y_r + 2 * n; memset(&it.op, 0, sizeof it.op);
                it.op.kind = MS_OP_ROT; it.op.alpha = st_theta[r];
                P.rot.push_back(it);
                extra += 2 * n;
            }
        } else if (stereo_on[r]) {
            dl = st_dl[r]; dr = st_dr[r];
            if (n % 2 == 0) {
                mode = 1; rbuf = 2 * plane + extra;
                const double* cf = bessel + (size_t)bessel_id[r] * n_coef;
                for (int k = 0; k < n_coef && k < 2 * MS_POST_K + 1; ++k) po.coef[k] = cf[k];
                extra += n;
            } else {
                mode = 2; rbuf = 2 * plane + extra + n;
                P.odd.push_back(y); P.odd.push_back(2 * plane + extra); P.odd.push_back(n); P.odd.push_back(dr);
                Item it; it.n = n; it.src = 2 * plane + extra; it.dst = 2 * plane + extra + n; memset(&it.op, 0, sizeof it.op);
                it.op.kind = MS_OP_ROT; it.op.alpha = st_theta[r];
                P.rot.push_back(it);
                extra += 2 * n;
            }
        }
        po.y = y; po.out = P.frames; po.rbuf = rbuf; po.n = (int32_t)n; po.stereo_mode = mode; po.dl = (int32_t)dl; po.dr = (int32_t)dr;
        po.drive = drive[r]; po.inv_tanh_drive = drive[r] > 0 ? 1.0 / tanh(drive[r]) : 1.0; po.peak = peak[r];
        // export_sr: ceil(n up / down) frames through the polyphase bank of the ratio (decimate.polyphase_bank fills the pool)
        int64_t n_x = n;
        if (S.ex_up[r] > 0) {
            const int64_t up = S.ex_up[r], down = S.ex_down[r], half = 10 * std::max(up, down);
            const int64_t taps = half / up + (up - 1 + half) / up + 1;
            n_x = (n * up + down - 1) / down;
            size_t k = 0;
            for (; k < P.bank_at.size(); ++k) if (P.ratios[2 * k] == up && P.ratios[2 * k + 1] == down) break;
            if (k == P.bank_at.size()) { P.ratios.push_back(up); P.ratios.push_back(down); P.bank_at.push_back(P.n_bank); P.n_bank += up * taps; }
            ms_export_render e;
            e.out = P.frames; e.out_end = P.frames + n_x; e.bank = P.bank_at[k]; e.bank_end = P.bank_at[k] + up * taps;
            e.rate[0] = (int32_t)up; e.rate[1] = (int32_t)down; e.rate[2] = (int32_t)half; e.rate[3] = (int32_t)taps;
            P.exp.push_back(e); P.export_of.push_back(r);
        }
        P.out_at[r] = P.frames; P.y_at[r] = y;
        P.frames += n_x;
        P.out_n[r] = n_x;
        P.alg[6] += n;
    }
    // ---- envelopes shared by several renders are tabulated once
    std::vector<EnvKey> envs;
    for (int r = 0; r < R; ++r) {
        const ms_ola_render& o = P.ola_r[(size_t)r];
        EnvKey key; key.n = o.out_n; key.a = o.A; key.d_end = o.D_end; key.sus_end = o.sus_end; key.has_rel = o.has_release;
        key.inv_a = o.inv_A; key.inv_d = o.inv_D; key.inv_r = o.inv_R; key.S = o.S; key.curve = o.curve;
        size_t k = 0;
        for (; k < envs.size(); ++k) if (same_env(envs[k], key)) break;
        if (k == envs.size()) envs.push_back(key);
        envs[k].members.push_back(r);
    }
    for (size_t k = 0; k < envs.size(); ++k) {
        if (envs[k].members.size() < 2) continue;
        for (int m : envs[k].members) P.ola_r[(size_t)m].env = P.env_n;
        P.env_reps.push_back(P.ola_r[(size_t)envs[k].members[0]]);
        P.env_n += envs[k].n;
    }
    P.mono_n = 2 * plane + extra;
}

// A slice in blocks of HP_BLOCK renders, the blocks handed out to `threads` threads and appended in order.
static const int HP_BLOCK = 32;
static int plan_chunk(Plan& P, const double* rows, int R, const Lanes& L, const int64_t* ir_len, const double* bessel, int n_coef, int threads) {
    P.pool_n = P.mono_n = P.frames = P.h_total = P.max_h = P.max_out_n = P.env_n = P.n_ir = P.n_bank = 0;
    memset(P.alg, 0, sizeof P.alg);
    const int nb = (R + HP_BLOCK - 1) / HP_BLOCK;
    std::vector<Plan> parts((size_t)nb); std::vector<Scal> scal((size_t)nb);
    std::atomic<int> next(0);
    auto work = [&]() {
        for (;;) {
            const int b = next.fetch_add(1);
            if (b >= nb) return;
            plan_range(parts[(size_t)b], scal[(size_t)b], rows, b * HP_BLOCK, std::min(R, (b + 1) * HP_BLOCK), L, ir_len);
        }
    };
    const int T = std::max(1, std::min(threads, nb));
    std::vector<std::thread> pool;
    for (int t = 1; t < T; ++t) pool.emplace_back(work);
    work();
    for (std::thread& t : pool) t.join();
    Scal S; std::vector<int64_t> ir_at_of; int64_t delta_at = -1;
    for (int b = 0; b < nb; ++b) {
        if (parts[(size_t)b].error_render >= 0) { P.error = parts[(size_t)b].error; P.error_render = parts[(size_t)b].error_render; return -1; }
        append_part(P, S, parts[(size_t)b], scal[(size_t)b], ir_at_of, delta_at, ir_len);
    }
    finish_plan(P, S, bessel, n_coef);
    return 0;
}

}  // namespace

extern "C" {
int ms_hp_field_count(void) { return F_COUNT; }
// numpy's PCG64(seed).state right after seeding, for tests and for the Python planner: out[4 i ..] = s_hi, s_lo, i_hi, i_lo
void ms_hp_pcg64_seed(const int64_t* seeds, int n, uint64_t* out) {
    for (int i = 0; i < n; ++i) {
        Pcg64 g; g.seed((uint64_t)seeds[i]);
        out[4 * i] = (uint64_t)(g.state >> 64); out[4 * i + 1] = (uint64_t)g.state; out[4 * i + 2] = (uint64_t)(g.inc >> 64); out[4 * i + 3] = (uint64_t)g.inc;
    }
}
// test hooks: the first `n` draws of default_rng(seed) of one kind (0 random, 1 integers(0, high), 2 exponential(1.0), 3 raw 64-bit)
void ms_hp_draws(int64_t seed, int kind, uint64_t high, int n, double* out) {
    Pcg64 g; g.seed((uint64_t)seed);
    for (int i = 0; i < n; ++i) {
        if (kind == 0) out[i] = g.next_double();
        else if (kind == 1) out[i] = (double)g.integers(high);
        else if (kind == 2) out[i] = g.standard_exponential();
        else { const uint64_t w = g.next64(); memcpy(&out[i], &w, 8); }
    }
}
void* ms_hp_plan(const double* rows, int n_renders, const int64_t* lane_ptr, const double* lane_t, const double* lane_v,
                 const int64_t* ir_len, const double* bessel, int n_coef, int threads) {
    Plan* P = new Plan();
    P->error_render = -1;
    Lanes L; L.ptr = lane_ptr; L.t = lane_t; L.v = lane_v;
    plan_chunk(*P, rows, n_renders, L, ir_len, bessel, n_coef, threads);
    return P;
}
const char* ms_hp_error(void* h, int* render) { Plan* P = (Plan*)h; *render = P->error_render; return P->error.c_str(); }
// sizes: element counts of every exported array, in the order of ms_hp_export
enum { HP_SY, HP_OLA_R, HP_ENV_REPS, HP_OLA_E, HP_FIR, HP_POST, HP_TAPS, HP_DUST, HP_TILT, HP_GRAIN, HP_ROT, HP_ODD, HP_IRS, HP_EXPORT,
       HP_RATIOS, HP_NSIZES };
void ms_hp_sizes(void* h, int64_t* sizes, int64_t* scalars /*pool_n mono_n frames h_total max_h max_out_n env_n, alg[7]*/) {
    Plan* P = (Plan*)h;
    sizes[HP_SY] = (int64_t)P->sy1.size(); sizes[HP_OLA_R] = (int64_t)P->ola_r.size(); sizes[HP_ENV_REPS] = (int64_t)P->env_reps.size();
    sizes[HP_OLA_E] = (int64_t)P->ola_e.size(); sizes[HP_FIR] = (int64_t)P->fir.size(); sizes[HP_POST] = (int64_t)P->post.size();
    sizes[HP_TAPS] = (int64_t)P->tap_off.size(); sizes[HP_DUST] = (int64_t)P->dust_pos.size(); sizes[HP_TILT] = (int64_t)P->tilt.size();
    sizes[HP_GRAIN] = (int64_t)P->grain.size(); sizes[HP_ROT] = (int64_t)P->rot.size(); sizes[HP_ODD] = (int64_t)P->odd.size() / 4;
    sizes[HP_IRS] = (int64_t)P->ir_order.size(); sizes[HP_EXPORT] = (int64_t)P->exp.size(); sizes[HP_RATIOS] = (int64_t)P->bank_at.size();
    scalars[0] = P->pool_n; scalars[1] = P->mono_n; scalars[2] = P->frames; scalars[3] = P->h_total; scalars[4] = P->max_h;
    scalars[5] = P->max_out_n; scalars[6] = P->env_n;
    for (int i = 0; i < 7; ++i) scalars[7 + i] = P->alg[i];
}
void ms_hp_export(void* h, void* sy1, void* sy2, void* ola_r, void* env_reps, void* ola_e, void* fir, void* post,
                  int32_t* tap_off, double* tap_delay, double* tap_raw, int32_t* dust_pos, double* dust_val,
                  void* tilt, void* grain, void* rot,
                  int64_t* odd, int64_t* ir_order, int64_t* out_at, int64_t* out_n, int64_t* y_at, int64_t* last, int64_t* srs,
                  void* exp, int64_t* export_of, int64_t* ratios) {
    Plan* P = (Plan*)h;
    auto cp = [](void* d, const void* s, size_t b) { if (b) memcpy(d, s, b); };
    cp(sy1, P->sy1.data(), P->sy1.size() * sizeof(ms_synth_evt)); cp(sy2, P->sy2.data(), P->sy2.size() * sizeof(ms_synth_evt));
    cp(ola_r, P->ola_r.data(), P->ola_r.size() * sizeof(ms_ola_render)); cp(env_reps, P->env_reps.data(), P->env_reps.size() * sizeof(ms_ola_render));
    cp(ola_e, P->ola_e.data(), P->ola_e.size() * sizeof(ms_ola_evt)); cp(fir, P->fir.data(), P->fir.size() * sizeof(ms_fir_render));
    cp(post, P->post.data(), P->post.size() * sizeof(ms_post_render));
    cp(tap_off, P->tap_off.data(), P->tap_off.size() * 4); cp(tap_delay, P->tap_delay.data(), P->tap_delay.size() * 8); cp(tap_raw, P->tap_raw.data(), P->tap_raw.size() * 8);
    cp(dust_pos, P->dust_pos.data(), P->dust_pos.size() * 4); cp(dust_val, P->dust_val.data(), P->dust_val.size() * 8);
    cp(tilt, P->tilt.data(), P->tilt.size() * sizeof(Item)); cp(grain, P->grain.data(), P->grain.size() * sizeof(Item));
    cp(rot, P->rot.data(), P->rot.size() * sizeof(Item));
    cp(odd, P->odd.data(), P->odd.size() * 8); cp(ir_order, P->ir_order.data(), P->ir_order.size() * 8);
    cp(out_at, P->out_at.data(), P->out_at.size() * 8); cp(out_n, P->out_n.data(), P->out_n.size() * 8); cp(y_at, P->y_at.data(), P->y_at.size() * 8);
    cp(last, P->last.data(), P->last.size() * 8); cp(srs, P->srs.data(), P->srs.size() * 8);
    cp(exp, P->exp.data(), P->exp.size() * sizeof(ms_export_render)); cp(export_of, P->export_of.data(), P->export_of.size() * 8);
    cp(ratios, P->ratios.data(), P->ratios.size() * 8);
}
void ms_hp_free(void* h) { delete (Plan*)h; }
}
