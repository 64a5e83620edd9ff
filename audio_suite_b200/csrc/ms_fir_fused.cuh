// ms_fir_fused.cuh -- the FIR stage (early_reflection_cloud + convolve_ir_short, main_v2.py:409-421, 438-445) for
// 65536-point overlap-save blocks, as three phases over ONE 65536-point complex scratch block per unit:
//
//   P1  columns:  x (two real blocks as re / im) -> 256-point FFTs over n1 -> twiddle W^(k1 n2)        -> S[n2][k1]
//   P2  rows:     S[.][k1] -> FFT over n2 -> * H[k1][k2] -> swap -> FFT -> twiddle W^(k1 n2') -> back to S[n2'][k1]
//                 with H[k1][k2] = IRspec[k1][k2] * (1 + E[k1 + 256 k2]) composed IN the tile: the reflection taps are
//                 folded modulo 256 with the modulation W^(off k1) and one more 256-point FFT gives row k1 of E
//   P3  columns:  S[n2][.] -> FFT over k1 -> valid outputs of both blocks (exact zeros outside the live range)
//
// Every 256-point FFT is WARP-LOCAL: a lane holds x[lane + 32 q] (q < 8) in registers, radix 8 . 8 . 4, two
// exchanges through the warp's own shared-memory row with __syncwarp only; the first pass reads its input and the
// last pass leaves its output in registers in the SAME layout (index lane + 32 m), so two transforms chain without
// touching shared memory and global loads / stores on the contiguous side go straight from / to registers
// (512 contiguous bytes per warp instruction).  The strided side of each phase goes through a transposing tile in
// shared memory (8 vectors x 256) so that global accesses are 64- / 128-byte segments.
//
// Each phase is its own launch, grid = (tiles, units): CTA (t, u) does tile t of unit u, and unit u owns scratch block
// u.  The launch boundary is the barrier between phases.  The CPU block emulator runs the same launches.

#ifdef MS_HOST_EMUL
#define MS_LDCG(p) (*(p))
#else
#define MS_LDCG(p) __ldcg(p)
#endif

#define FF_N 256                       // both factors of the 65536-point block
#define FF_TILE 8                      // vectors (columns or rows) per tile = warps per CTA
#define FF_NTHR (32 * FF_TILE)
#define FF_TILES (FF_N / FF_TILE)      // tiles per phase
#define FF_RS ((ms_pad(FF_N) + 1) | 1) // row stride of a tile in shared memory (odd: conflict-free transposes)
#define FF_RES_STRIDE (257 + 256)       // ints per render in the residue table

struct FirUnit {
    const real* in; real* out;        // the render's mono input / output planes
    const cpx* filt;                  // IR spectrum / B in [k1][k2] layout
    long long p0_a, p0_b;             // first input sample of block a / b (may be negative)
    int has_b, ols_n, ols_skip;       // ols_skip = taps - 1: leading outputs of a block that are discarded
    int live_lo, live_hi;             // outputs outside [live_lo, live_hi) are exactly zero (input support + taps)
    int tap_res;                      // >= 0: offset of this render's residue table (257 segment pointers + 256 owners); < 0: no reflection taps
    int _pad0, _pad1;
};
struct FirTables {
    const cpx* tw;                    // w_256^i
    const cpx* twM_hi; const cpx* twM_lo;   // W_65536^(1024 i), W_65536^i (i < 1024)
    const int* res_ptr;               // per render with taps: 257 offsets into the residue-sorted tap arrays, then the 256 residues by descending count
    const int* tap_off; const real* tap_gain;     // residue-sorted taps
};

// W_65536^e = exp(-2 pi i e / 65536) from the unit itself (sincospi of an exactly representable argument).  Profiling
// (ncu, B200) showed these kernels bound by LSU wavefronts, not by the FP64 pipe: a table lookup at a per-lane address
// costs up to 32 wavefronts per warp instruction, ~45 FP64 instructions cost a third of that in SM time.
MS_DEV cpx w65536(unsigned e) {
    real sn, cs;
    r_sincospi((real)(e & 65535u) * (real)(1.0 / 32768.0), &sn, &cs);
    return mk(cs, -sn);
}
// v[m] *= W_65536^(a (lane + 32 m)):  base W^(a lane) per lane, step W^(32 a) (warp-uniform: one broadcast lookup),
// powers by a depth-4 product tree
MS_DEV void twiddle_row(cpx* v, const FirTables& T, int a, int lane) {
    const cpx base = w65536((unsigned)(a * lane));
    const cpx st1 = tw2level(T.twM_hi, T.twM_lo, (unsigned)(32 * a) & 65535u);
    const cpx st2 = c_mul(st1, st1);
    cpx t0 = base, t1 = c_mul(base, st1);
    v[0] = c_mul(v[0], t0); v[1] = c_mul(v[1], t1);
#pragma unroll
    for (int m = 2; m < 8; m += 2) {
        t0 = c_mul(t0, st2); t1 = c_mul(t1, st2);
        v[m] = c_mul(v[m], t0); v[m + 1] = c_mul(v[m + 1], t1);
    }
}

// ---- phase 1: forward columns -----------------------------------------------------------------------------
MS_DEV void fir_p1_tile(const FirUnit& U, const FirTables& T, cpx* S, int tile, const Ctx& c) {
    cpx* s = (cpx*)c.smem;
    const int lane = c.tid & 31, warp = c.tid >> 5;
    const int c0 = tile * FF_TILE;
    {
        // all sixteen loads are issued before the first dependent store (ncu: with load and store in one loop body every
        // STS waited out its own LDG -- half of this kernel's stall samples)
        cpx ld[FF_N * FF_TILE / FF_NTHR];
        const real* in = U.in;
        const long long pa0 = U.p0_a + c0, pb0 = U.p0_b + c0, nn = U.ols_n;
        const int has_b = U.has_b;
#pragma unroll
        for (int i = 0; i < FF_N * FF_TILE / FF_NTHR; ++i) {
            const int e = c.tid + FF_NTHR * i, n1 = e >> 3, cc = e & 7;
            const long long pa = pa0 + (long long)n1 * FF_N + cc, pb = pb0 + (long long)n1 * FF_N + cc;
            ld[i].x = (pa >= 0 && pa < nn) ? __ldg(&in[pa]) : (real)0.;
            ld[i].y = (has_b && pb >= 0 && pb < nn) ? __ldg(&in[pb]) : (real)0.;
        }
#pragma unroll
        for (int i = 0; i < FF_N * FF_TILE / FF_NTHR; ++i) {
            const int e = c.tid + FF_NTHR * i, n1 = e >> 3, cc = e & 7;
            s[cc * FF_RS + ms_pad(n1)] = ld[i];
        }
    }
    c.sync();
    cpx v[8];
    cpx* sw = s + warp * FF_RS;
#pragma unroll
    for (int q = 0; q < 8; ++q) v[q] = sw[ms_pad(lane + 32 * q)];
    c.syncwarp();
    warp_fft256(v, sw, T.tw, lane, c);
    const int n2 = c0 + warp;
    twiddle_row(v, T, n2, lane);                            // W^(k1 n2), k1 = lane + 32 m
    cpx* dst = S + (size_t)n2 * FF_N + lane;
#pragma unroll
    for (int m = 0; m < 8; ++m) dst[32 * m] = v[m];
    c.sync();                                               // the next tile refills the transposing buffer
}

// ---- phase 2: rows (forward, filter, inverse) ---------------------------------------------------------------
// The reflection taps are real, so E is Hermitian: E[65536 - k] = conj E[k], i.e. row 256 - k1 is row k1 reversed and
// conjugated (E[256 - k1][k2] = conj E[k1][255 - k2]).  A CTA therefore takes SIXTEEN rows in two passes of eight: pass A
// the rows k1 = 8 t + 1 .. 8 t + 8 (every warp folds nothing twice: the fold and the extra FFT run once per PAIR), pass B
// their partners 256 - k1 = 248 - 8 t .. 255 - 8 t, which reuse the E rows of pass A reversed and conjugated.  Every warp
// does the same work (one E transform + two row transforms in pass A, two row transforms in pass B), so nobody idles
// at the barriers (ncu on the previous form -- four rows + four partners per tile, warps 0-3 owning the E rows -- showed
// 18 % of the stall samples at the barrier where warps 4-7 waited for them), and both tile fetches are eight contiguous
// rows = full 128-byte segments.  Rows 0 and 128 are their own partners: in the last tile (k1 = 121 .. 128) pass B would
// meet row 128 again; that slot takes row 0 instead, whose E row is folded (no modulation: W^0) into the slot row 128's E
// occupied -- nobody needs that one in pass B.
#define FF_EROWS 8
#define FF_TILES2 (FF_N / 16)          // CTAs per unit in phase 2
// fold: F[k1][r] = sum over taps with off = r (mod 256) of g W_65536^(off k1); a thread owns one residue for the tile's
// eight rows, four at a time (W^(off k1) steps by W^off from row to row).  Residues are handed out by descending tap
// count (perm), so the lanes of a warp run the same number of iterations.  Out of line: its registers (two sincospi per
// tap) stay out of the transform code's allocation.
MS_DEV_NOINLINE void fir_fold_taps(const int* MS_RESTRICT rp, const int* MS_RESTRICT tap_off, const real* MS_RESTRICT tap_gain,
                                   cpx* sE, int k_first, int tid) {
    const int r = __ldg(&rp[257 + tid]);
    const int t_begin = __ldg(&rp[r]), t_end = __ldg(&rp[r + 1]);
#pragma unroll 1
    for (int half = 0; half < FF_EROWS; half += 4) {
        cpx acc[4];
#pragma unroll
        for (int w = 0; w < 4; ++w) acc[w] = c_zero();
        for (int t = t_begin; t < t_end; ++t) {
            const unsigned off = (unsigned)__ldg(&tap_off[t]);
            const real g = __ldg(&tap_gain[t]);
            cpx tw = w65536(off * (unsigned)(k_first + half));
            const cpx st = w65536(off);
#pragma unroll
            for (int w = 0; w < 4; ++w) {
                acc[w] = mk(acc[w].x + g * tw.x, acc[w].y + g * tw.y);
                if (w < 3) tw = c_mul(tw, st);
            }
        }
#pragma unroll
        for (int w = 0; w < 4; ++w) sE[(half + w) * FF_RS + ms_pad(r)] = acc[w];
    }
}
// the unmodulated fold of row 0 (k1 = 0: F[r] = sum of the gains of residue r), into one E row
MS_DEV_NOINLINE void fir_fold_row0(const int* MS_RESTRICT rp, const real* MS_RESTRICT tap_gain, cpx* row, int tid) {
    const int r = __ldg(&rp[257 + tid]);
    real f0 = (real)0.;
    for (int t = __ldg(&rp[r]); t < __ldg(&rp[r + 1]); ++t) f0 += __ldg(&tap_gain[t]);
    row[ms_pad(r)] = mk(f0, (real)0.);
}
// one pass of eight rows: fetch, FFT, * H, swap, FFT, twiddle, back.  row0 + slot = global row of tile slot `slot`
// (slot_zero >= 0: that slot holds row 0 instead); this warp works on slot `my`, whose filter row is IRspec[row] *
// (1 + E) with E = sE[erow] (rev: reversed and conjugated); own_e: the warp first transforms its E row in place.
// (second half of a pass) v = this warp's row spectrum: * H (filter `filt`), swap, inverse, twiddle, tile back into S
MS_DEV void fir_p2_filter_store(cpx* v, const cpx* filt, const FirTables& T, cpx* S, cpx* sB, const cpx* swE, int row0, int slot_zero,
                                int my, int row, int rev, int taps, const Ctx& c) {
    const int lane = c.tid & 31;
    cpx* sw = sB + my * FF_RS;
    {
        const cpx* f = filt + (size_t)row * FF_N + lane;
#pragma unroll
        for (int m = 0; m < 8; ++m) {
            cpx h = __ldg(&f[32 * m]);
            if (taps) {
                const int k2 = lane + 32 * m;
                const cpx e = rev ? c_conj(swE[ms_pad(FF_N - 1 - k2)]) : swE[ms_pad(k2)];
                h = c_mul(h, mk(e.x + (real)1.0, e.y));
            }
            v[m] = c_swap(c_mul(v[m], h));
        }
    }
    c.syncwarp();
    warp_fft256(v, sw, T.tw, lane, c);                      // inverse over k2 (swapped domain): index n2' = lane + 32 m
    twiddle_row(v, T, row, lane);
    c.syncwarp();
#pragma unroll
    for (int m = 0; m < 8; ++m) sw[ms_pad(lane + 32 * m)] = v[m];
    c.sync();
    {
        const int rr = c.tid & 7;
        const int rw = rr == slot_zero ? 0 : row0 + rr;
        cpx* dst = S + (size_t)(c.tid >> 3) * FF_N + rw;
#pragma unroll
        for (int i = 0; i < FF_N * FF_TILE / FF_NTHR; ++i) dst[(size_t)(FF_NTHR / 8) * FF_N * i] = sB[rr * FF_RS + ms_pad((c.tid >> 3) + (FF_NTHR / 8) * i)];
    }
    c.sync();
}
// PAIR (space_ir_stereo, two rows equal on the input side): the row spectrum is filtered twice -- by U.filt back into S,
// by filt_r into S_r -- from one tile fetch, one E transform and one forward row FFT.  Each channel's arithmetic is that
// of a lone unit with its filter, so each result is bit-identical to it.
template <bool PAIR>
MS_DEV void fir_p2_pass(const FirUnit& U, const FirTables& T, cpx* S, cpx* sB, cpx* sE, int row0, int slot_zero, int my, int erow, int rev,
                        int own_e, int taps, const Ctx& c, const cpx* filt_r = nullptr, cpx* S_r = nullptr) {
    const int lane = c.tid & 31;
    cpx v[8];
    {   // the tile: S[n2][rows of the pass] -> sB[slot][n2]   (all loads in flight before the first store)
        const int rr = c.tid & 7;
        const int rw = rr == slot_zero ? 0 : row0 + rr;
        const cpx* src = S + (size_t)(c.tid >> 3) * FF_N + rw;
#pragma unroll
        for (int i = 0; i < FF_N * FF_TILE / FF_NTHR; ++i) v[i] = MS_LDCG(&src[(size_t)(FF_NTHR / 8) * FF_N * i]);
#pragma unroll
        for (int i = 0; i < FF_N * FF_TILE / FF_NTHR; ++i) sB[rr * FF_RS + ms_pad((c.tid >> 3) + (FF_NTHR / 8) * i)] = v[i];
    }
    c.sync();                                               // the tile and the folded rows are in place
    cpx* swE = sE + erow * FF_RS;
    if (taps && own_e) {                                    // the warp's own E row, in place (only its owner touches it from here on)
#pragma unroll
        for (int q = 0; q < 8; ++q) v[q] = swE[ms_pad(lane + 32 * q)];
        c.syncwarp();
        warp_fft256(v, swE, T.tw, lane, c);                 // v[m] = E[row][k2 = lane + 32 m]
        c.syncwarp();
#pragma unroll
        for (int m = 0; m < 8; ++m) swE[ms_pad(lane + 32 * m)] = v[m];
        c.syncwarp();
    }
    const int row = my == slot_zero ? 0 : row0 + my;
    cpx* sw = sB + my * FF_RS;
#pragma unroll
    for (int q = 0; q < 8; ++q) v[q] = sw[ms_pad(lane + 32 * q)];
    c.syncwarp();
    warp_fft256(v, sw, T.tw, lane, c);                      // v[m] = Z[row][k2 = lane + 32 m]
    if (PAIR) {
        cpx z[8];
#pragma unroll
        for (int m = 0; m < 8; ++m) z[m] = v[m];
        fir_p2_filter_store(v, U.filt, T, S, sB, swE, row0, slot_zero, my, row, rev, taps, c);
        fir_p2_filter_store(z, filt_r, T, S_r, sB, swE, row0, slot_zero, my, row, rev, taps, c);
    } else {
        fir_p2_filter_store(v, U.filt, T, S, sB, swE, row0, slot_zero, my, row, rev, taps, c);
    }
}
template <bool PAIR>
MS_DEV void fir_p2_tile(const FirUnit& U, const FirTables& T, cpx* S, int tile, const Ctx& c, const cpx* filt_r = nullptr, cpx* S_r = nullptr) {
    cpx* sB = (cpx*)c.smem;                                 // transposing tile + exchange rows
    cpx* sE = sB + FF_TILE * FF_RS;                         // E rows of pass A (natural order k2)
    const int warp = c.tid >> 5;
    const int k_first = 8 * tile + 1;
    const int last = tile == FF_TILES2 - 1;                 // k1 = 121 .. 128
    const int taps = U.tap_res >= 0;
    if (taps) { fir_fold_taps(T.res_ptr + U.tap_res, T.tap_off, T.tap_gain, sE, k_first, c.tid); }
    // pass A: rows k_first + w, each warp its own E row
    fir_p2_pass<PAIR>(U, T, S, sB, sE, k_first, -1, warp, warp, 0, 1, taps, c, filt_r, S_r);
    // pass B: partners 256 - (k_first + w) = rowB0 + (7 - w); in the last tile slot 0 (row 128 again) takes row 0
    const int rowB0 = FF_N - (k_first + 7);
    if (taps && last) { fir_fold_row0(T.res_ptr + U.tap_res, T.tap_gain, sE + 7 * FF_RS, c.tid); }
    const int slot = 7 - warp;
    fir_p2_pass<PAIR>(U, T, S, sB, sE, rowB0, last ? 0 : -1, slot, warp, (last && warp == 7) ? 0 : 1, (last && warp == 7) ? 1 : 0, taps, c,
                      filt_r, S_r);
}

// ---- phase 3: inverse columns, valid outputs ------------------------------------------------------------------
MS_DEV void fir_p3_tile(const FirUnit& U, const FirTables& T, const cpx* S, int tile, const Ctx& c) {
    cpx* s = (cpx*)c.smem;
    const int lane = c.tid & 31, warp = c.tid >> 5;
    const int c0 = tile * FF_TILE;
    cpx v[8];
    const cpx* src = S + (size_t)(c0 + warp) * FF_N + lane;
#pragma unroll
    for (int q = 0; q < 8; ++q) v[q] = MS_LDCG(&src[32 * q]);
    cpx* sw = s + warp * FF_RS;
    warp_fft256(v, sw, T.tw, lane, c);                      // v[m]: sample n1 = lane + 32 m of column c0 + warp (swapped domain)
    c.syncwarp();
#pragma unroll
    for (int m = 0; m < 8; ++m) sw[ms_pad(lane + 32 * m)] = v[m];
    c.sync();
#pragma unroll
    for (int i = 0; i < FF_N * FF_TILE / FF_NTHR; ++i) {
        const int e = c.tid + FF_NTHR * i, n1 = e >> 3, cc = e & 7;
        const int idx = n1 * FF_N + c0 + cc;
        if (idx < U.ols_skip) continue;
        const cpx val = s[cc * FF_RS + ms_pad(n1)];
        const long long qa = U.p0_a + idx, qb = U.p0_b + idx;
        if (qa < U.ols_n) U.out[qa] = (qa >= U.live_lo && qa < U.live_hi) ? val.y : (real)0;       // un-swap: re of the inverse
        if (U.has_b && qb < U.ols_n) U.out[qb] = (qb >= U.live_lo && qb < U.live_hi) ? val.x : (real)0;
    }
    c.sync();
}

// ---- one phase per launch: grid = (FF_TILES, units); scratch block u belongs to unit u -----------------------------
MS_DEV void fir_phase_body(int phase, const FirUnit* MS_RESTRICT units, FirTables T, cpx* scratch, const Ctx& c) {
    const FirUnit& U = units[c.by];
    cpx* S = scratch + (size_t)c.by * (FF_N * FF_N);
    if (phase == 1) fir_p1_tile(U, T, S, c.bx, c);
    else if (phase == 2) fir_p2_tile<false>(U, T, S, c.bx, c);
    else fir_p3_tile(U, T, S, c.bx, c);
}
// phase 2 of pair units (space_ir_stereo): unit c.by is a left channel whose right channel is unit c.by + pair_off, with
// scratch block c.by + pair_off.  P1 ran for the left unit only; P3 runs for both.
MS_DEV void fir_p2_pair_body(const FirUnit* MS_RESTRICT units, int pair_off, FirTables T, cpx* scratch, const Ctx& c) {
    const FirUnit& U = units[c.by];
    fir_p2_tile<true>(U, T, scratch + (size_t)c.by * (FF_N * FF_N), c.bx, c, units[c.by + pair_off].filt,
                      scratch + (size_t)(c.by + pair_off) * (FF_N * FF_N));
}

// ---- reflection taps sorted by residue (off mod 256), once per plan ------------------------------------------------
// One CTA of 256 threads per render with taps: thread r counts and then copies the taps of residue r in tap order
// (deterministic, no atomics); res_ptr gets the 257 segment boundaries (absolute positions in the sorted arrays).
struct FirSortJob { int tap_begin, tap_end, res_at, _pad; };
MS_DEV void fir_sort_taps_body(const FirSortJob* MS_RESTRICT jobs, const int* MS_RESTRICT tap_off, const real* MS_RESTRICT tap_gain,
                               int* res_ptr, int* soff, real* sgain, const Ctx& c) {
    const FirSortJob J = jobs[c.by];
    int* cnt = (int*)c.smem;                                // 257 segment starts + 256 counts
    const int r = c.tid;
    int n = 0;
    for (int t = J.tap_begin; t < J.tap_end; ++t) {
        const int off = __ldg(&tap_off[t]);
        if (off >= 0 && off < FF_N * FF_N && (off & 255) == r) ++n;
    }
    cnt[r] = n;
    c.sync();
    if (r == 0) {
        int acc = J.tap_begin;
        for (int i = 0; i < 256; ++i) { const int k = cnt[i]; cnt[i] = acc; acc += k; }
        cnt[256] = acc;
    }
    c.sync();
    int at = cnt[r];
    res_ptr[J.res_at + r] = at;
    if (r == 0) res_ptr[J.res_at + 256] = cnt[256];
    // residues by descending tap count (ties by index): thread t of the fold owns residue perm[t], so the lanes of a
    // warp see (nearly) equal loop counts
    int* cn = cnt + 257;
    cn[r] = n;
    c.sync();
    int rank = 0;
    for (int i = 0; i < 256; ++i) { const int k = cn[i]; rank += (k > n || (k == n && i < r)) ? 1 : 0; }
    res_ptr[J.res_at + 257 + rank] = r;
    for (int t = J.tap_begin; t < J.tap_end; ++t) {
        const int off = __ldg(&tap_off[t]);
        if (off >= 0 && off < FF_N * FF_N && (off & 255) == r) { soff[at] = off; sgain[at] = __ldg(&tap_gain[t]); ++at; }
    }
}
