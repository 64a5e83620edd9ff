// ms_fft_core.cuh -- shared-memory Stockham FFT building blocks (forward DFT only).
//
// The inverse transform is never coded separately: IDFT(x) = swap(DFT(swap(x))) where swap
// exchanges real and imaginary parts, and every stage here is linear, so an inverse is "swap on the
// way in, swap on the way out" around the same forward passes (the inter-pass twiddles of a
// decimation-in-time inverse turn into forward twiddles under the same swap).
//
// A "tile" is `cnt` independent vectors of length F living in shared memory.  Each radix-R pass is
// the autosort Stockham step: butterfly j (0 <= j < F/R) reads x[j + q*F/R], q < R, multiplies by
// w_{Ns*R}^{q*(j mod Ns)}, takes a length-R DFT and writes to (j - j mod Ns)*R + (j mod Ns) + q*Ns.
// Passes ping-pong between two shared-memory buffers.  Natural order in, natural order out.

#define MS_MAX_RADICES 12

// Tile geometry: element i of vector v sits at complex index  v*vs + pad(i*es)  where pad() skews every
// 128 bytes of complex data (16 float2 / 8 double2 = all 32 banks) by one slot: that kills the stride-R
// bank conflicts of the early Stockham writes in the contiguous layout and is harmless in the column layout.
struct TileGeom {
    int cnt;   // vectors in the tile
    int vs;    // stride between vectors (float2 units, already padded)
    int es;    // stride between consecutive elements of one vector before padding
    int colmajor;  // 1: consecutive threads walk vectors (column tiles), 0: walk elements (row tiles)
};
MS_HD int ms_pad(int a) { return a + (a >> (sizeof(cpx) == 16 ? 3 : 4)); }
MS_HD int tile_addr(const TileGeom& g, int v, int i) { return v * g.vs + ms_pad(i * g.es); }

struct RadixPlan {
    int F;                       // vector length
    int nrad;                    // number of passes
    unsigned char rad[MS_MAX_RADICES];
    unsigned mg_ns[MS_MAX_RADICES];   // magic multipliers: x / Ns_i  == umulhi(x, mg_ns[i])  (0: divisor is 1)
    unsigned mg_pv[MS_MAX_RADICES];   //                    x / (F / rad_i)
    unsigned short tws[MS_MAX_RADICES];   // twiddle stride of pass i: F / (Ns_i * rad_i)
    unsigned mg_F;                    //                    x / F
};
// q = x / d for 0 <= x < 2^16-ish ranges used here (x * d' never overflows): m = floor(2^32 / d) + 1
static inline unsigned ms_magic(unsigned d) { return d <= 1 ? 0u : (unsigned)(0x100000000ull / d) + 1u; }
MS_HD unsigned ms_mulhi32(unsigned a, unsigned b) {
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return (unsigned)(((unsigned long long)a * b) >> 32);
#endif
}
MS_HD int ms_fastdiv(int x, unsigned magic) { return magic ? (int)ms_mulhi32((unsigned)x, magic) : x; }

// Factor F into radices from {8,4,2,3,5}.  Returns 0 if F has another prime factor.
static inline int ms_make_radix_plan(int F, RadixPlan* p) {
    p->F = F; p->nrad = 0;
    int e2 = 0, m = F;
    while (m % 2 == 0) { m /= 2; ++e2; }
    int n8 = e2 / 3, rem = e2 % 3;
    int n4 = 0, n2 = 0;
    if (rem == 1) { if (n8 > 0) { --n8; n4 = 2; } else n2 = 1; }
    else if (rem == 2) n4 = 1;
    for (int i = 0; i < n8; ++i) p->rad[p->nrad++] = 8;
    for (int i = 0; i < n4; ++i) p->rad[p->nrad++] = 4;
    for (int i = 0; i < n2; ++i) p->rad[p->nrad++] = 2;
    while (m % 5 == 0) { m /= 5; if (p->nrad >= MS_MAX_RADICES) return 0; p->rad[p->nrad++] = 5; }
    while (m % 3 == 0) { m /= 3; if (p->nrad >= MS_MAX_RADICES) return 0; p->rad[p->nrad++] = 3; }
    int Ns = 1;
    for (int i = 0; i < p->nrad; ++i) {
        p->mg_ns[i] = ms_magic((unsigned)Ns);
        p->mg_pv[i] = ms_magic((unsigned)(F / p->rad[i]));
        Ns *= p->rad[i];
        p->tws[i] = (unsigned short)(F / Ns);
    }
    p->mg_F = ms_magic((unsigned)F);
    return m == 1;
}


// ---- length-R forward DFTs in registers ---------------------------------------------------------
template <int R> struct Bfly;

template <> struct Bfly<2> {
    static MS_DEV void run(cpx* a) {
        cpx t = a[0];
        a[0] = c_add(t, a[1]);
        a[1] = c_sub(t, a[1]);
    }
};
template <> struct Bfly<4> {
    static MS_DEV void run(cpx* a) {
        cpx t0 = c_add(a[0], a[2]), t1 = c_sub(a[0], a[2]);
        cpx t2 = c_add(a[1], a[3]), t3 = c_mul_mi(c_sub(a[1], a[3]));
        a[0] = c_add(t0, t2); a[1] = c_add(t1, t3);
        a[2] = c_sub(t0, t2); a[3] = c_sub(t1, t3);
    }
};
template <> struct Bfly<3> {
    static MS_DEV void run(cpx* a) {
        const real h = (real)0.86602540378443864676;   // sin(2 pi / 3)
        cpx s = c_add(a[1], a[2]), d = c_sub(a[1], a[2]);
        cpx m = mk(a[0].x - (real)0.5 * s.x, a[0].y - (real)0.5 * s.y);
        cpx r = mk(h * d.y, -h * d.x);   // (-i h) * d
        a[0] = c_add(a[0], s);
        a[1] = c_add(m, r);
        a[2] = c_sub(m, r);
    }
};
template <> struct Bfly<5> {
    static MS_DEV void run(cpx* a) {
        const real c1 = (real)0.30901699437494742410, c2 = -(real)0.80901699437494742410;
        const real s1 = (real)0.95105651629515357212, s2 = (real)0.58778525229247312917;
        cpx p1 = c_add(a[1], a[4]), m1 = c_sub(a[1], a[4]);
        cpx p2 = c_add(a[2], a[3]), m2 = c_sub(a[2], a[3]);
        cpx a0 = a[0];
        cpx e1 = mk(a0.x + c1 * p1.x + c2 * p2.x, a0.y + c1 * p1.y + c2 * p2.y);
        cpx e2 = mk(a0.x + c2 * p1.x + c1 * p2.x, a0.y + c2 * p1.y + c1 * p2.y);
        cpx u1 = mk(s1 * m1.x + s2 * m2.x, s1 * m1.y + s2 * m2.y);
        cpx u2 = mk(s2 * m1.x - s1 * m2.x, s2 * m1.y - s1 * m2.y);
        cpx r1 = c_mul_mi(u1), r2 = c_mul_mi(u2);  // -i * u
        a[0] = mk(a0.x + p1.x + p2.x, a0.y + p1.y + p2.y);
        a[1] = c_add(e1, r1); a[4] = c_sub(e1, r1);
        a[2] = c_add(e2, r2); a[3] = c_sub(e2, r2);
    }
};
template <> struct Bfly<8> {
    static MS_DEV void run(cpx* a) {
        const real h = (real)0.70710678118654752440;
        cpx e[4] = {a[0], a[2], a[4], a[6]};
        cpx o[4] = {a[1], a[3], a[5], a[7]};
        Bfly<4>::run(e);
        Bfly<4>::run(o);
        cpx o1 = mk(h * (o[1].x + o[1].y), h * (o[1].y - o[1].x));      // * (1 - i)/sqrt2
        cpx o2 = c_mul_mi(o[2]);                                                // * -i
        cpx o3 = mk(h * (o[3].y - o[3].x), -h * (o[3].x + o[3].y));     // * (-1 - i)/sqrt2
        a[0] = c_add(e[0], o[0]); a[4] = c_sub(e[0], o[0]);
        a[1] = c_add(e[1], o1);   a[5] = c_sub(e[1], o1);
        a[2] = c_add(e[2], o2);   a[6] = c_sub(e[2], o2);
        a[3] = c_add(e[3], o3);   a[7] = c_sub(e[3], o3);
    }
};

// ---- one Stockham pass over a tile ----------------------------------------------------------------
// Out of place (src -> dst, two shared-memory buffers ping-pong): a thread finishes one butterfly
// before it starts the next, so nothing but the R values of a butterfly lives in registers and one
// barrier per pass suffices.  tw = table of w_F^i (i < F), forward sign.  Integer divisions by the
// per-pass constants go through host-computed magic multipliers.
template <int R, int CM>
MS_DEV void stockham_pass(const cpx* MS_RESTRICT src, cpx* MS_RESTRICT dst, const TileGeom& g, int per_vec, int Ns, int tws,
                          unsigned mg_ns, unsigned mg_pv, unsigned mg_cnt,
                          const cpx* MS_RESTRICT tw, const Ctx& c) {
    const int nb = per_vec * g.cnt;
#pragma unroll 2
    for (int b = c.tid; b < nb; b += c.nthr) {
        int vec, j;
        if (CM) { j = ms_fastdiv(b, mg_cnt); vec = b - j * g.cnt; } else { vec = ms_fastdiv(b, mg_pv); j = b - vec * per_vec; }
        const int k = j - ms_fastdiv(j, mg_ns) * Ns;
        cpx v[R];
#pragma unroll
        for (int q = 0; q < R; ++q) v[q] = src[tile_addr(g, vec, j + q * per_vec)];
        if (k != 0) {
            // powers of w = w_F^(k*tws): column-major tiles load w, w^2, w^4 (broadcast loads, each rounded once); row tiles
            // (a table address per lane) load w and square (see stockham_pass_ip)
            const cpx w1 = __ldg(&tw[k * tws]);
            if (R == 2) { v[1] = c_mul(v[1], w1); }
            else {
                const cpx w2 = CM ? __ldg(&tw[2 * k * tws]) : c_mul(w1, w1);
                if (R == 3) { v[1] = c_mul(v[1], w1); v[2] = c_mul(v[2], w2); }
                else {
                    const cpx w3 = c_mul(w1, w2);
                    if (R == 4) { v[1] = c_mul(v[1], w1); v[2] = c_mul(v[2], w2); v[3] = c_mul(v[3], w3); }
                    else {
                        const cpx w4 = CM ? __ldg(&tw[4 * k * tws]) : c_mul(w2, w2);
                        v[1] = c_mul(v[1], w1); v[2] = c_mul(v[2], w2); v[3] = c_mul(v[3], w3); v[4] = c_mul(v[4], w4);
                        if (R == 8) {
                            v[5] = c_mul(v[5], c_mul(w4, w1)); v[6] = c_mul(v[6], c_mul(w4, w2)); v[7] = c_mul(v[7], c_mul(w4, w3));
                        }
                    }
                }
            }
        }
        Bfly<R>::run(v);
        const int base = (j - k) * R + k;
#pragma unroll
        for (int q = 0; q < R; ++q) dst[tile_addr(g, vec, base + q * Ns)] = v[q];
    }
    c.sync();
}

// Full forward FFT of every vector of the tile.  `a` holds the input (caller synchronised after
// filling it), `b` is the second buffer of the same size.  Returns the buffer that holds the result.
MS_DEV unsigned ms_magic_dev(int d) { return d <= 1 ? 0u : (unsigned)(0x100000000ull / (unsigned)d) + 1u; }
template <int CM>
MS_DEV cpx* tile_fft(cpx* a, cpx* b, const TileGeom& g, const RadixPlan& p, const cpx* MS_RESTRICT tw, const Ctx& c) {
    int Ns = 1;
    const unsigned mg_cnt = CM ? ms_magic_dev(g.cnt) : 0u;
    int per_vec = p.F;
    for (int i = 0; i < p.nrad; ++i) {
        const int r = p.rad[i];
        const unsigned mn = p.mg_ns[i], mp = p.mg_pv[i];
        const int tws = p.tws[i];
        per_vec = tws * Ns;                      // F / r
        switch (r) {
            case 8: stockham_pass<8, CM>(a, b, g, per_vec, Ns, tws, mn, mp, mg_cnt, tw, c); break;
            case 4: stockham_pass<4, CM>(a, b, g, per_vec, Ns, tws, mn, mp, mg_cnt, tw, c); break;
            case 2: stockham_pass<2, CM>(a, b, g, per_vec, Ns, tws, mn, mp, mg_cnt, tw, c); break;
            case 3: stockham_pass<3, CM>(a, b, g, per_vec, Ns, tws, mn, mp, mg_cnt, tw, c); break;
            default: stockham_pass<5, CM>(a, b, g, per_vec, Ns, tws, mn, mp, mg_cnt, tw, c); break;
        }
        cpx* t = a; a = b; b = t;
        Ns *= r;
    }
    return a;
}

// (The generic passes stay ping-pong: run in place, a thread must hold ALL its butterflies of a pass in registers at
//  once -- 8..10 double-complex values for the radix 4/5/3/2 passes -- and at the 64-register budget that spills:
//  measured grain stage 17.2 -> 20.8 ms.  The static power-of-two tiles are radix 8 (+ radix-4 passes) and gain.)
// ---- in-place pass (static power-of-two tiles) ------------------------------------------------------
// In place: every thread pulls the inputs of its (at most BPT) butterflies into registers and transforms them, the
// CTA synchronises, then the results go back into the SAME buffer at the autosort positions.  Two barriers per
// pass, ONE tile buffer: half the shared memory of a ping-pong Stockham, i.e. more CTAs per SM, which is what these
// latency-bound passes need (measured on 256 x 256 FIR-stage tiles: 19.2 -> 15.3 ms).  tw = table of w_F^i (i < F), forward
// sign.  Integer divisions by the per-pass constants go through host-computed magic multipliers.
template <int R, int CM, int BPT>
MS_DEV void stockham_pass_ip(cpx* MS_RESTRICT buf, const TileGeom& g, int per_vec, int Ns, int tws,
                             unsigned mg_ns, unsigned mg_pv, unsigned mg_cnt, const cpx* MS_RESTRICT tw, const Ctx& c) {
    const int nb = per_vec * g.cnt;
    cpx v[BPT][R];
    int at[BPT], vecs[BPT];
#pragma unroll
    for (int u = 0; u < BPT; ++u) {
        const int b = c.tid + u * c.nthr;
        vecs[u] = -1;
        if (b < nb) {
            int vec, j;
            if (CM) { j = ms_fastdiv(b, mg_cnt); vec = b - j * g.cnt; } else { vec = ms_fastdiv(b, mg_pv); j = b - vec * per_vec; }
            const int k = j - ms_fastdiv(j, mg_ns) * Ns;
#pragma unroll
            for (int q = 0; q < R; ++q) v[u][q] = buf[tile_addr(g, vec, j + q * per_vec)];
            if (k != 0) {
                // powers of w = w_F^(k*tws).  Column-major tiles: the threads of a warp share a few k, the loads are
                // broadcasts -- w, w^2, w^4 come from the table (each rounded once).  Row tiles: every lane has its own k,
                // a lookup costs the L1 data pipe up to 32 sectors -- only w is loaded, the powers are squared.
                const cpx w1 = __ldg(&tw[k * tws]);
                if (R == 2) { v[u][1] = c_mul(v[u][1], w1); }
                else {
                    const cpx w2 = CM ? __ldg(&tw[2 * k * tws]) : c_mul(w1, w1);
                    if (R == 3) { v[u][1] = c_mul(v[u][1], w1); v[u][2] = c_mul(v[u][2], w2); }
                    else {
                        const cpx w3 = c_mul(w1, w2);
                        v[u][1] = c_mul(v[u][1], w1); v[u][2] = c_mul(v[u][2], w2); v[u][3] = c_mul(v[u][3], w3);
                        if (R > 4) {
                            const cpx w4 = CM ? __ldg(&tw[4 * k * tws]) : c_mul(w2, w2);
                            v[u][4 % R] = c_mul(v[u][4 % R], w4);
                            if (R == 8) {
                                v[u][5 % R] = c_mul(v[u][5 % R], c_mul(w4, w1)); v[u][6 % R] = c_mul(v[u][6 % R], c_mul(w4, w2));
                                v[u][7 % R] = c_mul(v[u][7 % R], c_mul(w4, w3));
                            }
                        }
                    }
                }
            }
            Bfly<R>::run(v[u]);
            at[u] = (j - k) * R + k; vecs[u] = vec;
        }
    }
    c.sync();
#pragma unroll
    for (int u = 0; u < BPT; ++u) {
        if (vecs[u] >= 0) {
#pragma unroll
            for (int q = 0; q < R; ++q) buf[tile_addr(g, vecs[u], at[u] + q * Ns)] = v[u][q];
        }
    }
    c.sync();
}
// Literal geometry: the magic divisions, strides and padded addresses fold into immediates.
template <unsigned D> struct MsMagic { static constexpr unsigned v = D <= 1 ? 0u : (unsigned)(0x100000000ull / (D ? D : 1)) + 1u; };
#define ms_magic_c(D) (MsMagic<(D)>::v)
// Static power-of-two transforms of CNT vectors of length F, F * CNT elements = 8 per thread (CNT * F / 8 threads),
// in place: 128 = 8.4.4, 1024 = 8.8.4.4.  Used by the block-wide in-tile Bluestein columns (B1 = 256 and 512 are warp-local).
template <int CM, int F, int CNT>
MS_DEV cpx* tile_fft_pow2(cpx* a, const TileGeom& g, const cpx* MS_RESTRICT tw, const Ctx& c) {
    static_assert(F == 128 || F == 1024, "static in-place tiles: 128 or 1024 points");
    constexpr unsigned mc = ms_magic_c(CNT);
    constexpr int P = F / 8;
    stockham_pass_ip<8, CM, 1>(a, g, P, 1, P, ms_magic_c(1), ms_magic_c(P), mc, tw, c);
    if (F == 128) {
        stockham_pass_ip<4, CM, 2>(a, g, 32, 8, 4, ms_magic_c(8), ms_magic_c(32), mc, tw, c);
        stockham_pass_ip<4, CM, 2>(a, g, 32, 32, 1, ms_magic_c(32), ms_magic_c(32), mc, tw, c);
    } else {        // 1024
        stockham_pass_ip<8, CM, 1>(a, g, 128, 8, 16, ms_magic_c(8), ms_magic_c(128), mc, tw, c);
        stockham_pass_ip<4, CM, 2>(a, g, 256, 64, 4, ms_magic_c(64), ms_magic_c(256), mc, tw, c);
        stockham_pass_ip<4, CM, 2>(a, g, 256, 256, 1, ms_magic_c(256), ms_magic_c(256), mc, tw, c);
    }
    return a;
}
// ---- warp-local 256-point forward FFT ---------------------------------------------------------------------
// in: v[q] = x[lane + 32 q];  out: v[m] = X[lane + 32 m].  sw: the warp's shared-memory row (FF_RS entries).
// The caller guarantees that nobody else touches sw and that the warp is converged.
MS_DEV void warp_fft256(cpx* v, cpx* sw, const cpx* MS_RESTRICT tw, int lane, const Ctx& c) {
    Bfly<8>::run(v);                                        // pass 1: Ns = 1, no twiddles; output q of butterfly j -> 8 j + q
#pragma unroll
    for (int q = 0; q < 8; ++q) sw[ms_pad(lane * 8 + q)] = v[q];
    c.syncwarp();
#pragma unroll
    for (int q = 0; q < 8; ++q) v[q] = sw[ms_pad(lane + 32 * q)];
    c.syncwarp();
    {                                                       // pass 2: Ns = 8, twiddle w_64^(q k) = w_256^(4 q k)
        const int k = lane & 7;
        // (one table load; the other powers by squaring: ncu has these kernels at ~90 % of the L1 data pipe, and the seven
        //  twiddle loads of a transform cost as many wavefronts as the transform's own data)
        const cpx w1 = __ldg(&tw[4 * k]), w2 = c_mul(w1, w1), w4 = c_mul(w2, w2);
        const cpx w3 = c_mul(w1, w2);
        v[1] = c_mul(v[1], w1); v[2] = c_mul(v[2], w2); v[3] = c_mul(v[3], w3); v[4] = c_mul(v[4], w4);
        v[5] = c_mul(v[5], c_mul(w4, w1)); v[6] = c_mul(v[6], c_mul(w4, w2)); v[7] = c_mul(v[7], c_mul(w4, w3));
        Bfly<8>::run(v);
        const int base = (lane - k) * 8 + k;
#pragma unroll
        for (int q = 0; q < 8; ++q) sw[ms_pad(base + 8 * q)] = v[q];
    }
    c.syncwarp();
#pragma unroll
    for (int q = 0; q < 8; ++q) v[q] = sw[ms_pad(lane + 32 * q)];
    c.syncwarp();
    {                                                       // pass 3: Ns = 64, radix 4; butterflies j = lane (even m) and lane + 32 (odd m)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int j = lane + 32 * h;
            const cpx w1 = __ldg(&tw[j]), w2 = c_mul(w1, w1);
            const cpx w3 = c_mul(w1, w2);
            cpx a[4] = {v[h], c_mul(v[2 + h], w1), c_mul(v[4 + h], w2), c_mul(v[6 + h], w3)};
            Bfly<4>::run(a);
            v[h] = a[0]; v[2 + h] = a[1]; v[4 + h] = a[2]; v[6 + h] = a[3];      // X[j + 64 q] -> m = 2 q + h
        }
    }
}

// ---- warp-local 512-point forward FFT -----------------------------------------------------------------------
// in: v[q] = x[lane + 32 q], q < 16;  out: v[m] = X[lane + 32 m].  Radix 8 . 8 . 8, two butterflies per lane and pass,
// two exchanges through the warp's own shared-memory row (ms_pad(512) + 1 entries), __syncwarp only.
MS_DEV void warp_fft512(cpx* v, cpx* sw, const cpx* MS_RESTRICT tw, int lane, const Ctx& c) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {                           // pass 1: Ns = 1; butterfly j = lane + 32 h takes x[j + 64 q] = v[2 q + h]
        cpx a[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) a[q] = v[2 * q + h];
        Bfly<8>::run(a);
#pragma unroll
        for (int q = 0; q < 8; ++q) sw[ms_pad(8 * (lane + 32 * h) + q)] = a[q];
    }
    c.syncwarp();
#pragma unroll
    for (int q = 0; q < 16; ++q) v[q] = sw[ms_pad(lane + 32 * q)];
    c.syncwarp();
    {                                                       // pass 2: Ns = 8, twiddle w_64^(q k) = w_512^(8 q k), k = j mod 8 = lane mod 8
        const int k = lane & 7;
        const cpx w1 = __ldg(&tw[8 * k]), w2 = c_mul(w1, w1), w4 = c_mul(w2, w2);
        const cpx w3 = c_mul(w1, w2), w5 = c_mul(w4, w1), w6 = c_mul(w4, w2), w7 = c_mul(w4, w3);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            cpx a[8] = {v[h], c_mul(v[2 + h], w1), c_mul(v[4 + h], w2), c_mul(v[6 + h], w3),
                        c_mul(v[8 + h], w4), c_mul(v[10 + h], w5), c_mul(v[12 + h], w6), c_mul(v[14 + h], w7)};
            Bfly<8>::run(a);
            const int base = (lane + 32 * h - k) * 8 + k;
#pragma unroll
            for (int q = 0; q < 8; ++q) sw[ms_pad(base + 8 * q)] = a[q];
        }
    }
    c.syncwarp();
#pragma unroll
    for (int q = 0; q < 16; ++q) v[q] = sw[ms_pad(lane + 32 * q)];
    c.syncwarp();
#pragma unroll
    for (int h = 0; h < 2; ++h) {                           // pass 3: Ns = 64, k = j = lane + 32 h, twiddle w_512^(q j); X[j + 64 q] -> m = 2 q + h
        const int j = lane + 32 * h;
        const cpx w1 = __ldg(&tw[j]), w2 = c_mul(w1, w1), w4 = c_mul(w2, w2);
        const cpx w3 = c_mul(w1, w2), w5 = c_mul(w4, w1), w6 = c_mul(w4, w2), w7 = c_mul(w4, w3);
        cpx a[8] = {v[h], c_mul(v[2 + h], w1), c_mul(v[4 + h], w2), c_mul(v[6 + h], w3),
                    c_mul(v[8 + h], w4), c_mul(v[10 + h], w5), c_mul(v[12 + h], w6), c_mul(v[14 + h], w7)};
        Bfly<8>::run(a);
#pragma unroll
        for (int q = 0; q < 8; ++q) v[2 * q + h] = a[q];
    }
}
