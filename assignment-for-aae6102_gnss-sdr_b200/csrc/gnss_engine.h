// gnss_engine.h -- the N = 16 * 125 * Q prime-factor FFT engine, one task per call.
//
// N = samples per ms (signal.Sample): 58 000 = 16*125*29, 26 000 = 16*125*13.
// 16, 125 and Q are pairwise coprime, so the N-point DFT is a twiddle-free 3-D
// DFT (Good-Thomas).  With the input index mapped by the "Good" map
//      n = (a*M1 + b*M2 + c*M3) mod N,          M1 = N/16, M2 = N/125, M3 = N/Q
// and the output index by the CRT map (m mod 16, m mod 125, m mod Q) = (a',b',c'):
//      Y[a',b',c'] = sum_{a,b,c} Z[a,b,c] W16^(a a') W125^(b b') WQ^(c c').
//
// A unit (one N-point transform) is spread over a thread-block cluster of R
// CTAs; CTA r keeps rows a in [r*16/R, (r+1)*16/R) of the [16][Q][125] array in
// shared memory ("D buffer", layout [a_local][c][pos]).  Four passes:
//   pass1  load (functor) + DFT-Q over c          task = (a_local, b)
//   pass2  125 = 5 x 25 : DFT-5 over b1 + W125    task = (row, b2),  b = 25 b1 + b2
//   pass3  DFT-25 over b2                         task = (row, k1);  pos 25 k1 + k2 holds b' = k1 + 5 k2
//   pass4  DFT-16 over a, columns split over the R CTAs (two adjacent columns per task, 16-byte
//          loads); reads the other CTAs' D buffers through distributed shared memory; store functor
//          (|.|^2 accumulate for the search, spectrum store for K0/K1)
// The functions below do ONE task each and take the thread's task index, so the
// same code runs under the CUDA kernels (gnss_kernels.cu) and under the CPU
// emulation used by the test-suite (tests/emu/).
//
// Replaces the arithmetic of acquisition.m:56-59 (fft / ifft built-ins).
#pragma once
#include "gnss_radix.h"

#if defined(__CUDACC__)
#include <cuda_runtime.h>
#else
#include <cmath>
#endif

namespace gnss {

template <int Q>
struct Geo {
    static constexpr int N = 2000 * Q;
    static constexpr int ROW = 125 * Q;           // columns (c', pos) per a-row
    static constexpr int NX = 16 * (2 * Q - 1) * 125;   // elements of a c-extended forward spectrum (K1 output)
    static constexpr int M1 = 125 * Q, M2 = 16 * Q, M3 = 2000;
    static constexpr int INV1 = cmodinv(M1 % 16, 16);
    static constexpr int INV2 = cmodinv(M2 % 125, 125);
    static constexpr int INV3 = cmodinv(M3 % Q, Q);
    static constexpr int E1 = M1 * INV1, E2 = M2 * INV2, E3 = M3 * INV3;   // CRT idempotents (< N each)
    static_assert(Q % 2 == 1 && Q % 5 != 0, "Q must be coprime to 2000");
    static_assert(INV1 && INV2 && INV3, "no modular inverse");

    GNSS_HD static int good(int a, int b, int c) { return (a * M1 + b * M2 + c * M3) % N; }
    GNSS_HD static int crt(int a, int b, int c) { return (a * E1 + b * E2 + c * E3) % N; }
    // storage index of Good coordinates (a,b,c) in a spectrum held in "G layout" [16][Q][125]
    GNSS_HD static int gidx(int a, int b, int c) { return (a * Q + c) * 125 + b; }
    // column id (c', pos) -> b' (pos = 25*k1 + k2 holds b' = k1 + 5*k2)
    GNSS_HD static int bprime_of_pos(int pos) { return pos / 25 + 5 * (pos % 25); }
    GNSS_HD static int pos_of_bprime(int bp) { return 25 * (bp % 5) + bp / 5; }
    // output lag / frequency index of (a', column)
    GNSS_HD static int lag_of(int ap, int col) {
        const int cp = col / 125, pos = col - cp * 125;
        return crt(ap, bprime_of_pos(pos), cp);
    }
    // Good coordinates of frequency index (k - s): shift amounts per axis (SURVEY A.7)
    GNSS_HD static void shift_coords(int s, int& sa, int& sb, int& sc) {
        int sm = s % N; if (sm < 0) sm += N;
        sa = (int)(((long long)sm * INV1) % 16);
        sb = (int)(((long long)sm * INV2) % 125);
        sc = (int)(((long long)sm * INV3) % Q);
    }
    GNSS_HD static void cell_of_lag(int m, int& ap, int& col) {
        ap = m & 15;
        col = (m % Q) * 125 + pos_of_bprime(m % 125);
    }
};

// Transposed exchange layout ("XT") of the cooperative search kernel: pass 3 leaves its results for pass 4
// directly in the L2-resident exchange buffer as [16 a][25 k2][NTP] with t = c'*5 + k1 fastest, so that the
// 25 stores of a pass-3 task are coalesced across the lanes of a warp (no shared-memory write, no copy-out
// pass) and pass 4 still reads 16-byte pairs.  NTP = 5Q + 1 keeps rows even (pair alignment); column t = 5Q
// of every k2 row is padding.
template <int Q>
struct GeoX {
    static constexpr int NT = 5 * Q;               // pass-3 tasks per a-row
    static constexpr int NTP = NT + (NT & 1);      // padded (even)
    static constexpr int RSX = 25 * NTP;           // cf per a-row of the exchange buffer
    GNSS_HD static bool valid(int e) { return e < RSX && (e % NTP) < NT; }
    // lag of (a', e)
    GNSS_HD static int lag_of(int ap, int e) {
        const int k2 = e / NTP, t = e - k2 * NTP;
        const int cp = t / 5, k1 = t - cp * 5;
        return Geo<Q>::crt(ap, k1 + 5 * k2, cp);
    }
    GNSS_HD static void cell_of_lag(int m, int& ap, int& e) {
        ap = m & 15;
        const int bp = m % 125;
        e = (bp / 5) * NTP + (m % Q) * 5 + (bp % 5);
    }
};
template <int Q, int R>
struct SplitX {
    static constexpr int CHX = 2 * ((GeoX<Q>::RSX + 2 * R - 1) / (2 * R));   // exchange columns per CTA (even)
    static constexpr int ACC_ELEMS = 16 * CHX;
    static constexpr int P4_TASKS = CHX / 2;
};

template <int Q, int R>
struct Split {
    static_assert(R == 1 || R == 2 || R == 4 || R == 8 || R == 16, "CTAs per transform");
    static constexpr int A = 16 / R;                       // a-rows per CTA
    static constexpr int ROW = Geo<Q>::ROW;                // real columns per a-row
    static constexpr int RS = ROW + (ROW & 1);             // a-row stride in cf: even, so column pairs are 16-B aligned
    static constexpr int CH = 2 * ((ROW + 2 * R - 1) / (2 * R));   // pass-4 columns per CTA (even)
    static constexpr int D_ELEMS = A * RS;                 // cf per CTA
    static constexpr int ACC_ELEMS = 16 * CH;              // floats per CTA
    static constexpr int NR = A * Q;                       // (a_local, c') rows of 125 per CTA
    static constexpr int P1_TASKS = A * 125;
    static constexpr int P2_H = (Q + 15) / 16;             // half-warps per (a_local, b2) column of Q rows
    static constexpr int P2_TASKS = A * 25 * P2_H * 16;    // lane slots (slots with c' >= Q idle)
    static constexpr int P3_TASKS = NR * 5;
    static constexpr int P4_TASKS = CH / 2;                // column PAIRS
};

// ------------------------------------------------------------------ pass 1
// compute half: load (functor) + DFT-Q over c, result left in registers
template <int Q, int R, class Loader>
GNSS_HD void pass1_compute(int task, int rank, const Loader& ld, cf (&z)[Q]) {
    using S = Split<Q, R>;
    const int al = task / 125, b = task - al * 125;
    if constexpr (Loader::kStreams) {
        const auto ctx = ld.template begin<Q>(rank * S::A + al, b);
        dft_odd_stream<Q>([&](auto cc) { return ld.template at<Q, decltype(cc)::value>(ctx); }, z);
    } else {
        ld.template load<Q>(rank * S::A + al, b, z);
        dft_odd<Q>(z);
    }
}
// store half: D[a_local][c'][b]
template <int Q, int R>
GNSS_HD void pass1_store(int task, const cf (&z)[Q], cf* __restrict__ D) {
    using S = Split<Q, R>;
    const int al = task / 125, b = task - al * 125;
    cf* dst = D + al * S::RS + b;
    static_for<0, Q>([&](auto cc) {
        constexpr int C = decltype(cc)::value;
        dst[C * 125] = z[C];
    });
}
template <int Q, int R, class Loader>
GNSS_HD void pass1_task(int task, int rank, const Loader& ld, cf* __restrict__ D) {
    cf z[Q];
    pass1_compute<Q, R>(task, rank, ld, z);
    pass1_store<Q, R>(task, z, D);
}

// ------------------------------------------------------------------ pass 2
// Twiddle table: tw[b2*4 + (k1-1)] describes W125^(b2*k1) = c + i*s (s <= 0) as {c, 0, -s, s}: one 16-byte
// (broadcast) load gives the scalar c and the register pair (-s, s) that the two packed instructions of the
// complex multiply take as they are (u*w = c*u + (-s, s) (.) (u.y, u.x)).
struct alignas(16) Tw4 {
    float c, pad, ns, s;
};
GNSS_HD cf cmul_tw4(cf u, const Tw4& w) {
#ifdef GNSS_PACKED
    const float2 t = __fmul2_rn(f2(u), make_float2(w.c, w.c));
    return fc(__ffma2_rn(make_float2(u.y, u.x), make_float2(w.ns, w.s), t));
#else
    return mk(u.x * w.c + u.y * w.ns, u.y * w.c + u.x * w.s);
#endif
}
// Lane slot -> (a_local, b2, c'): the 16 lanes of a half-warp walk 16 consecutive c' of ONE (a_local, b2)
// column.  Row stride 125 cf = 13 bank-pairs (mod 16), a generator of Z16, so each half-warp touches 16
// distinct bank-pairs: conflict-free 64-bit accesses, and the twiddle reads are broadcasts.  Slots with
// c' >= Q idle (Q = 13: 3 of 16, Q = 29: 3 of 32); the denser mapping that wraps into the next b2 cost
// 1.4-2.0x the shared-memory wavefronts (ncu r01).
// One cell = column ab = a_local*25 + b2, row c: DFT-5 over b1 (b = 25*b1 + b2) + the W125 twiddle.
template <int Q, int R>
GNSS_HD cf* pass2_cell_ptr(int ab, int c, cf* __restrict__ D, int& b2) {
    using S = Split<Q, R>;
    if constexpr (S::A == 1) {
        b2 = ab;
        return D + c * 125 + ab;
    } else {
        const int al = ab / 25;
        b2 = ab - al * 25;
        return D + al * S::RS + c * 125 + b2;
    }
}
template <int Q, int R>
GNSS_HD void pass2_cell(int ab, int c, cf* __restrict__ D, const Tw4* __restrict__ tw) {
    int b2;
    cf* p = pass2_cell_ptr<Q, R>(ab, c, D, b2);
    cf u[5] = {p[0], p[25], p[50], p[75], p[100]};
    const Tw4* w = tw + 4 * b2;
    const Tw4 w1 = w[0], w2 = w[1], w3 = w[2], w4 = w[3];
    dft_odd<5>(u);
    p[0] = u[0];
    p[25] = cmul_tw4(u[1], w1);
    p[50] = cmul_tw4(u[2], w2);
    p[75] = cmul_tw4(u[3], w3);
    p[100] = cmul_tw4(u[4], w4);
}
// two cells of one row at once: all loads, then all math, then all stores (memory-level parallelism)
template <int Q, int R>
GNSS_HD void pass2_cell2(int ab0, int ab1, int c, cf* __restrict__ D, const Tw4* __restrict__ tw) {
    int b20, b21;
    cf* p0 = pass2_cell_ptr<Q, R>(ab0, c, D, b20);
    cf* p1 = pass2_cell_ptr<Q, R>(ab1, c, D, b21);
    cf u[5] = {p0[0], p0[25], p0[50], p0[75], p0[100]};
    cf v[5] = {p1[0], p1[25], p1[50], p1[75], p1[100]};
    const Tw4* wu = tw + 4 * b20;
    const Tw4* wv = tw + 4 * b21;
    const Tw4 wu1 = wu[0], wu2 = wu[1], wu3 = wu[2], wu4 = wu[3];
    const Tw4 wv1 = wv[0], wv2 = wv[1], wv3 = wv[2], wv4 = wv[3];
    dft_odd<5>(u);
    dft_odd<5>(v);
    p0[0] = u[0];
    p1[0] = v[0];
    p0[25] = cmul_tw4(u[1], wu1);
    p1[25] = cmul_tw4(v[1], wv1);
    p0[50] = cmul_tw4(u[2], wu2);
    p1[50] = cmul_tw4(v[2], wv2);
    p0[75] = cmul_tw4(u[3], wu3);
    p1[75] = cmul_tw4(v[3], wv3);
    p0[100] = cmul_tw4(u[4], wu4);
    p1[100] = cmul_tw4(v[4], wv4);
}
// The whole pass for a CTA of T threads.  Half-warp hw = tid/16 (+ T/16 per round) serves row block
// h = hw % P2_H of column ab = hw / P2_H; T/16 is a multiple of P2_H, so a thread's row c is fixed and its
// columns are ab0, ab0 + G, ab0 + 2G, ... : no per-round index arithmetic beyond one addition.
template <int Q, int R, int T>
GNSS_HD void pass2_cta(int tid, cf* __restrict__ D, const Tw4* __restrict__ tw) {
    using S = Split<Q, R>;
    static_assert((T / 16) % S::P2_H == 0, "half-warps per CTA must be a multiple of the row blocks");
    constexpr int G = (T / 16) / S::P2_H;          // columns per round
    constexpr int NAB = S::A * 25;
    const int hw = tid >> 4;
    const int c = (hw % S::P2_H) * 16 + (tid & 15);
    if (c >= Q) return;
    int ab = hw / S::P2_H;
    for (; ab + G < NAB; ab += 2 * G) pass2_cell2<Q, R>(ab, ab + G, c, D, tw);
    if (ab < NAB) pass2_cell<Q, R>(ab, c, D, tw);
}
// slot form (CPU emulation): slot = half-warp * 16 + lane over all P2_TASKS lane slots
template <int Q, int R>
GNSS_HD void pass2_task(int slot, cf* __restrict__ D, const Tw4* __restrict__ tw) {
    using S = Split<Q, R>;
    const int hw = slot >> 4, l = slot & 15;
    const int c = (hw % S::P2_H) * 16 + l;
    if (c >= Q) return;
    pass2_cell<Q, R>(hw / S::P2_H, c, D, tw);
}

// ------------------------------------------------------------------ pass 3
template <int Q, int R>
GNSS_HD void pass3_task(int task, cf* __restrict__ D) {
    using S = Split<Q, R>;
    const int al = task / (5 * Q);    // task = row*5 + k1, row = a_local*Q + c'
    cf* p = D + task * 25 + al * (S::RS - S::ROW);   // row*125 + 25*k1 (+ a-row padding)
    cf v[25];
    static_for<0, 25>([&](auto ic) {
        constexpr int I = decltype(ic)::value;
        v[I] = p[I];
    });
    dft25(v);                          // v[5*q1+q2] = X[q1 + 5*q2]
    static_for<0, 25>([&](auto ic) {
        constexpr int I = decltype(ic)::value;       // output index k2 = I
        p[I] = v[5 * (I % 5) + I / 5];
    });
}

// pass 3, results to the XT exchange buffer instead of back into D.  xrow0 = &buf[a = rank*A][0][0].
template <int Q, int R>
GNSS_HD void pass3_task_xt(int task, const cf* __restrict__ D, cf* __restrict__ xrow0) {
    using S = Split<Q, R>;
    using X = GeoX<Q>;
    const int al = task / (5 * Q);
    const cf* p = D + task * 25 + al * (S::RS - S::ROW);
    cf v[25];
    static_for<0, 25>([&](auto ic) {
        constexpr int I = decltype(ic)::value;
        v[I] = p[I];
    });
    dft25(v);
    cf* q = xrow0 + al * X::RSX + (task - al * X::NT);        // [al][k2 = 0][t]
    static_for<0, 25>([&](auto ic) {
        constexpr int I = decltype(ic)::value;                 // k2 = I
        q[I * X::NTP] = v[5 * (I % 5) + I / 5];
    });
}
// pass 4 over the XT buffer: task j = exchange columns (e, e+1), e = rank*CHX + 2j
template <int Q, int R, class Storer>
GNSS_HD void pass4_task_xt(int j, int rank, const cf* __restrict__ X, Storer& st) {
    using GX = GeoX<Q>;
    using SX = SplitX<Q, R>;
    const int t = 2 * j;
    const int e = rank * SX::CHX + t;
    if (t >= SX::CHX || e >= GX::RSX) return;
    cf w0[16], w1[16];
    static_for<0, 16>([&](auto ac) {
        constexpr int Aidx = decltype(ac)::value;
        const cf2 v = ld_cg2(reinterpret_cast<const cf2*>(X + Aidx * GX::RSX + e));
        w0[Aidx] = v.lo;
        w1[Aidx] = v.hi;
    });
    dft16(w0);
    dft16(w1);
    st.template store2x<Q, R>(t, w0, w1);
}

// ------------------------------------------------------------------ pass 4
// Dall[r] = D buffer of cluster CTA r (DSMEM-mapped on the GPU).  One task = two adjacent columns:
// the 16 rows are fetched with 16-byte loads (half the number of remote requests).
template <int Q, int R, class Storer>
GNSS_HD void pass4_task(int j, int rank, cf* const* Dall, Storer& st) {
    using S = Split<Q, R>;
    const int t = 2 * j;
    const int col = rank * S::CH + t;
    if (t >= S::CH || col >= S::ROW) return;
    cf w0[16], w1[16];
    static_for<0, 16>([&](auto ac) {
        constexpr int Aidx = decltype(ac)::value;
        const cf2 v = *reinterpret_cast<const cf2*>(Dall[Aidx / S::A] + (Aidx % S::A) * S::RS + col);
        w0[Aidx] = v.lo;
        w1[Aidx] = v.hi;
    });
    dft16(w0);                         // w[4*k1+k2] = Y[a' = k1 + 4*k2]
    dft16(w1);
    st.template store2<Q, R>(col, t, w0, w1);
}

// Same pass, but the 16 rows come from one flat [16][RS] array in global memory (the L2-resident
// exchange buffer the cluster's CTAs copied their finished rows into), read with L2-only loads.
template <int Q, int R, class Storer>
GNSS_HD void pass4_task_flat(int j, int rank, const cf* __restrict__ X, Storer& st) {
    using S = Split<Q, R>;
    const int t = 2 * j;
    const int col = rank * S::CH + t;
    if (t >= S::CH || col >= S::ROW) return;
    cf w0[16], w1[16];
    static_for<0, 16>([&](auto ac) {
        constexpr int Aidx = decltype(ac)::value;
        const cf2 v = ld_cg2(reinterpret_cast<const cf2*>(X + Aidx * S::RS + col));
        w0[Aidx] = v.lo;
        w1[Aidx] = v.hi;
    });
    dft16(w0);
    dft16(w1);
    st.template store2<Q, R>(col, t, w0, w1);
}

// ================================================================== functors
// ---- search (K2): Z = Cc * X_base[k - s], accumulate |Y|^2 ----
struct SearchLoader {
    const cf* __restrict__ cc;      // conj(fft(code))/N of this PRN, G layout [16][Q][125]
    const cf* __restrict__ x;       // fft(wiped-off block) of this (base, block), c-extended G layout
                                    // [16][2Q-1][125] (plane c and c+Q hold the same data), so the
                                    // rotation (c - sc) mod Q is a plain offset
    int sa, sb, sc;                 // bin shift in Good coordinates (SURVEY A.7)
    static constexpr bool kStreams = true;
    struct Ctx { const cf* pc; const cf* px; };
    template <int Q>
    GNSS_HD Ctx begin(int a, int b) const {
        const int as = (a - sa) & 15;
        int bs = b - sb; if (bs < 0) bs += 125;
        const int c0 = (sc == 0) ? 0 : Q - sc;
        Ctx c;
        c.pc = cc + (a * Q) * 125 + b;
        c.px = x + (as * (2 * Q - 1) + c0) * 125 + bs;
        return c;
    }
    template <int Q, int C>
    GNSS_HD cf at(const Ctx& c) const {
#if defined(GNSS_EXPERIMENT_NOCC)      // timing only (wrong results): no code-spectrum traffic
        return cmul_scalar(mk(1.0f + (float)C, 0.5f), ld_ro(c.px + C * 125));
#elif defined(GNSS_EXPERIMENT_NOX)     // timing only: no forward-spectrum traffic
        return cmul_scalar(ld_ro(c.pc + C * 125), mk(1.0f + (float)C, 0.5f));
#else
        return cmul_scalar(ld_ro(c.pc + C * 125), ld_ro(c.px + C * 125));
#endif
    }
    template <int Q>
    GNSS_HD void load(int a, int b, cf (&z)[Q]) const {
        const int as = (a - sa) & 15;
        int bs = b - sb; if (bs < 0) bs += 125;
        const int c0 = (sc == 0) ? 0 : Q - sc;       // (0 - sc) mod Q
        const cf* pc = cc + (a * Q) * 125 + b;
        const cf* px = x + (as * (2 * Q - 1) + c0) * 125 + bs;
        static_for<0, Q>([&](auto c_) {
            constexpr int C = decltype(c_)::value;
            z[C] = cmul_scalar(ld_ro(pc + C * 125), ld_ro(px + C * 125));
        });
    }
};

struct PowerAccumStorer {
    float* __restrict__ acc;        // [16][CH] (or [16][CHX] in the XT layout) floats of this CTA
    template <int Q, int R>
    GNSS_HD void store2x(int t, const cf (&w0)[16], const cf (&w1)[16]) {
        constexpr int CHX = SplitX<Q, R>::CHX;
        static_for<0, 16>([&](auto i_) {
            constexpr int I = decltype(i_)::value;
            constexpr int AP = (I / 4) + 4 * (I % 4);
            cf* p = reinterpret_cast<cf*>(acc + AP * CHX + t);
            cf v = *p;
            v.x = cnorm_acc(w0[I], v.x);
            v.y = cnorm_acc(w1[I], v.y);
            *p = v;
        });
    }
    template <int Q, int R>
    GNSS_HD void store2(int /*col*/, int t, const cf (&w0)[16], const cf (&w1)[16]) {
        constexpr int CH = Split<Q, R>::CH;
        static_for<0, 16>([&](auto i_) {
            constexpr int I = decltype(i_)::value;               // w[I], I = 4*k1 + k2
            constexpr int AP = (I / 4) + 4 * (I % 4);            // a' = k1 + 4*k2
            cf* p = reinterpret_cast<cf*>(acc + AP * CH + t);    // t even, CH even: 8-byte aligned
            cf v = *p;
            v.x = cnorm_acc(w0[I], v.x);
            v.y = cnorm_acc(w1[I], v.y);
            *p = v;
        });
    }
};

// Register-resident accumulator of the cooperative search kernel (r02; VERDICT r01 item 2-ii): every engine variant has at most
// ONE pass-4 task per thread (P4_TASKS <= T), so the 2 x 16 accumulators of that task can stay in registers for all
// K blocks of a row; shared memory sees them once per row (dump before the row end) instead of a read-modify-write
// per block.
struct RegAccumStorer {
    float (&a0)[16];
    float (&a1)[16];
    template <int Q, int R>
    GNSS_HD void store2x(int /*t*/, const cf (&w0)[16], const cf (&w1)[16]) {
        static_for<0, 16>([&](auto i_) {
            constexpr int I = decltype(i_)::value;
            constexpr int AP = (I / 4) + 4 * (I % 4);
            a0[AP] = cnorm_acc(w0[I], a0[AP]);
            a1[AP] = cnorm_acc(w1[I], a1[AP]);
        });
    }
};

// ---- spectrum store (K0 / K1): write Y to global in G layout of the *next* transform ----
struct SpectrumStorer {
    cf* __restrict__ out;
    float scale;                    // 1 for K1, 1/N for K0
    int conj;                       // 1 for K0 (store conj(fft(code))/N)
    int extended;                   // 1 for K1: c-extended layout [16][2Q-1][125], planes c and c+Q
    template <int Q, int R>
    GNSS_HD void store1(int col, const cf (&w)[16]) {
        using G = Geo<Q>;
        const int cp = col / 125, pos = col - cp * 125;
        const int bp = G::bprime_of_pos(pos);
        const int bg = (bp * G::INV2) % 125, cg = (cp * G::INV3) % Q;
        const int planes = extended ? 2 * Q - 1 : Q;
        static_for<0, 16>([&](auto i_) {
            constexpr int I = decltype(i_)::value;
            constexpr int AP = (I / 4) + 4 * (I % 4);
            constexpr int AG = (AP * G::INV1) % 16;
            cf v = w[I];
            v.x *= scale;
            v.y *= conj ? -scale : scale;
            out[(AG * planes + cg) * 125 + bg] = v;
            if (extended && cg + Q < planes) out[(AG * planes + cg + Q) * 125 + bg] = v;
        });
    }
    template <int Q, int R>
    GNSS_HD void store2(int col, int /*t*/, const cf (&w0)[16], const cf (&w1)[16]) {
        store1<Q, R>(col, w0);
        if (col + 1 < Geo<Q>::ROW) store1<Q, R>(col + 1, w1);
    }
};

// ---- code replica loader (K0): real +-1 samples, natural order ----
struct CodeLoader {
    static constexpr bool kStreams = false;
    const int8_t* __restrict__ scode;   // N samples of this PRN (acquisition.m:51)
    template <int Q>
    GNSS_HD void load(int a, int b, cf (&z)[Q]) const {
        static_for<0, Q>([&](auto c_) {
            constexpr int C = decltype(c_)::value;
            z[C] = mk((float)scode[Geo<Q>::good(a, b, C)], 0.f);
        });
    }
};

// ---- wipe-off loader (K1): acquisition.m:43,56 with exact phase, plus the M-ms fold (A.8) ----
GNSS_HD void carrier_sincos(double f_hz, double fs_hz, long long n1 /*1-based sample index*/,
                            float& co, float& si) {
    // cycles = f*(n)/Fs ; f*n is exact in double for integer-Hz f (|f*n| < 2^53)
    const double cyc = (f_hz * (double)n1) / fs_hz;
    const double fr = cyc - floor(cyc);                  // [0,1)
#if defined(__CUDA_ARCH__)
    sincospif((float)(2.0 * fr), &si, &co);
#else
    const double ang = 2.0 * 3.14159265358979323846 * fr;
    co = (float)cos(ang);
    si = (float)sin(ang);
#endif
}

struct WipeoffLoader {
    static constexpr bool kStreams = false;
    const void* __restrict__ raw;   // start of this coherent block (sample 0 of the block)
    int data_type;                  // 1 real, 2 I/Q          (file.dataType)
    int precision;                  // 1 int8, 2 int16        (file.dataPrecision)
    int coh_ms;                     // M
    double f_hz, fs_hz;             // IF + doppler of this base, Fs
    float mean_i, mean_q;           // int16 path only (acquisition.m:32)
    template <int Q>
    GNSS_HD void load(int a, int b, cf (&z)[Q]) const {
        constexpr int N = Geo<Q>::N;
        static_for<0, Q>([&](auto c_) {
            constexpr int C = decltype(c_)::value;
            const int n = Geo<Q>::good(a, b, C);
            float ax = 0.f, ay = 0.f;
            for (int j = 0; j < coh_ms; ++j) {
                const long long idx = (long long)j * N + n;
                float xi, xq;
                if (precision == 2) {
                    const int16_t* p = (const int16_t*)raw;
                    xi = (float)p[2 * idx] - mean_i;
                    xq = (float)p[2 * idx + 1] - mean_q;
                } else if (data_type == 2) {
                    const int8_t* p = (const int8_t*)raw;
                    xi = (float)p[2 * idx];
                    xq = (float)p[2 * idx + 1];
                } else {
                    xi = (float)((const int8_t*)raw)[idx];
                    xq = 0.f;
                }
                float co, si;
                carrier_sincos(f_hz, fs_hz, idx + 1, co, si);
                ax += xi * co - xq * si;
                ay += xi * si + xq * co;
            }
            z[C] = mk(ax, ay);
        });
    }
};

// ---- fine-frequency loader (acquisition.m:104-110): code wipe-off of the long block, decimated by L,
//      modulated for residue r of the zero-padded spectrum.  The length-F (F = K*L*N) spectrum of the
//      L*N code-stripped samples s[n] is  X[K*(q1 + N*q2) + r] = sum_{n2<L} W_L^{n2 q2} W_{LN}^{n2 q1}
//      DFT_N{ s[L*n1 + n2] * exp(-2*pi*i*(L*n1+n2)*r/F) }[q1] : K*L transforms of N points. ----
struct FineLoader {
    static constexpr bool kStreams = false;
    const void* __restrict__ raw;        // (L+1) ms block as read at acquisition.m:91/96
    const uint16_t* __restrict__ chip;   // [L*N] chip index of sample t (acquisition.m:104-105), 0-based
    const int8_t* __restrict__ ca;       // [1023] C/A chips of this SV
    int data_type, precision;
    float mean_i, mean_q;                // int16 path (acquisition.m:94)
    int start;                           // 0-based first sample = N - codedelay - 1 (acquisition.m:106)
    int L, n2, r;
    long long F;                         // fftlength = L*N*datalen (acquisition.m:108)
    // decimated sample n1 (of N), code-stripped and modulated for residue r
    GNSS_HD cf sample(int n1) const {
        const long long n = (long long)L * n1 + n2;
        const long long idx = (long long)start + n;
        float xi, xq;
        if (precision == 2) {
            const int16_t* p = (const int16_t*)raw;
            xi = (float)p[2 * idx] - mean_i;
            xq = (float)p[2 * idx + 1] - mean_q;
        } else if (data_type == 2) {
            const int8_t* p = (const int8_t*)raw;
            xi = (float)p[2 * idx];
            xq = (float)p[2 * idx + 1];
        } else {
            xi = (float)((const int8_t*)raw)[idx];
            xq = 0.f;
        }
        const float cv = (float)ca[chip[n]];
        xi *= cv;
        xq *= cv;
        const long long m = (n * (long long)r) % F;          // exact phase numerator
        const double fr = (double)m / (double)F;
        float co, si;
#if defined(__CUDA_ARCH__)
        sincospif((float)(2.0 * fr), &si, &co);
#else
        co = (float)cos(2.0 * 3.14159265358979323846 * fr);
        si = (float)sin(2.0 * 3.14159265358979323846 * fr);
#endif
        // (xi + i xq) * (co - i si)
        return mk(xi * co + xq * si, xq * co - xi * si);
    }
    template <int Q>
    GNSS_HD void load(int a, int b, cf (&z)[Q]) const {
        static_for<0, Q>([&](auto c_) {
            constexpr int C = decltype(c_)::value;
            z[C] = sample(Geo<Q>::good(a, b, C));
        });
    }
};

// ---- zero-padded shapes: each ms of n_ms < N samples is the start of an N-point transform ----
// K1 (acquisition.m:43,56): WipeoffLoader with the fold's stride and the sample count per ms taken at run time;
// inputs n >= n_ms are the zero padding.  The carrier phase is that of sample j*n_ms + n + 1 of the coherent block.
struct PadWipeoffLoader {
    static constexpr bool kStreams = false;
    const void* __restrict__ raw;   // start of this coherent block
    int data_type, precision, coh_ms;
    int n_ms;                       // samples per ms
    double f_hz, fs_hz;
    float mean_i, mean_q;
    template <int Q>
    GNSS_HD void load(int a, int b, cf (&z)[Q]) const {
        static_for<0, Q>([&](auto c_) {
            constexpr int C = decltype(c_)::value;
            const int n = Geo<Q>::good(a, b, C);
            float ax = 0.f, ay = 0.f;
            if (n < n_ms) {
                for (int j = 0; j < coh_ms; ++j) {
                    const long long idx = (long long)j * n_ms + n;
                    float xi, xq;
                    if (precision == 2) {
                        const int16_t* p = (const int16_t*)raw;
                        xi = (float)p[2 * idx] - mean_i;
                        xq = (float)p[2 * idx + 1] - mean_q;
                    } else if (data_type == 2) {
                        const int8_t* p = (const int8_t*)raw;
                        xi = (float)p[2 * idx];
                        xq = (float)p[2 * idx + 1];
                    } else {
                        xi = (float)((const int8_t*)raw)[idx];
                        xq = 0.f;
                    }
                    float co, si;
                    carrier_sincos(f_hz, fs_hz, idx + 1, co, si);
                    ax += xi * co - xq * si;
                    ay += xi * si + xq * co;
                }
            }
            z[C] = mk(ax, ay);
        });
    }
};

// Bluestein stage 1: a[n] = x[n] * conj(ch[n]) for n < n, zero beyond.  `Src` gives x[n] through sample(n).
struct NaturalSource {
    const cf* __restrict__ in;
    GNSS_HD cf sample(int n) const { return in[n]; }
};
template <class Src>
struct ChirpLoader {
    static constexpr bool kStreams = false;
    Src src;
    const cf* __restrict__ chirp;
    int n;
    template <int Q>
    GNSS_HD void load(int a, int b, cf (&z)[Q]) const {
        static_for<0, Q>([&](auto c_) {
            constexpr int C = decltype(c_)::value;
            const int m = Geo<Q>::good(a, b, C);
            if (m < n) {
                const cf v = src.sample(m), c = chirp[m];
                z[C] = mk(v.x * c.x + v.y * c.y, v.y * c.x - v.x * c.y);       // v * conj(c)
            } else {
                z[C] = mk(0.f, 0.f);
            }
        });
    }
};
// Bluestein stage 2 input: conj(FFT(a) * H)
struct ConjProdLoader {
    static constexpr bool kStreams = false;
    const cf* __restrict__ v;
    const cf* __restrict__ filt;
    template <int Q>
    GNSS_HD void load(int a, int b, cf (&z)[Q]) const {
        static_for<0, Q>([&](auto c_) {
            constexpr int C = decltype(c_)::value;
            const int m = Geo<Q>::good(a, b, C);
            const cf p = cmul_scalar(v[m], filt[m]);
            z[C] = mk(p.x, -p.y);
        });
    }
};
// Bluestein stage 2 output W: X[k] = conj(ch[k] * W[k]) / N' for k < n, natural order; k >= n is dropped
struct ChirpStorer {
    cf* __restrict__ out;
    const cf* __restrict__ chirp;
    int n;
    float scale;                    // 1 / N'
    GNSS_HD void put(int k, cf w) {
        if (k < n) {
            const cf p = cmul_scalar(chirp[k], w);
            out[k] = mk(p.x * scale, -p.y * scale);
        }
    }
    template <int Q, int R>
    GNSS_HD void store2(int col, int, const cf (&w0)[16], const cf (&w1)[16]) {
        static_for<0, 16>([&](auto i_) {
            constexpr int I = decltype(i_)::value;
            constexpr int AP = (I / 4) + 4 * (I % 4);
            put(Geo<Q>::lag_of(AP, col), w0[I]);
            if (col + 1 < Geo<Q>::ROW) put(Geo<Q>::lag_of(AP, col + 1), w1[I]);
        });
    }
};

// natural-order store: out[frequency index] (used by the fine stage and the FFT test hook)
struct NaturalStorerHD {
    cf* __restrict__ out;
    template <int Q, int R>
    GNSS_HD void store2(int col, int, const cf (&w0)[16], const cf (&w1)[16]) {
        static_for<0, 16>([&](auto i_) {
            constexpr int I = decltype(i_)::value;
            constexpr int AP = (I / 4) + 4 * (I % 4);
            out[Geo<Q>::lag_of(AP, col)] = w0[I];
            if (col + 1 < Geo<Q>::ROW) out[Geo<Q>::lag_of(AP, col + 1)] = w1[I];
        });
    }
};

// ================================================================== row-end helpers
struct RowPeak {
    float peak;        // max accumulated power
    int lag;           // first lag attaining it
};
GNSS_HD bool peak_better(float v, int m, float bv, int bm) { return v > bv || (v == bv && m < bm); }

}  // namespace gnss
