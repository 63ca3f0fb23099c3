// gnss_kernels.cuh -- sm_100a kernels around the engine passes (gnss_engine.h).
//
//   code_kernel    K0  fft(code replica) -> conj(.)/N, G layout          (acquisition.m:58, once per handle)
//   wipe_kernel    K1  wipe-off (+ M-ms fold) + forward FFT per (base, block)   (acquisition.m:56-57)
//   search_kernel  K2  per (PRN, bin) row: for each of the K blocks multiply the two spectra in the
//                      load stage, transform, |.|^2, accumulate on chip; then K3 = row peak, first-index
//                      argmax, sum of squares and windowed sum of squares   (acquisition.m:59,62-63,67)
//   natural_kernel     plain forward DFT (test hook)
//   wipe_pad_kernel, chirp_*_kernel   K1 and the Bluestein N-point DFTs of a shape zero-padded into the transform
//
// One transform = one thread-block cluster of R CTAs; each CTA keeps 16/R rows of the
// [16][Q][125] prime-factor array in shared memory, pass 4 pulls the other CTAs' rows through
// distributed shared memory (cluster.map_shared_rank).  The non-coherent accumulator of a row
// (N floats) lives in shared memory, split over the cluster, for the whole K loop: HBM/L2 only
// ever sees the two input spectra and one 24-byte candidate per row.
#pragma once
#include <cooperative_groups.h>
#include <climits>
#include "gnss_internal.h"

namespace gnss {
namespace cg = cooperative_groups;

struct NaturalLoader {
    static constexpr bool kStreams = false;
    const cf* __restrict__ in;
    template <int Q>
    __device__ __forceinline__ void load(int a, int b, cf (&z)[Q]) const {
        static_for<0, Q>([&](auto c_) {
            constexpr int C = decltype(c_)::value;
            z[C] = in[Geo<Q>::good(a, b, C)];
        });
    }
};
struct NaturalStorer {
    cf* __restrict__ out;
    template <int Q, int R>
    __device__ __forceinline__ void store2(int col, int, const cf (&w0)[16], const cf (&w1)[16]) {
        static_for<0, 16>([&](auto i_) {
            constexpr int I = decltype(i_)::value;
            constexpr int AP = (I / 4) + 4 * (I % 4);
            out[Geo<Q>::lag_of(AP, col)] = w0[I];
            if (col + 1 < Geo<Q>::ROW) out[Geo<Q>::lag_of(AP, col + 1)] = w1[I];
        });
    }
};

// cluster barrier halves (barrier.cluster): arrive = "I am done with the others' shared memory",
// wait = "everybody has arrived".  Splitting them lets pass 1's loads and DFT-Q run in the shadow.
template <int R>
__device__ __forceinline__ void cl_arrive() {
    if constexpr (R > 1) asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
}
template <int R>
__device__ __forceinline__ void cl_wait() {
    if constexpr (R > 1) asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
    else __syncthreads();
}
template <int R>
__device__ __forceinline__ void cl_sync() {
    cl_arrive<R>();
    cl_wait<R>();
}

template <int Q, int R, int T>
__device__ __forceinline__ void pass2_all(cf* D, const Tw4* tw, int tid) {
    pass2_cta<Q, R, T>(tid, D, tw);
}

// pass 3 over the CTA.  (A 5-lanes-per-task cooperative form for the few leftover tasks -- P3_TASKS is
// just above the thread count -- was measured in r01 and LOST 8 %: its address arithmetic raised the
// register pressure of the surrounding code, which sits at the 128-register limit.  Plain rounds it is.)
template <int Q, int R, int T>
__device__ __forceinline__ void pass3_all(cf* D, const Tw4* tw, int tid) {
    using S = Split<Q, R>;
    (void)tw;
    for (int t = tid; t < S::P3_TASKS; t += T) pass3_task<Q, R>(t, D);
}

struct RedScratch {
    float wv[32];
    int wm[32];
    double ws[32];
    // this CTA's slot, read by the other CTAs of the cluster
    float peak; int lag; double sum_all; double sum_win;
    // cluster-wide winner, broadcast inside the CTA
    float g_peak; int g_lag;
};

template <int Q, int R>
struct Smem {
    using S = Split<Q, R>;
    static constexpr size_t d_bytes = (size_t)S::D_ELEMS * sizeof(cf);
    static constexpr size_t acc_floats = S::ACC_ELEMS > SplitX<Q, R>::ACC_ELEMS ? S::ACC_ELEMS : SplitX<Q, R>::ACC_ELEMS;
    static constexpr size_t acc_bytes = acc_floats * sizeof(float);
    static constexpr size_t tw_bytes = 100 * sizeof(Tw4);
    static constexpr size_t red_bytes = ((sizeof(RedScratch) + 15) / 16) * 16;
    static constexpr size_t transform = d_bytes + tw_bytes;
    static constexpr size_t search = d_bytes + acc_bytes + tw_bytes + red_bytes;
};

__device__ __forceinline__ void fill_tw125(Tw4* tw, int tid, int T) {
    for (int j = tid; j < 100; j += T) {          // entry j = b2*4 + (k1-1): W125^(b2*k1)
        double s, c;
        sincospi(-2.0 * (double)((j >> 2) * ((j & 3) + 1)) / 125.0, &s, &c);
        Tw4 w;
        w.c = (float)c; w.pad = 0.f; w.ns = -(float)s; w.s = (float)s;
        tw[j] = w;
    }
}

// (value, first index) max + double sum over the CTA; result valid in thread 0.
template <int T>
__device__ __forceinline__ void block_reduce(float& v, int& m, double& s, RedScratch* rs) {
    constexpr unsigned full = 0xffffffffu;
    constexpr int NW = T / 32;
#pragma unroll
    for (int off = 16; off; off >>= 1) {
        const float ov = __shfl_down_sync(full, v, off);
        const int om = __shfl_down_sync(full, m, off);
        const double os = __shfl_down_sync(full, s, off);
        if (peak_better(ov, om, v, m)) { v = ov; m = om; }
        s += os;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { rs->wv[warp] = v; rs->wm[warp] = m; rs->ws[warp] = s; }
    __syncthreads();
    if (warp == 0) {
        v = lane < NW ? rs->wv[lane] : -1.f;
        m = lane < NW ? rs->wm[lane] : INT_MAX;
        s = lane < NW ? rs->ws[lane] : 0.0;
#pragma unroll
        for (int off = 16; off; off >>= 1) {
            const float ov = __shfl_down_sync(full, v, off);
            const int om = __shfl_down_sync(full, m, off);
            const double os = __shfl_down_sync(full, s, off);
            if (peak_better(ov, om, v, m)) { v = ov; m = om; }
            s += os;
        }
    }
    __syncthreads();
}

// passes 1-4 of one transform; cluster-wide barriers around the DSMEM pass
template <int Q, int R, int T, class Loader, class Storer>
__device__ __forceinline__ void unit_device(const Loader& ld, Storer& st, cf* D, cf* const* Dall,
                                            const Tw4* tw, int rank, int tid) {
    using S = Split<Q, R>;
    for (int t = tid; t < S::P1_TASKS; t += T) pass1_task<Q, R>(t, rank, ld, D);
    __syncthreads();
    pass2_all<Q, R, T>(D, tw, tid);
    __syncthreads();
    pass3_all<Q, R, T>(D, tw, tid);
    cl_sync<R>();
    for (int t = tid; t < S::P4_TASKS; t += T) pass4_task<Q, R>(t, rank, Dall, st);
    cl_sync<R>();
}

// Same, for the K-block loop of the search: the barrier that protects D from being overwritten while
// other CTAs still read it (end of pass 4) is split -- arrive right after pass 4, wait only when
// pass 1 of the NEXT unit has its DFT-Q results in registers and wants to store them.
// Precondition: one cl_arrive() is pending on entry; postcondition: one is pending on exit.
template <int Q, int R, int T, class Loader, class Storer>
__device__ __forceinline__ void unit_device_pipelined(const Loader& ld, Storer& st, cf* D, cf* const* Dall,
                                                      const Tw4* tw, int rank, int tid) {
    using S = Split<Q, R>;
    {
        cf z[Q];
        const bool has = tid < S::P1_TASKS;
        if (has) pass1_compute<Q, R>(tid, rank, ld, z);
        cl_wait<R>();
        if (has) pass1_store<Q, R>(tid, z, D);
    }
    for (int t = tid + T; t < S::P1_TASKS; t += T) pass1_task<Q, R>(t, rank, ld, D);
    __syncthreads();
    pass2_all<Q, R, T>(D, tw, tid);
    __syncthreads();
    pass3_all<Q, R, T>(D, tw, tid);
    cl_sync<R>();
    for (int t = tid; t < S::P4_TASKS; t += T) pass4_task<Q, R>(t, rank, Dall, st);
    cl_arrive<R>();
}

#define GNSS_KERNEL_PROLOGUE                                                     \
    using S = Split<Q, R>;                                                       \
    using G = Geo<Q>;                                                            \
    (void)sizeof(G);                                                             \
    cg::cluster_group cluster = cg::this_cluster();                              \
    const int tid = threadIdx.x;                                                 \
    const int rank = (R > 1) ? (int)cluster.block_rank() : 0;                    \
    const int unit = blockIdx.x / R;                                             \
    extern __shared__ __align__(16) unsigned char smem_raw[];                    \
    cf* D = reinterpret_cast<cf*>(smem_raw);                                     \
    cf* Dall[R];                                                                 \
    _Pragma("unroll") for (int r = 0; r < R; ++r)                                \
        Dall[r] = (R > 1) ? cluster.map_shared_rank(D, r) : D;

template <int Q, int R, int T, int MINB>
__global__ void __launch_bounds__(T, MINB) code_kernel(CodeArgs a) {
    GNSS_KERNEL_PROLOGUE
    Tw4* tw = reinterpret_cast<Tw4*>(D + S::D_ELEMS);
    fill_tw125(tw, tid, T);
    __syncthreads();
    CodeLoader ld{a.scode + (size_t)unit * G::N};
    SpectrumStorer st{a.cc + (size_t)unit * G::N, 1.0f / (float)G::N, 1, 0};
    unit_device<Q, R, T>(ld, st, D, Dall, tw, rank, tid);
}

template <int Q, int R, int T, int MINB>
__global__ void __launch_bounds__(T, MINB) wipe_kernel(WipeArgs a) {
    GNSS_KERNEL_PROLOGUE
    Tw4* tw = reinterpret_cast<Tw4*>(D + S::D_ELEMS);
    fill_tw125(tw, tid, T);
    __syncthreads();
    const int base = unit / a.K, k = unit - base * a.K;
    WipeoffLoader ld;
    ld.raw = (const unsigned char*)a.raw + (size_t)k * a.block_bytes;
    ld.data_type = a.data_type;
    ld.precision = a.precision;
    ld.coh_ms = a.coh_ms;
    ld.f_hz = a.base_freq_hz[base];
    ld.fs_hz = a.fs_hz;
    ld.mean_i = a.means ? (float)a.means[0] : 0.f;
    ld.mean_q = a.means ? (float)a.means[1] : 0.f;
    SpectrumStorer st{a.x + (size_t)unit * G::NX, 1.0f, 0, 1};
    unit_device<Q, R, T>(ld, st, D, Dall, tw, rank, tid);
}

// ---- K1 v2: wipe-off (+ M-ms fold) + forward FFT with cp.async-staged comb rows (acquisition.m:56-57) ----
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N_>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N_) : "memory"); }

// residue n mod 16 of every sample an a-row reads (M2 and M3 are multiples of 16)
template <int Q>
GNSS_HD int comb_row_of(int a) { return (a * (Geo<Q>::M1 % 16)) % 16; }

template <int Q, int R, int T, int MINB>
__global__ void __launch_bounds__(T, MINB) wipe2_kernel(Wipe2Args a) {
    GNSS_KERNEL_PROLOGUE
    Tw4* tw = reinterpret_cast<Tw4*>(D + S::D_ELEMS);
    unsigned char* stage = reinterpret_cast<unsigned char*>(tw + 100);          // [2 buffers][A rows][pitch]
    fill_tw125(tw, tid, T);
    const int base = unit / a.K, k = unit - base * a.K;
    const double w = a.base_w[base];
    const float mean_i = a.means ? (float)a.means[0] : 0.f, mean_q = a.means ? (float)a.means[1] : 0.f;
    const int pitch = a.pitch, bps = a.bps, M = a.coh_ms;
    // stage ms j of this coherent block: rows rho(a) of the CTA's A a-rows, 16-byte chunks, all threads
    auto stage_ms = [&](int j, int buf) {
        const int chunks = pitch >> 4;
        for (int i = tid; i < S::A * chunks; i += T) {
            const int al = i / chunks, ch = i - al * chunks;
            const int rho = comb_row_of<Q>(rank * S::A + al);
            const unsigned char* src = a.comb + ((size_t)((size_t)k * M + j) * 16 + rho) * pitch + (size_t)ch * 16;
            cp_async16(stage + ((size_t)buf * S::A + al) * pitch + (size_t)ch * 16, src);
        }
        cp_async_commit();
    };
    // steps s = round * M + j; step s reads buffer s & 1 while step s + 1 is being staged into the other one
    // (M == 1: a single buffer, staged once, serves every round)
    constexpr int ROUNDS = (S::P1_TASKS + T - 1) / T;
    const int n_steps = (M > 1) ? ROUNDS * M : 1;
    stage_ms(0, 0);
    int step = 0;
    for (int t0 = 0; t0 < S::P1_TASKS; t0 += T) {
        const int task = t0 + tid;
        const bool has = task < S::P1_TASKS;
        const int al = has ? task / 125 : 0, b = has ? task - al * 125 : 0;
        const int arow = rank * S::A + al;
        cf z[Q];
        static_for<0, Q>([&](auto c_) { z[decltype(c_)::value] = mk(0.f, 0.f); });
        for (int j = 0; j < M; ++j) {
            const int buf = (M > 1) ? (step & 1) : 0;
            if (M > 1 || t0 == 0) {
                if (step + 1 < n_steps) { stage_ms((j + 1) % M, buf ^ 1); cp_async_wait<1>(); }
                else cp_async_wait<0>();
                __syncthreads();                         // everybody's chunks of this step have landed
            }
            if (has) {
                const unsigned char* row = stage + ((size_t)buf * S::A + al) * pitch;
                static_for<0, Q>([&](auto c_) {
                    constexpr int C = decltype(c_)::value;
                    const int n = Geo<Q>::good(arow, b, C);
                    const int m = n >> 4;                 // position in the comb row (n = 16 m + rho)
                    float xi, xq;
                    if (bps == 2) {
                        const unsigned short v = *reinterpret_cast<const unsigned short*>(row + 2 * m);
                        xi = (float)(signed char)(v & 0xff);
                        xq = (float)(signed char)(v >> 8);
                    } else if (bps == 4) {
                        const unsigned v = *reinterpret_cast<const unsigned*>(row + 4 * m);
                        xi = (float)(short)(v & 0xffff) - mean_i;
                        xq = (float)(short)(v >> 16) - mean_q;
                    } else {
                        xi = (float)(signed char)row[m];
                        xq = 0.f;
                    }
                    // acquisition.m:43: exp(i*2*pi*f*n1/Fs), n1 = 1-based index inside the coherent block
                    const double cyc = w * (double)((long long)j * Geo<Q>::N + n + 1);
                    const float fr = (float)(cyc - floor(cyc));
                    float si, co;
                    sincospif(2.0f * fr, &si, &co);
                    z[C].x += xi * co - xq * si;
                    z[C].y += xi * si + xq * co;
                });
            }
            if (M > 1) __syncthreads();                  // this buffer is the target of the next-but-one staging
            ++step;
        }
        if (has) {
            dft_odd<Q>(z);
            pass1_store<Q, R>(task, z, D);
        }
    }
    cp_async_wait<0>();
    __syncthreads();
    pass2_all<Q, R, T>(D, tw, tid);
    __syncthreads();
    pass3_all<Q, R, T>(D, tw, tid);
    cl_sync<R>();
    SpectrumStorer st{a.x + (size_t)unit * G::NX, 1.0f, 0, 1};
    for (int t = tid; t < S::P4_TASKS; t += T) pass4_task<Q, R>(t, rank, Dall, st);
    cl_sync<R>();
}

template <int Q, int R, int T, int MINB>
__global__ void __launch_bounds__(T, MINB) natural_kernel(NaturalArgs a) {
    GNSS_KERNEL_PROLOGUE
    Tw4* tw = reinterpret_cast<Tw4*>(D + S::D_ELEMS);
    fill_tw125(tw, tid, T);
    __syncthreads();
    NaturalLoader ld{a.in + (size_t)unit * G::N};
    NaturalStorer st{a.out + (size_t)unit * G::N};
    unit_device<Q, R, T>(ld, st, D, Dall, tw, rank, tid);
}

// fine-frequency transforms: unit = ((sv * K) + r) * L + n2
template <int Q, int R, int T, int MINB>
__global__ void __launch_bounds__(T, MINB) fine_kernel(FineArgs a) {
    GNSS_KERNEL_PROLOGUE
    Tw4* tw = reinterpret_cast<Tw4*>(D + S::D_ELEMS);
    fill_tw125(tw, tid, T);
    __syncthreads();
    const int n2 = unit % a.L, r = (unit / a.L) % a.K, sv = unit / (a.L * a.K);
    FineLoader ld;
    ld.raw = a.raw;
    ld.chip = a.chip;
    ld.ca = a.ca + (size_t)sv * 1023;
    ld.data_type = a.data_type;
    ld.precision = a.precision;
    ld.mean_i = a.means ? (float)a.means[0] : 0.f;
    ld.mean_q = a.means ? (float)a.means[1] : 0.f;
    ld.start = a.start[sv];
    ld.L = a.L;
    ld.n2 = n2;
    ld.r = r;
    ld.F = a.F;
    NaturalStorerHD st{a.u + (size_t)unit * G::N};
    unit_device<Q, R, T>(ld, st, D, Dall, tw, rank, tid);
}

// ---- zero-padded shapes (samples per ms < N) ----
// K1 for a padded shape: wipe_kernel with the fold stride and the zero padding of PadWipeoffLoader
template <int Q, int R, int T, int MINB>
__global__ void __launch_bounds__(T, MINB) wipe_pad_kernel(WipeArgs a) {
    GNSS_KERNEL_PROLOGUE
    Tw4* tw = reinterpret_cast<Tw4*>(D + S::D_ELEMS);
    fill_tw125(tw, tid, T);
    __syncthreads();
    const int base = unit / a.K, k = unit - base * a.K;
    PadWipeoffLoader ld;
    ld.raw = (const unsigned char*)a.raw + (size_t)k * a.block_bytes;
    ld.data_type = a.data_type;
    ld.precision = a.precision;
    ld.coh_ms = a.coh_ms;
    ld.n_ms = a.n_ms;
    ld.f_hz = a.base_freq_hz[base];
    ld.fs_hz = a.fs_hz;
    ld.mean_i = a.means ? (float)a.means[0] : 0.f;
    ld.mean_q = a.means ? (float)a.means[1] : 0.f;
    SpectrumStorer st{a.x + (size_t)unit * G::NX, 1.0f, 0, 1};
    unit_device<Q, R, T>(ld, st, D, Dall, tw, rank, tid);
}

// Bluestein stage 1 of gnssacq_fft_forward: v[unit] = FFT_N(conj(ch) * in[unit], zero-padded)
template <int Q, int R, int T, int MINB>
__global__ void __launch_bounds__(T, MINB) chirp_in_kernel(ChirpArgs c) {
    GNSS_KERNEL_PROLOGUE
    Tw4* tw = reinterpret_cast<Tw4*>(D + S::D_ELEMS);
    fill_tw125(tw, tid, T);
    __syncthreads();
    ChirpLoader<NaturalSource> ld{NaturalSource{c.in + (size_t)unit * c.n}, c.chirp, c.n};
    NaturalStorerHD st{c.v + (size_t)unit * G::N};
    unit_device<Q, R, T>(ld, st, D, Dall, tw, rank, tid);
}

// Bluestein stage 1 of the fine stage: the samples of fine_kernel's unit ((sv * K) + r) * L + n2, chirped and padded
template <int Q, int R, int T, int MINB>
__global__ void __launch_bounds__(T, MINB) fine_chirp_kernel(FineArgs a, ChirpArgs c) {
    GNSS_KERNEL_PROLOGUE
    Tw4* tw = reinterpret_cast<Tw4*>(D + S::D_ELEMS);
    fill_tw125(tw, tid, T);
    __syncthreads();
    const int n2 = unit % a.L, r = (unit / a.L) % a.K, sv = unit / (a.L * a.K);
    FineLoader f;
    f.raw = a.raw;
    f.chip = a.chip;
    f.ca = a.ca + (size_t)sv * 1023;
    f.data_type = a.data_type;
    f.precision = a.precision;
    f.mean_i = a.means ? (float)a.means[0] : 0.f;
    f.mean_q = a.means ? (float)a.means[1] : 0.f;
    f.start = a.start[sv];
    f.L = a.L;
    f.n2 = n2;
    f.r = r;
    f.F = a.F;
    ChirpLoader<FineLoader> ld{f, c.chirp, c.n};
    NaturalStorerHD st{c.v + (size_t)unit * G::N};
    unit_device<Q, R, T>(ld, st, D, Dall, tw, rank, tid);
}

// Bluestein stage 2: out[unit] = conj(ch * FFT_N(conj(v[unit] * H))) / N, first n outputs
template <int Q, int R, int T, int MINB>
__global__ void __launch_bounds__(T, MINB) chirp_out_kernel(ChirpArgs c) {
    GNSS_KERNEL_PROLOGUE
    Tw4* tw = reinterpret_cast<Tw4*>(D + S::D_ELEMS);
    fill_tw125(tw, tid, T);
    __syncthreads();
    ConjProdLoader ld{c.v + (size_t)unit * G::N, c.filt};
    ChirpStorer st{c.out + (size_t)unit * c.n, c.chirp, c.n, 1.0f / (float)G::N};
    unit_device<Q, R, T>(ld, st, D, Dall, tw, rank, tid);
}

template <int Q, int R, int T, int MINB>
__global__ void __launch_bounds__(T, MINB) search_kernel(SearchArgs a) {
    GNSS_KERNEL_PROLOGUE
    float* acc = reinterpret_cast<float*>(D + S::D_ELEMS);
    Tw4* tw = reinterpret_cast<Tw4*>(acc + Smem<Q, R>::acc_floats);
    RedScratch* rs = reinterpret_cast<RedScratch*>(tw + 100);
    const int row = a.rows ? a.rows[unit] : a.row_first + unit;   // row = bin * P + prn_index (PRN fastest: rows in
    const int p = row % a.P, b = row / a.P;     // flight share the same forward spectra in L2)

    fill_tw125(tw, tid, T);
    for (int e = tid; e < S::ACC_ELEMS; e += T) acc[e] = 0.f;
    __syncthreads();

    int sa, sb, sc;
    G::shift_coords(a.bin_shift[b], sa, sb, sc);
    const cf* ccp = a.cc + (size_t)p * G::N;
    const cf* xb = a.x + (size_t)a.bin_base[b] * a.K * G::NX;
    PowerAccumStorer st{acc};
    cl_arrive<R>();
    for (int k = 0; k < a.K; ++k) {
        SearchLoader ld{ccp, xb + (size_t)k * G::NX, sa, sb, sc};
        unit_device_pipelined<Q, R, T>(ld, st, D, Dall, tw, rank, tid);
    }
    cl_wait<R>();

    // ---- K3: row peak (first index on ties), sum of squares, windowed sum of squares ----
    float bv = -1.f;
    int bm = INT_MAX;
    double ss = 0.0;
    for (int e = tid; e < S::ACC_ELEMS; e += T) {
        const int ap = e / S::CH, t = e - ap * S::CH;
        const int col = rank * S::CH + t;
        const int m = G::lag_of(ap, col);
        if (col < S::ROW && m < a.n_lags) {         // (m >= n_lags: zero padding of a padded shape)
            const float v = acc[e];
            if (peak_better(v, m, bv, bm)) { bv = v; bm = m; }
            ss += (double)v * (double)v;
            if (a.surface) a.surface[((size_t)p * a.B + b) * a.n_lags + m] = v;
        }
    }
    block_reduce<T>(bv, bm, ss, rs);
    if (tid == 0) { rs->peak = bv; rs->lag = bm; rs->sum_all = ss; }
    if constexpr (R > 1) cluster.sync(); else __syncthreads();
    if (tid == 0) {
        float gv = -1.f;
        int gm = INT_MAX;
        for (int r = 0; r < R; ++r) {
            const RedScratch* o = (R > 1) ? cluster.map_shared_rank(rs, r) : rs;
            const float ov = o->peak;
            const int om = o->lag;
            if (peak_better(ov, om, gv, gm)) { gv = ov; gm = om; }
        }
        rs->g_peak = gv;
        rs->g_lag = gm;
    }
    __syncthreads();
    const int gm = rs->g_lag;
    double wsum = 0.0;
    for (int i = tid; i < 2 * a.w - 1; i += T) {
        const int m = gm - (a.w - 1) + i;
        if (m >= 0 && m < a.n_lags) {
            int ap, col;
            G::cell_of_lag(m, ap, col);
            if (col / S::CH == rank) {
                const float v = acc[ap * S::CH + (col - rank * S::CH)];
                wsum += (double)v * (double)v;
            }
        }
    }
    float dv = -1.f;
    int dm = INT_MAX;
    block_reduce<T>(dv, dm, wsum, rs);
    if (tid == 0) rs->sum_win = wsum;
    if constexpr (R > 1) cluster.sync(); else __syncthreads();
    if (rank == 0 && tid == 0) {
        double s_all = 0.0, s_win = 0.0;
        for (int r = 0; r < R; ++r) {
            const RedScratch* o = (R > 1) ? cluster.map_shared_rank(rs, r) : rs;
            s_all += o->sum_all;
            s_win += o->sum_win;
        }
        Candidate c;
        c.peak = rs->g_peak;
        c.lag = rs->g_lag;
        c.sum_all = s_all;
        c.sum_win = s_win;
        a.cand[(size_t)p * a.cand_stride + b] = c;
    }
    if constexpr (R > 1) cluster.sync();   // keep every CTA's shared memory alive until rank 0 has read it
}

// K2, L2-exchange variant.  Pass 4 needs every CTA's finished rows; pulling them through DSMEM is
// bandwidth bound (~10 B/clk/SM each way, ncu r01b: 33 % of the kernel).  Here each CTA copies its
// finished rows (coalesced 16-B stores) into a double-buffered exchange array that stays L2-resident,
// signals the cluster barrier, runs pass 1 of the NEXT block while the barrier and the stores drain,
// and only then waits and runs pass 4 from L2.  D is private again, so only CTA-local barriers guard it.
// Persistent: gridDim.x / R clusters, each looping over rows; the cluster index selects the exchange slot.
template <int Q, int R, int T, int MINB>
__global__ void __launch_bounds__(T, MINB) search_kernel_l2x(SearchArgs a) {
    GNSS_KERNEL_PROLOGUE
    (void)Dall;
    float* acc = reinterpret_cast<float*>(D + S::D_ELEMS);
    Tw4* tw = reinterpret_cast<Tw4*>(acc + Smem<Q, R>::acc_floats);
    RedScratch* rs = reinterpret_cast<RedScratch*>(tw + 100);
    const int ncl = gridDim.x / R, slot = unit;
    cf* xch = a.scratch + (size_t)slot * 2 * 16 * S::RS;
    fill_tw125(tw, tid, T);
    PowerAccumStorer st{acc};

    for (int lrow = slot; lrow < a.n_rows; lrow += ncl) {
        const int row = a.rows ? a.rows[lrow] : a.row_first + lrow;
        const int p = row % a.P, b = row / a.P;
        for (int e = tid; e < S::ACC_ELEMS; e += T) acc[e] = 0.f;
        int sa, sb, sc;
        G::shift_coords(a.bin_shift[b], sa, sb, sc);
        const cf* ccp = a.cc + (size_t)p * G::N;
        const cf* xb = a.x + (size_t)a.bin_base[b] * a.K * G::NX;
        {
            SearchLoader ld{ccp, xb, sa, sb, sc};
            for (int t = tid; t < S::P1_TASKS; t += T) pass1_task<Q, R>(t, rank, ld, D);
        }
        __syncthreads();
        pass2_all<Q, R, T>(D, tw, tid);
        __syncthreads();
        pass3_all<Q, R, T>(D, tw, tid);
        // Software pipeline over the K blocks.  Per iteration: rows of block k leave for L2 (posted
        // stores), passes 1-2 of block k+1 run while they drain and while the other CTAs catch up,
        // then pass 4 of block k reads all 16 rows back from L2, then pass 3 of block k+1.
        for (int k = 0; k < a.K; ++k) {
            const bool more = k + 1 < a.K;
            cf* buf = xch + (size_t)(k & 1) * 16 * S::RS;
            __syncthreads();                           // pass 3 of block k complete in D
            {
                const float4* src = reinterpret_cast<const float4*>(D);
                float4* dst = reinterpret_cast<float4*>(buf + (size_t)rank * S::A * S::RS);
                for (int i = tid; i < S::D_ELEMS / 2; i += T) dst[i] = src[i];
            }
            if (more) {
                SearchLoader ld{ccp, xb + (size_t)(k + 1) * G::NX, sa, sb, sc};
                cf z[Q];
                const bool has = tid < S::P1_TASKS;
                if (has) pass1_compute<Q, R>(tid, rank, ld, z);
                __syncthreads();                       // every thread has finished copying D out
                if (has) pass1_store<Q, R>(tid, z, D);
                for (int t = tid + T; t < S::P1_TASKS; t += T) pass1_task<Q, R>(t, rank, ld, D);
            }
            cl_arrive<R>();                            // release: my rows of block k are in L2 by now
            if (more) {
                __syncthreads();
                pass2_all<Q, R, T>(D, tw, tid);
            }
            cl_wait<R>();                              // acquire: everybody's rows of block k
            for (int t = tid; t < S::P4_TASKS; t += T) pass4_task_flat<Q, R>(t, rank, buf, st);
            if (more) {
                __syncthreads();
                pass3_all<Q, R, T>(D, tw, tid);
            }
        }
        __syncthreads();

        // ---- K3 (identical to search_kernel) ----
        float bv = -1.f;
        int bm = INT_MAX;
        double ss = 0.0;
        for (int e = tid; e < S::ACC_ELEMS; e += T) {
            const int ap = e / S::CH, t = e - ap * S::CH;
            const int col = rank * S::CH + t;
            const int m = G::lag_of(ap, col);
            if (col < S::ROW && m < a.n_lags) {         // (m >= n_lags: zero padding of a padded shape)
                const float v = acc[e];
                if (peak_better(v, m, bv, bm)) { bv = v; bm = m; }
                ss += (double)v * (double)v;
                if (a.surface) a.surface[((size_t)p * a.B + b) * a.n_lags + m] = v;
            }
        }
        block_reduce<T>(bv, bm, ss, rs);
        if (tid == 0) { rs->peak = bv; rs->lag = bm; rs->sum_all = ss; }
        if constexpr (R > 1) cluster.sync(); else __syncthreads();
        if (tid == 0) {
            float gv = -1.f;
            int gm = INT_MAX;
            for (int r = 0; r < R; ++r) {
                const RedScratch* o = (R > 1) ? cluster.map_shared_rank(rs, r) : rs;
                const float ov = o->peak;
                const int om = o->lag;
                if (peak_better(ov, om, gv, gm)) { gv = ov; gm = om; }
            }
            rs->g_peak = gv;
            rs->g_lag = gm;
        }
        __syncthreads();
        const int gm = rs->g_lag;
        double wsum = 0.0;
        for (int i = tid; i < 2 * a.w - 1; i += T) {
            const int m = gm - (a.w - 1) + i;
            if (m >= 0 && m < a.n_lags) {
                int ap, col;
                G::cell_of_lag(m, ap, col);
                if (col / S::CH == rank) {
                    const float v = acc[ap * S::CH + (col - rank * S::CH)];
                    wsum += (double)v * (double)v;
                }
            }
        }
        float dv = -1.f;
        int dm = INT_MAX;
        block_reduce<T>(dv, dm, wsum, rs);
        if (tid == 0) rs->sum_win = wsum;
        if constexpr (R > 1) cluster.sync(); else __syncthreads();
        if (rank == 0 && tid == 0) {
            double s_all = 0.0, s_win = 0.0;
            for (int r = 0; r < R; ++r) {
                const RedScratch* o = (R > 1) ? cluster.map_shared_rank(rs, r) : rs;
                s_all += o->sum_all;
                s_win += o->sum_win;
            }
            Candidate c;
            c.peak = rs->g_peak;
            c.lag = rs->g_lag;
            c.sum_all = s_all;
            c.sum_win = s_win;
            a.cand[(size_t)p * a.cand_stride + b] = c;
        }
        if constexpr (R > 1) cluster.sync(); else __syncthreads();   // slots are rewritten by the next row
    }
}

// K2, cooperative variant: no thread-block clusters at all.  A transform is shared by a GROUP of R
// consecutive CTAs of a cooperative (all-co-resident) persistent grid; rows are exchanged through the
// L2-resident buffer exactly as in search_kernel_l2x, and the group barrier is an arrival counter in
// global memory (one red.release by thread 0 after the CTA barrier, one ld.acquire spin by thread 0
// before it).  Gains over the cluster kernels: every SM is usable (4-CTA clusters leave 16 of 148 SMs
// idle, ncu r01: 33 clusters resident), and only one thread pays the release fence.
__device__ __forceinline__ void group_arrive(unsigned* ctr) {
#ifdef GNSS_EXPERIMENT_NOFENCE   // timing only: results invalid
    asm volatile("red.relaxed.gpu.global.add.u32 [%0], 1;" ::"l"(ctr) : "memory");
#else
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ctr) : "memory");
#endif
}
__device__ __forceinline__ void group_arrive_n(unsigned* ctr, unsigned n) {
    asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(ctr), "r"(n) : "memory");
}
__device__ __forceinline__ void group_spin(const unsigned* ctr, unsigned target) {
    // acquire polls.  (Relaxed polls + one acquire fence, with and without __nanosleep back-off, were
    // measured in r01 and were 1-2 % slower: the slower acquire poll is its own back-off.)
    unsigned v;
    do {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory");
    } while ((int)(v - target) < 0);
}

// Tail hand-over helpers of the cooperative kernel (cold: kept out of line so that the K loop's code and
// register allocation stay what they are without them).
template <int Q, int R, int T>
__device__ __noinline__ void publish_plane(float* acc, float* dst, int tid) {
    using SX = SplitX<Q, R>;
    for (int j = tid; j < SX::P4_TASKS; j += T) {
#pragma unroll
        for (int ap = 0; ap < 16; ++ap) {
            float2* p = reinterpret_cast<float2*>(acc + ap * SX::CHX + 2 * j);
            __stcg(reinterpret_cast<float2*>(dst + ap * SX::CHX + 2 * j), *p);
            *p = make_float2(0.f, 0.f);
        }
    }
}
template <int Q, int R, int T>
__device__ __noinline__ void merge_planes(float* acc, const float* planes, int n_planes, int tid) {
    constexpr int ACC4 = SplitX<Q, R>::ACC_ELEMS / 4;
    const float4* src = reinterpret_cast<const float4*>(planes);
    float4* a4 = reinterpret_cast<float4*>(acc);
    int q = tid;
    for (; q + T < ACC4; q += 2 * T) {             // two cells' chains at once: twice the loads in flight
        float4 v = a4[q], w = a4[q + T];
#pragma unroll 4
        for (int k = 0; k < n_planes; ++k) {
            const float4 o = __ldcg(src + (size_t)k * (R * ACC4) + q);
            const float4 u = __ldcg(src + (size_t)k * (R * ACC4) + q + T);
            v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
            w.x += u.x; w.y += u.y; w.z += u.z; w.w += u.w;
        }
        a4[q] = v;
        a4[q + T] = w;
    }
    for (; q < ACC4; q += T) {
        float4 v = a4[q];
#pragma unroll 8
        for (int k = 0; k < n_planes; ++k) {
            const float4 o = __ldcg(src + (size_t)k * (R * ACC4) + q);
            v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
        }
        a4[q] = v;
    }
}

// The software pipeline runs ACROSS row boundaries: passes 1-3 of the next row's first block overlap the
// exchange of this row's last block (a per-row pipeline idles 0.6 of a block time per row: nothing at
// K = 20 blocks per row, 10 % at K = 2 -- BASELINE config 5 has 64 032 rows of 2 blocks).
// Timing-only switches (results invalid by construction, never defined in the product build):
// GNSS_EXPERIMENT_NOSPIN skips the group barrier wait, GNSS_EXPERIMENT_NOBAR also every CTA barrier of
// the loop; r01 measured 3.13 / 7.52 ms and 3.01 / 7.55 ms with them: all synchronisation costs 6-9 %.
#ifdef GNSS_EXPERIMENT_NOBAR
#define GNSS_KSYNC() __syncwarp()
#else
#define GNSS_KSYNC() __syncthreads()
#endif
#ifdef GNSS_TIMELINE
#define GNSS_TL(i) do { if (tl_iter == 6 && group == 0 && (tid & 31) == 0) a.timeline[(rank * (T / 32) + (tid >> 5)) * 32 + (i)] = clock64(); } while (0)
#else
#define GNSS_TL(i) do { } while (0)
#endif
template <int Q, int R, int T, int MINB>
__global__ void __launch_bounds__(T, MINB) search_kernel_coop(SearchArgs a) {
    using S = Split<Q, R>;
    using G = Geo<Q>;
    using GX = GeoX<Q>;
    using SX = SplitX<Q, R>;
    const int tid = threadIdx.x;
    // The task counts of passes 2 and 3 are not multiples of the CTA size, so some warp runs one extra
    // round in each; warp 0 also pays the release fence of the group barrier.  Rotating the thread index
    // per pass hands the extra rounds to different warps (ncu r01k: warp 0 was the straggler of every phase).
    // (Per-warp release + arrive right after pass 3 instead of one cumulative release was measured: +1-3 %.)
    const int tid2 = (tid + T - 32) % T;          // pass 2: last warp first
    const int tid3 = (tid + T - (64 % T)) % T;    // pass 3: second-to-last warp first
    const int rank = blockIdx.x % R, group = blockIdx.x / R, ngroups = gridDim.x / R;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cf* D = reinterpret_cast<cf*>(smem_raw);
    float* acc = reinterpret_cast<float*>(D + S::D_ELEMS);                 // [16][CHX] (XT layout)
    Tw4* tw = reinterpret_cast<Tw4*>(acc + Smem<Q, R>::acc_floats);
    RedScratch* rs = reinterpret_cast<RedScratch*>(tw + 100);
    constexpr size_t XBUF = (size_t)16 * GX::RSX;                          // cf per exchange buffer
    cf* xch = a.scratch + (size_t)group * 2 * XBUF;
    unsigned* ctr = a.group_ctr + group;
    Candidate* slots = a.row_slots + (size_t)group * R;
    unsigned target = 0;
    fill_tw125(tw, tid, T);
    // Register-resident accumulator (r02, VERDICT r01 item 2-ii): every variant has at most ONE pass-4 task per thread,
    // so its 2 x 16 accumulators can live in registers for all K blocks of a row; shared memory sees them once per row
    // (dump_acc before the row end) instead of a read-modify-write per block.  Used where the registers allow it:
    // Q = 13 compiles to 124 registers without spills (config 2: 2.946 -> 2.899 ms, same-box A/B, rows byte-identical);
    // at Q = 29 pass 1 already needs all 128 and the accumulators spill (6.82 -> 8.33 ms), so it keeps the shared-memory
    // accumulator (profiles/r02/ab_regacc_v15.txt).
    constexpr bool kRoomy = (T * MINB <= 512);            // 128 registers per thread available
    constexpr bool kRegAcc = (Q <= 13) && kRoomy && (SX::P4_TASKS <= T);
    float racc0[16], racc1[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) { racc0[q] = 0.f; racc1[q] = 0.f; }
    RegAccumStorer rst{racc0, racc1};
    PowerAccumStorer st{acc};
    // registers -> shared-memory accumulator (this thread's two columns), registers cleared
    auto dump_acc = [&]() {
        if constexpr (kRegAcc) {
            if (tid < SX::P4_TASKS) {
#pragma unroll
                for (int ap = 0; ap < 16; ++ap) {
                    *reinterpret_cast<float2*>(acc + ap * SX::CHX + 2 * tid) = make_float2(racc0[ap], racc1[ap]);
                    racc0[ap] = 0.f; racc1[ap] = 0.f;
                }
            }
        }
    };
    const int n_rows = a.n_rows;              // the launch's rows: a.rows[0 .. n_rows), or [row_first, row_first + n_rows)
    auto loader_of = [&](int lrow) {          // loader of block 0 of a row (two or three dependent table reads: once per row)
        const int row = a.rows ? a.rows[lrow] : a.row_first + lrow;
        const int p = row % a.P, b = row / a.P;
        int sa, sb, sc;
        G::shift_coords(a.bin_shift[b], sa, sb, sc);
        return SearchLoader{a.cc + (size_t)p * G::N, a.x + (size_t)a.bin_base[b] * a.K * G::NX, sa, sb, sc};
    };
    // Schedule.  floor(n_rows / ngroups) full rounds of whole rows, strided (row = round*ngroups + group: at
    // any time the groups work on neighbouring rows, i.e. on the same forward spectra -- contiguous row ranges
    // per group were measured 7 % slower at Q = 29).  The n_tail remaining rows are dealt out in units of one
    // block of one row, as contiguous ranges [tb(g), tb(g+1)) of u = tail_row*K + k, so every group gets the
    // same amount of the tail.  A tail row cut by a range boundary is finished by the group holding its first
    // block; the groups holding its later blocks publish each block's power plane in HBM and arrive on a
    // counter of the finishing group, which adds the planes in block order: the sum is bit-identical to an
    // uncut row's, so results do not depend on how many rows (PRNs) the handle has.  Publishing groups never
    // wait for anything, so nobody waits on a waiter.  row_granular: whole rows only (no planes needed).
    const int full = n_rows / ngroups, tail_base = full * ngroups, n_tail = n_rows - tail_base;
    auto tb = [&](int g) -> int {                  // 32-bit on purpose (a 64-bit division here costs the Q = 29 kernel
                                                   // 14 spilled registers); the host checks ngroups^2 * K < 2^32
        return a.row_granular ? (g < n_tail ? g : n_tail) * a.K : (int)((unsigned)g * (unsigned)(n_tail * a.K) / (unsigned)ngroups);
    };
    // The group's work as a list of row parts {row, first block, end block}: `full` whole rows, then the tail
    // range cut at its row boundary (it is at most K units long, so it touches at most two rows).  The loop
    // only carries the part index and the block counter; a part is looked up when it begins and when it ends.
    struct Part { int row, kb, ke; };
    auto part = [&](int i) -> Part {
        if (i < full) return Part{i * ngroups + group, 0, a.K};
        const int t0 = tb(group), t1 = tb(group + 1), r0 = t0 / a.K, e0 = min(t1, (r0 + 1) * a.K);
        if (i == full) return Part{tail_base + r0, t0 - r0 * a.K, e0 - r0 * a.K};
        return Part{tail_base + r0 + 1, 0, t1 - e0};
    };
    auto count_parts = [&]() -> int {
        const int t0 = tb(group), t1 = tb(group + 1);
        return full + (t0 < t1 ? 1 + (min(t1, (t0 / a.K + 1) * a.K) < t1) : 0);
    };
    if (count_parts() == 0) return;
    int i = 0, par = 0;
    const Part first = part(0);
    int left = first.ke - first.kb;                // blocks of part i still to do, this one included
    bool later = first.kb > 0;                     // part i continues a row that an earlier group finishes
    for (int e = tid; e < SX::ACC_ELEMS; e += T) acc[e] = 0.f;
    SearchLoader ld = loader_of(first.row);
    ld.x += (size_t)first.kb * G::NX;
    for (int t = tid; t < S::P1_TASKS; t += T) pass1_task<Q, R>(t, rank, ld, D);
    __syncthreads();
    pass2_all<Q, R, T>(D, tw, tid2);
    __syncthreads();
    // pass 3 leaves its results directly in the L2-resident exchange buffer (transposed "XT" layout: the 25
    // stores of a task are coalesced across the warp) -- no shared-memory write, no copy-out pass
    for (int t = tid3; t < S::P3_TASKS; t += T) pass3_task_xt<Q, R>(t, D, xch + (size_t)rank * S::A * GX::RSX);
#ifdef GNSS_TIMELINE
    int tl_iter = 0;
#endif
    for (;;) {
#ifdef GNSS_TIMELINE
        ++tl_iter;
#endif
        GNSS_TL(0);
        const bool last_of_part = (left == 1);
        const bool more = !last_of_part || i + 1 < count_parts();
        const cf* buf = xch + (size_t)par * XBUF;          // rows of the current block (all CTAs write into it)
        cf* nbuf = xch + (size_t)(par ^ 1) * XBUF;         // ... of the next block
        par ^= 1;
        target += R;
        if (more) {
            if (last_of_part) {
                const Part np = part(i + 1);
                ld = loader_of(np.row);
                ld.x += (size_t)np.kb * G::NX;
            } else {
                ld.x += G::NX;
            }
            cf z[Q];
            const bool has = tid < S::P1_TASKS;
            if (has) pass1_compute<Q, R>(tid, rank, ld, z);
            // A thread's SECOND pass-1 task (variants with two a-rows per CTA) is computed ahead of the barrier as well where
            // the registers allow it (Q = 13: 2 x 26): its loads and DFT-Q then overlap the other warps' pass 3 / pass 4
            // instead of sitting between the two barriers (config 2: 2.893 -> 2.848 ms, profiles/r02/ab_p1x2_v16.txt).
            constexpr bool kTwo = (Q <= 13) && kRoomy && (S::P1_TASKS > T) && (S::P1_TASKS <= 2 * T);
            cf z2[kTwo ? Q : 1];
            const bool has2 = kTwo && tid + T < S::P1_TASKS;
            if constexpr (kTwo) { if (has2) pass1_compute<Q, R>(tid + T, rank, ld, z2); }
            GNSS_TL(1);
            GNSS_KSYNC();                          // every thread is done with pass 3 of the current block
            GNSS_TL(2);
            if (tid == 0) group_arrive(ctr);       // release (cumulative over the CTA barrier): its rows are in L2
            GNSS_TL(3);
            if (has) pass1_store<Q, R>(tid, z, D);
            if constexpr (kTwo) {
                if (has2) pass1_store<Q, R>(tid + T, z2, D);
            } else if constexpr (S::P1_TASKS > T) {
                for (int t = tid + T; t < S::P1_TASKS; t += T) pass1_task<Q, R>(t, rank, ld, D);
            }
            GNSS_TL(4);
            GNSS_KSYNC();
            GNSS_TL(5);
            pass2_all<Q, R, T>(D, tw, tid2);
            GNSS_TL(6);
        } else {
            GNSS_KSYNC();
            if (tid == 0) group_arrive(ctr);
        }
#ifndef GNSS_EXPERIMENT_NOSPIN
        if (tid == 0) group_spin(ctr, target);     // acquire: everybody's rows of this block are in L2
#endif
        GNSS_TL(7);
        GNSS_KSYNC();
        GNSS_TL(8);
        // pass 4 of this block and pass 3 of the next share a barrier interval: the L2 latency of the
        // former hides under the arithmetic of the latter.  (Moving pass 3 in front of the group
        // barrier to add slack was measured in r01 and lost 3 %.)
        // The two are independent inside the interval, so half of the warps (1 and 2 of every four) run them in the
        // opposite order: while the others wait for pass 4's L2 loads these issue pass 3's arithmetic, and vice versa
        // (one copy of each body; the order is a runtime switch, not duplicated code).  Measured r02, same box:
        // 7.05 -> 6.87 ms / 3.09 -> 2.96 ms; warp parity or the upper half as the flipped set are within 1 % of it
        // (profiles/r02/ab_flip_v14.txt).  A CTA whose warps all sit in the same phase uses the FMA pipe and the
        // L1 data pipe in turns; the flip takes a little of that lockstep away.
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {
            const int flip = (((tid >> 5) + 1) >> 1) & 1;
            if ((half ^ flip) == 0) {
                if constexpr (kRegAcc) {
                    if (tid < SX::P4_TASKS) pass4_task_xt<Q, R>(tid, rank, buf, rst);
                } else {
                    for (int t = tid; t < SX::P4_TASKS; t += T) pass4_task_xt<Q, R>(t, rank, buf, st);
                }
            } else if (more) {
                for (int t = tid3; t < S::P3_TASKS; t += T) pass3_task_xt<Q, R>(t, D, nbuf + (size_t)rank * S::A * GX::RSX);
            }
        }
        GNSS_TL(10);
        if (later) {
            // A later part of a tail row that an earlier group finishes: publish this block's power plane on
            // its own (slot = block index in the row, in the finisher's slab), so that the finisher can add the
            // planes one by one in block order -- bit for bit the sum an uncut row gets.  Every thread moves
            // the columns its own pass-4 tasks accumulated (program order: no barrier) and re-zeroes them.
            const Part cp = part(i);
            const int kk = cp.ke - left;           // this block's index in its row
            int gf = group - 1;                    // the finisher: last group whose range starts at or before the row's
            while (tb(gf) > (cp.row - tail_base) * a.K) --gf;
            float* dst = a.partial + (((size_t)gf * (a.K - 1) + (kk - 1)) * R + rank) * SX::ACC_ELEMS;
            dump_acc();                            // (publish_plane moves the columns of the thread's own task: program order)
            publish_plane<Q, R, T>(acc, dst, tid);
            if (last_of_part) {
                __syncthreads();
                if (tid == 0) group_arrive_n(a.part_ctr + (size_t)gf * R + rank, (unsigned)(cp.ke - cp.kb));   // release
            }
        } else if (last_of_part) {
            dump_acc();
            __syncthreads();                       // this group's blocks of the row are in the accumulator
            const Part cp = part(i);
            const int row = cp.row;
            if (cp.ke < a.K) {
                // blocks cp.ke .. K-1 were done by the following groups: add their planes in block order
                if (tid == 0) group_spin(a.part_ctr + (size_t)group * R + rank, (unsigned)(a.K - cp.ke));
                __syncthreads();
                merge_planes<Q, R, T>(acc, a.partial + (((size_t)group * (a.K - 1) + (cp.ke - 1)) * R + rank) * SX::ACC_ELEMS,
                                      a.K - cp.ke, tid);
                __syncthreads();
            }
            const int grow = a.rows ? a.rows[row] : a.row_first + row, p = grow % a.P, b = grow / a.P;
            float bv = -1.f;
            int bm = INT_MAX;
            double ss = 0.0;
            if (a.surface || a.n_lags < G::N) {   // debug path and padded shapes: every cell's lag is needed
                for (int e = tid; e < SX::ACC_ELEMS; e += T) {
                    const int ap = e / SX::CHX, t = e - ap * SX::CHX;
                    const int ex = rank * SX::CHX + t;
                    if (GX::valid(ex)) {
                        const int m = GX::lag_of(ap, ex);
                        if (m < a.n_lags) {        // (m >= n_lags: zero padding of a padded shape)
                            const float v = acc[e];
                            if (peak_better(v, m, bv, bm)) { bv = v; bm = m; }
                            ss += (double)v * (double)v;
                            if (a.surface) a.surface[((size_t)p * a.B + b) * a.n_lags + m] = v;
                        }
                    }
                }
            } else {
                // The lag of a cell costs ~40 integer instructions (two divisions, a CRT): only compute it
                // for cells that can still win.  The padding columns hold exact zeros (their inputs are never
                // written: the exchange buffer is zero-initialised), so they need no validity test here --
                // a zero cell only matters when the whole row is zero, and then ties resolve by lag below.
                const float4* a4 = reinterpret_cast<const float4*>(acc);
                for (int q = tid; q < SX::ACC_ELEMS / 4; q += T) {
                    const float4 v = a4[q];
                    ss += (double)v.x * v.x + (double)v.y * v.y + (double)v.z * v.z + (double)v.w * v.w;
                    const float vm = fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w));
                    if (vm >= bv) {                // candidate (ties included): resolve exactly
                        const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            const int e = 4 * q + u;
                            const int ap = e / SX::CHX, t = e - ap * SX::CHX;
                            const int ex = rank * SX::CHX + t;
                            if (vv[u] >= bv && GX::valid(ex)) {
                                const int m = GX::lag_of(ap, ex);
                                if (peak_better(vv[u], m, bv, bm)) { bv = vv[u]; bm = m; }
                            }
                        }
                    }
                }
            }
            block_reduce<T>(bv, bm, ss, rs);
            target += R;
            if (tid == 0) {
                Candidate c; c.peak = bv; c.lag = bm; c.sum_all = ss; c.sum_win = 0.0;
                slots[rank] = c;
                group_arrive(ctr);
                group_spin(ctr, target);
                float gv = -1.f;
                int gm = INT_MAX;
                for (int r = 0; r < R; ++r) {
                    const float ov = __ldcg(&slots[r].peak);
                    const int om = __ldcg(&slots[r].lag);
                    if (peak_better(ov, om, gv, gm)) { gv = ov; gm = om; }
                }
                rs->g_peak = gv;
                rs->g_lag = gm;
            }
            __syncthreads();
            const int gm = rs->g_lag;
            double wsum = 0.0;
            for (int i = tid; i < 2 * a.w - 1; i += T) {
                const int m = gm - (a.w - 1) + i;
                if (m >= 0 && m < a.n_lags) {
                    int ap, ex;
                    GX::cell_of_lag(m, ap, ex);
                    if (ex / SX::CHX == rank) {
                        const float v = acc[ap * SX::CHX + (ex - rank * SX::CHX)];
                        wsum += (double)v * (double)v;
                    }
                }
            }
            float dv = -1.f;
            int dm = INT_MAX;
            block_reduce<T>(dv, dm, wsum, rs);
            // Every thread has read its window cells (block_reduce ends with a CTA barrier): the accumulator can be
            // cleared while thread 0 finishes the row.  No second group barrier: each CTA publishes its two partial sums
            // and takes a ticket (acq_rel); the LAST of the R CTAs to do so adds the partials IN RANK ORDER (bit-identical
            // whichever CTA that is) and writes the candidate.  Nobody waits for anybody here.  The slots are not touched
            // again before the next row end, and every block in between has a group barrier that the finisher joins
            // only after this.
            if constexpr (!kRegAcc)                // (register accumulators: every cell is overwritten by the next dump)
                for (int e = tid; e < SX::ACC_ELEMS; e += T) acc[e] = 0.f;
            if (tid == 0) {
                slots[rank].sum_win = wsum;
                unsigned old;
                asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;" : "=r"(old) : "l"(a.row_ticket + group) : "memory");
                if ((old + 1) % R == 0) {
                    double s_all = 0.0, s_win = 0.0;
                    for (int r = 0; r < R; ++r) {
                        s_all += __ldcg(&slots[r].sum_all);
                        s_win += __ldcg(&slots[r].sum_win);
                    }
                    Candidate c;
                    c.peak = rs->g_peak;
                    c.lag = rs->g_lag;
                    c.sum_all = s_all;
                    c.sum_win = s_win;
                    a.cand[(size_t)p * a.cand_stride + b] = c;
                }
            }
            // (the next write to acc is pass 4 of the next block, several CTA barriers away)
        }
        if (!more) break;
        if (last_of_part) {
            const Part np = part(++i);
            left = np.ke - np.kb;
            later = np.kb > 0;
        } else {
            --left;
        }
    }
}

// ------------------------------------------------------------------ launch glue
template <class K, class A>
static cudaError_t launch_clustered(K kern, const A& args, int units, int R, int T, size_t smem, cudaStream_t s) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(units * R), 1, 1);
    cfg.blockDim = dim3((unsigned)T, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)R;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    A copy = args;
    return cudaLaunchKernelEx(&cfg, kern, copy);
}

template <int Q, int R, int T, int MINB>
struct Variant {
    // K0 / K1 / fine / test transforms always use DSMEM clusters; the portable cluster limit is 8 CTAs, so a
    // 16-CTA search variant borrows the (8, 256) transform kernels (spectrum layouts do not depend on R).
    static constexpr int RT = R > 8 ? 8 : R;
    static constexpr int TT = R > 8 ? 256 : T;
    static constexpr int MT = R > 8 ? 2 : MINB;
    static cudaError_t prepare() {
        cudaError_t e;
        e = cudaFuncSetAttribute(code_kernel<Q, RT, TT, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<Q, RT>::transform);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(wipe_kernel<Q, RT, TT, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<Q, RT>::transform);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(wipe2_kernel<Q, RT, TT, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(natural_kernel<Q, RT, TT, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<Q, RT>::transform);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(fine_kernel<Q, RT, TT, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<Q, RT>::transform);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(wipe_pad_kernel<Q, RT, TT, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<Q, RT>::transform);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(chirp_in_kernel<Q, RT, TT, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<Q, RT>::transform);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(fine_chirp_kernel<Q, RT, TT, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<Q, RT>::transform);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(chirp_out_kernel<Q, RT, TT, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<Q, RT>::transform);
        if (e != cudaSuccess) return e;
        e = cudaFuncSetAttribute(search_kernel_coop<Q, R, T, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<Q, R>::search);
        if (e != cudaSuccess) return e;

        e = cudaFuncSetAttribute(search_kernel_l2x<Q, R, T, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<Q, R>::search);
        if (e != cudaSuccess) return e;
        return cudaFuncSetAttribute(search_kernel<Q, R, T, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Smem<Q, R>::search);
    }
    static cudaError_t launch_search_l2x(const SearchArgs& a, int clusters, cudaStream_t s) {
        if (R > 8) return cudaErrorInvalidConfiguration;
        return launch_clustered(search_kernel_l2x<Q, R, T, MINB>, a, clusters, R, T, Smem<Q, R>::search, s);
    }
    static cudaError_t launch_search_coop(const SearchArgs& a, int groups, cudaStream_t s) {
        SearchArgs copy = a;
        void* args[] = {&copy};
        return cudaLaunchCooperativeKernel((const void*)search_kernel_coop<Q, R, T, MINB>, dim3((unsigned)(groups * R)),
                                           dim3((unsigned)T), args, Smem<Q, R>::search, s);
    }
    static int max_groups_coop() {
        int per_sm = 0, dev = 0, sms = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, search_kernel_coop<Q, R, T, MINB>, T, Smem<Q, R>::search) != cudaSuccess) { cudaGetLastError(); return 0; }
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        return per_sm * sms / R;
    }
    static int max_clusters_l2x() {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(R * 1024), 1, 1);
        cfg.blockDim = dim3((unsigned)T, 1, 1);
        cfg.dynamicSmemBytes = Smem<Q, R>::search;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = (unsigned)R;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, search_kernel_l2x<Q, R, T, MINB>, &cfg) != cudaSuccess) { cudaGetLastError(); return 0; }
        return n;
    }
    static cudaError_t launch_code(const CodeArgs& a, int units, cudaStream_t s) {
        return launch_clustered(code_kernel<Q, RT, TT, MT>, a, units, RT, TT, Smem<Q, RT>::transform, s);
    }
    static cudaError_t launch_wipe(const WipeArgs& a, int units, cudaStream_t s) {
        return launch_clustered(wipe_kernel<Q, RT, TT, MT>, a, units, RT, TT, Smem<Q, RT>::transform, s);
    }
    static size_t smem_wipe2(int pitch, int coh_ms) {
        return Smem<Q, RT>::transform + (size_t)(coh_ms > 1 ? 2 : 1) * Split<Q, RT>::A * (size_t)pitch;
    }
    static cudaError_t launch_wipe2(const Wipe2Args& a, int units, cudaStream_t s) {
        return launch_clustered(wipe2_kernel<Q, RT, TT, MT>, a, units, RT, TT, smem_wipe2(a.pitch, a.coh_ms), s);
    }
    static cudaError_t launch_natural(const NaturalArgs& a, int units, cudaStream_t s) {
        return launch_clustered(natural_kernel<Q, RT, TT, MT>, a, units, RT, TT, Smem<Q, RT>::transform, s);
    }
    static cudaError_t launch_fine(const FineArgs& a, int units, cudaStream_t s) {
        return launch_clustered(fine_kernel<Q, RT, TT, MT>, a, units, RT, TT, Smem<Q, RT>::transform, s);
    }
    static cudaError_t launch_wipe_pad(const WipeArgs& a, int units, cudaStream_t s) {
        return launch_clustered(wipe_pad_kernel<Q, RT, TT, MT>, a, units, RT, TT, Smem<Q, RT>::transform, s);
    }
    static cudaError_t launch_chirp_in(const ChirpArgs& c, int units, cudaStream_t s) {
        return launch_clustered(chirp_in_kernel<Q, RT, TT, MT>, c, units, RT, TT, Smem<Q, RT>::transform, s);
    }
    static cudaError_t launch_fine_chirp(const FineArgs& a, const ChirpArgs& c, int units, cudaStream_t s) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(units * RT), 1, 1);
        cfg.blockDim = dim3((unsigned)TT, 1, 1);
        cfg.dynamicSmemBytes = Smem<Q, RT>::transform;
        cfg.stream = s;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = (unsigned)RT;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        FineArgs fa = a;
        ChirpArgs ca = c;
        return cudaLaunchKernelEx(&cfg, fine_chirp_kernel<Q, RT, TT, MT>, fa, ca);
    }
    static cudaError_t launch_chirp_out(const ChirpArgs& c, int units, cudaStream_t s) {
        return launch_clustered(chirp_out_kernel<Q, RT, TT, MT>, c, units, RT, TT, Smem<Q, RT>::transform, s);
    }
    static cudaError_t launch_search(const SearchArgs& a, int rows, cudaStream_t s) {
        if (R > 8) return cudaErrorInvalidConfiguration;       // DSMEM variant needs a portable cluster
        return launch_clustered(search_kernel<Q, R, T, MINB>, a, rows, R, T, Smem<Q, R>::search, s);
    }
    static constexpr VariantOps ops() {
        return VariantOps{Q, R, T, Smem<Q, R>::search, Smem<Q, RT>::transform,
                          &prepare, &launch_code, &launch_wipe, &launch_wipe2, &smem_wipe2, &launch_natural, &launch_fine, &launch_search,
                          &launch_search_l2x, &max_clusters_l2x,
                          (size_t)2 * 16 * (Split<Q, R>::RS > GeoX<Q>::RSX ? Split<Q, R>::RS : GeoX<Q>::RSX) * sizeof(cf),
                          &launch_search_coop, &max_groups_coop,
                          (size_t)R * SplitX<Q, R>::ACC_ELEMS * sizeof(float),
                          &launch_wipe_pad, &launch_chirp_in, &launch_fine_chirp, &launch_chirp_out};
    }
};

}  // namespace gnss
