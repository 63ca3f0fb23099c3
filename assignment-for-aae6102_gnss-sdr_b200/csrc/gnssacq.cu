// gnssacq.cu -- C-ABI host side of libgnssacq.so (include/gnssacq.h).
//
// Owns: config validation, the C/A code tables (generateCAcode.m, acquisition.m:50-51), the
// HBM-resident cache of conj(fft(code))/N, pinned IF staging, the Doppler-bin -> (base, shift)
// plan (SURVEY A.7), kernel sequencing on one stream, and K4 (per-PRN winner, noise floor, SNR,
// threshold: acquisition.m:62-70).  No CPU fallback: every numeric step of the search runs in the
// sm_100a kernels of gnss_kernels.cuh.
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <chrono>
#include <cstring>
#include <string>
#include <vector>
#include <cooperative_groups.h>
#if defined(__x86_64__)
#include <emmintrin.h>
#endif

#include "../../include/gnssacq.h"
#include "gnss_internal.h"

using namespace gnss;

#define GNSSACQ_VERSION_STR "gnssacq 0.2.0 (sm_100a)"

namespace {

thread_local std::string g_create_error;

// ---------------------------------------------------------------- C/A code (generateCAcode.m)
const int kG2Delay[51] = {5,   6,   7,   8,   17,  18,  139, 140, 141, 251, 252, 254, 255, 256, 257, 258, 469,
                          470, 471, 472, 473, 474, 509, 512, 513, 514, 515, 516, 859, 860, 861, 862, 145, 175,
                          52,  21,  237, 235, 886, 657, 634, 762, 355, 1012, 176, 603, 130, 359, 595, 68,  386};

// Bit form of the +-1 registers: value -1 <-> bit 1 (product of -1s == XOR of bits).
void ca_chips(int prn, int8_t* out) {
    uint8_t g1[1023], g2[1023];
    uint32_t r1 = 0x3ff, r2 = 0x3ff;   // stage k at bit (k-1); all ones == all -1 (generateCAcode.m:34,49)
    for (int i = 0; i < 1023; ++i) {
        g1[i] = (r1 >> 9) & 1;                                                    // output = stage 10
        g2[i] = (r2 >> 9) & 1;
        const uint32_t f1 = ((r1 >> 2) ^ (r1 >> 9)) & 1;                          // taps 3,10
        const uint32_t f2 = ((r2 >> 1) ^ (r2 >> 2) ^ (r2 >> 5) ^ (r2 >> 7) ^ (r2 >> 8) ^ (r2 >> 9)) & 1;   // 2,3,6,8,9,10
        r1 = ((r1 << 1) | f1) & 0x3ff;
        r2 = ((r2 << 1) | f2) & 0x3ff;
    }
    const int d = kG2Delay[prn - 1];
    for (int i = 0; i < 1023; ++i) {
        const uint8_t g2d = g2[(i + 1023 - d) % 1023];        // g2 rotated right by d (generateCAcode.m:61)
        // +-1 values: v = 1 - 2*bit ; CAcode = -(v1*v2) = -(1 - 2*(b1^b2))
        out[i] = (int8_t)((g1[i] ^ g2d) ? 1 : -1);
    }
}

// acquisition.m:50-51 -- scode(n) = [CA CA](ceil(n*(fc/Fs))), n = 1..N, ratio formed first, in double.
void code_replica(const gnssacq_config& c, int prn, int8_t* out) {
    int8_t ca[1023];
    ca_chips(prn, ca);
    const double ratio = c.code_hz / c.fs_hz;
    for (int n = 1; n <= c.samples_per_ms; ++n) {
        long idx = (long)std::ceil((double)n * ratio);    // 1-based into the doubled code
        if (idx < 1) idx = 1;
        out[n - 1] = ca[(idx - 1) % 1023];
    }
}

// ---------------------------------------------------------------- small kernels
// K4: acquisition.m:62-70 from the per-row candidates.
__global__ void finalize_kernel(const Candidate* __restrict__ cand, int P, int B, int N, int w, double fmin,
                                double fstep, double thr, const int* __restrict__ prn_ids,
                                gnssacq_result* __restrict__ out, int cand_stride, int bin0) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const Candidate* row = cand + (size_t)p * cand_stride;
    float g = -1.f;
    for (int b = 0; b < B; ++b) g = fmaxf(g, row[b].peak);
    int fbin = -1, cp = INT_MAX;
    for (int b = 0; b < B; ++b) {
        if (row[b].peak == g) {
            if (fbin < 0) fbin = b;                     // first bin attaining the maximum (:62)
            cp = min(cp, row[b].lag);                   // first code phase attaining it (:63)
        }
    }
    if (fbin < 0) { fbin = 0; cp = 0; }
    const Candidate c = row[fbin];
    const int cp1 = cp + 1;                             // MATLAB's 1-based codePhase
    const long long cnt = (long long)max(cp1 - w, 0) + (long long)max(N - cp1 - w + 1, 0);   // :67-68 index set
    const double noise = (c.sum_all - c.sum_win) / (double)cnt;
    const double pk = (double)g;
    // (g < 0: a row-range handle used alone that owns none of this PRN's rows -- nothing to report)
    const double snr = g < 0.f ? nan("") : 10.0 * log10(pk * pk / noise);
    gnssacq_result r;
    r.prn = prn_ids[p];
    r.acquired = (snr >= thr) ? 1 : 0;                  // :70 (NaN compares false)
    r.code_phase = cp;
    r.doppler_bin = bin0 + fbin;                        // index in the full grid (bin0 != 0: the handle owns a bin range)
    r.doppler_hz = fmin + fstep * (double)(bin0 + fbin);   // :64
    r.peak = pk;
    r.noise_meansq = noise;
    r.snr_db = snr;
    r.fine_freq_hz = nan("");
    out[p] = r;
}

// K1a (r02): re-order the raw IF block (acquisition.m:27-38's bytes, as read) into 16 comb rows per millisecond:
// out[ms][rho][m] = sample 16*m + rho of that ms (see Wipe2Args).  Input is read with 16-byte vector loads
// (8 packed int8 I/Q samples per load, fully coalesced) -- `raw` may be a PEER pointer: on ranks > 0 of a
// multi-GPU search this kernel is what pulls the IF block out of rank 0's HBM over NVLink, so no separate
// broadcast is needed.  Until the root's "IF ready" flag, which this kernel waits for, that buffer holds whatever it
// held before (the previous block, a half-finished upload), so nothing else on such a rank reads `raw`: the int16
// means are summed from the comb copy.  A CTA handles TM consecutive m of one ms (TM*16 samples, contiguous in the input).
constexpr int kCombTM = 256;
// Flags of the multi-GPU exchange live in the ROOT GPU's memory; other GPUs read / write them over NVLink.
__device__ __forceinline__ void flag_store_sys(unsigned* p, unsigned v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned flag_load_sys(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// spin until *p >= epoch (wrap-safe); gives up after ~4 s of GPU clock and records it in *timeout (never hangs a box)
__device__ __forceinline__ void flag_wait_sys(const unsigned* p, unsigned epoch, unsigned* timeout) {
    const long long t0 = clock64();
    while ((int)(flag_load_sys(p) - epoch) < 0) {
        if (clock64() - t0 > 8000000000ll) { if (timeout) atomicExch(timeout, 1u); break; }
        __nanosleep(200);
    }
}
__global__ void __launch_bounds__(256) comb_kernel(const unsigned char* __restrict__ raw, unsigned char* __restrict__ out,
                                                   int rows_per_ms /* N/16 */, int bps, int pitch, int tiles_per_ms,
                                                   unsigned* flag_publish, const unsigned* flag_wait, unsigned epoch,
                                                   unsigned* timeout) {
    extern __shared__ __align__(16) unsigned smem_w[];       // [TM][4*bps + 1] words (one pad word per m: conflict-free column reads)
    // multi-GPU: the root announces that its IF buffer holds this step's block (it does, by stream order);
    // every other shard waits for that before pulling the block out of the root's HBM
    if (flag_publish && blockIdx.x == 0 && threadIdx.x == 0) flag_store_sys(flag_publish, epoch);
    if (flag_wait) {
        if (threadIdx.x == 0) flag_wait_sys(flag_wait, epoch, timeout);
        __syncthreads();
    }
    const int ms = blockIdx.x / tiles_per_ms, tile = blockIdx.x - ms * tiles_per_ms;
    const int m0 = tile * kCombTM, tm = min(kCombTM, rows_per_ms - m0);
    const int W = 4 * bps;                                    // words per m (16 samples)
    const uint4* src = reinterpret_cast<const uint4*>(raw + ((size_t)ms * rows_per_ms + m0) * 16 * bps);
    const int n_vec = tm * bps;                               // uint4 per tile: tm * 16 * bps / 16
    for (int i = threadIdx.x; i < n_vec; i += blockDim.x) {
        const uint4 v = src[i];
        const int m = i / bps, part = i - m * bps;            // `bps` uint4 per m
        unsigned* d = smem_w + m * (W + 1) + part * 4;
        d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
    }
    __syncthreads();
    const unsigned char* sb = reinterpret_cast<const unsigned char*>(smem_w);
    for (int e = threadIdx.x; e < 16 * tm; e += blockDim.x) {
        const int rho = e / tm, m = e - rho * tm;
        const unsigned char* p = sb + (size_t)m * (W + 1) * 4 + rho * bps;
        unsigned char* q = out + ((size_t)ms * 16 + rho) * pitch + (size_t)(m0 + m) * bps;
        if (bps == 2) *reinterpret_cast<unsigned short*>(q) = *reinterpret_cast<const unsigned short*>(p);
        else if (bps == 4) *reinterpret_cast<unsigned*>(q) = *reinterpret_cast<const unsigned*>(p);
        else *q = *p;
    }
}

// non-root shard, after K2: its candidates are in the root's table (stores issued by the preceding kernel)
__global__ void xchg_done_kernel(unsigned* flag, unsigned epoch) {
    __threadfence_system();
    flag_store_sys(flag, epoch);
}
// root, before K4: every other shard has delivered this step's candidates
__global__ void xchg_wait_kernel(const unsigned* done_flags, int world, unsigned long long has_rows, unsigned epoch, unsigned* timeout) {
    const int r = 1 + (int)threadIdx.x;
    if (r >= world) return;
    // with fewer PRNs (or rows) than shards a shard may end up with nothing to search: it never reports
    if ((has_rows >> r) & 1ull) flag_wait_sys(done_flags + r, epoch, timeout);
}

// acquisition.m:30-32 -- per-component mean of the int16 I/Q block (exact integer sums).  On the comb-row path the
// sums scan the handle's comb copy, i.e. the block as pulled (its zero pad pairs included), on the K1 v1 path the IF
// block itself; means_kernel divides by the true sample count N*K*M either way.
__global__ void sum_int16_kernel(const int16_t* __restrict__ s, long long n_pairs, long long* __restrict__ sums) {
    long long si = 0, sq = 0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_pairs;
         i += (long long)gridDim.x * blockDim.x) {
        si += s[2 * i];
        sq += s[2 * i + 1];
    }
    for (int off = 16; off; off >>= 1) {
        si += __shfl_down_sync(0xffffffffu, si, off);
        sq += __shfl_down_sync(0xffffffffu, sq, off);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd((unsigned long long*)&sums[0], (unsigned long long)si);
        atomicAdd((unsigned long long*)&sums[1], (unsigned long long)sq);
    }
}
__global__ void means_kernel(const long long* __restrict__ sums, long long n_pairs, double* __restrict__ means) {
    means[0] = (double)sums[0] / (double)n_pairs;
    means[1] = (double)sums[1] / (double)n_pairs;
}

// Fine-frequency combine (acquisition.m:110-116): for every (sv, r, q1) the L decimated spectra are
// twiddled and combined by a direct DFT-L, giving X[K*(q1 + N*q2) + r]; |X|^2 feeds a first-index
// argmax in the reference's index order (after fftshift for I/Q data), packed as
// (float bits << 32) | (0xFFFFFFFF - index) so one 64-bit max implements value-then-lowest-index.
__global__ void __launch_bounds__(256) fine_combine_kernel(const cf* __restrict__ u, int K, int L, int N, long long F,
                                                           int shifted, unsigned long long* __restrict__ best) {
    __shared__ cf wl[16];
    __shared__ unsigned long long wbest[8];
    const int r = blockIdx.y, sv = blockIdx.z;
    if (threadIdx.x < L) {
        double s, c;
        sincospi(-2.0 * (double)threadIdx.x / (double)L, &s, &c);
        wl[threadIdx.x] = mk((float)c, (float)s);
    }
    __syncthreads();
    const int q1 = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long key = 0ull;
    if (q1 < N) {
        cf v[16];
        const cf* base = u + ((size_t)(sv * K + r) * L) * N + q1;
        const long long LN = (long long)L * N;
        for (int n2 = 0; n2 < L; ++n2) {
            const cf x = base[(size_t)n2 * N];
            const long long m = ((long long)n2 * q1) % LN;
            float si, co;
            sincospif((float)(2.0 * (double)m / (double)LN), &si, &co);
            v[n2] = mk(x.x * co + x.y * si, x.y * co - x.x * si);       // x * exp(-2 pi i m / LN)
        }
        for (int q2 = 0; q2 < L; ++q2) {
            float yr = 0.f, yi = 0.f;
            for (int n2 = 0; n2 < L; ++n2) {
                const cf w = wl[(n2 * q2) % L];
                yr += v[n2].x * w.x - v[n2].y * w.y;
                yi += v[n2].x * w.y + v[n2].y * w.x;
            }
            const long long k = (long long)K * ((long long)q1 + (long long)N * q2) + r;
            const long long j = shifted ? (k + F / 2) % F : k;
            const float pw = yr * yr + yi * yi;
            const unsigned long long cand = ((unsigned long long)__float_as_uint(pw) << 32) |
                                            (unsigned long long)(0xFFFFFFFFu - (unsigned)j);
            key = cand > key ? cand : key;
        }
    }
    for (int off = 16; off; off >>= 1) {
        const unsigned long long o = __shfl_down_sync(0xffffffffu, key, off);
        key = o > key ? o : key;
    }
    if ((threadIdx.x & 31) == 0) wbest[threadIdx.x >> 5] = key;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) key = wbest[w] > key ? wbest[w] : key;
        atomicMax(best + sv, key);
    }
}

// FP32 FMA peak probe: 16 independent FFMA chains per thread, 8 CTAs x 256 threads per SM.
__global__ void __launch_bounds__(256) fma_peak_kernel(float* out, int iters, float a, float b) {
    float v[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = (float)(threadIdx.x + i) * 1e-3f;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int r = 0; r < 8; ++r) {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = fmaf(v[i], a, b);
        }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += v[i];
    if (s == 123.456f) out[0] = s;   // never true; keeps the chains alive
}

}  // namespace

// ---------------------------------------------------------------- tracking correlators (SURVEY 8f-2)
// trackingCT.m:85-118 for a batch of channels: numSample samples from the channel's position in the resident
// recording, carrier replica exp(i(2 pi f n/Fs + remPhase)) (:103-106), "Inphase" = imag(x.*carr), "Quadrature"
// = real(x.*carr) (:112-113), code replicas Code(ceil(t)+1), t = spacing + remChip + n*codeFreq/Fs (:96-101), and
// the sums per tap (:115-117).  Float64 throughout, like the reference: the kernel is latency-, not flop-bound.
constexpr int kTrackMaxChannels = 64, kTrackMaxTaps = 32, kTrackChunks = 32, kTrackTapsPerThread = 8, kTrackThreads = 256;

struct TrackArgs {
    const void* raw;
    int data_type, precision;
    double fs_hz;
    const gnssacq_channel* ch;
    int n_taps;
    const double* spacing;
    const int8_t* ca;
    const double* mean;       // [channels][2] (int16 path) or nullptr
    double* partial;          // [channels][kTrackChunks][n_taps][2]
};

__device__ __forceinline__ void track_sample(const TrackArgs& a, long long idx, double mi, double mq, double& xr, double& xi) {
    if (a.precision == 2) {
        const int16_t* p = (const int16_t*)a.raw;
        xr = (double)p[2 * idx] - mi;
        xi = (double)p[2 * idx + 1] - mq;
    } else if (a.data_type == 2) {
        const char2 v = ((const char2*)a.raw)[idx];
        xr = (double)v.x;
        xi = (double)v.y;
    } else {
        xr = (double)((const int8_t*)a.raw)[idx];
        xi = 0.0;
    }
}

// trackingCT.m:90-92: per-integration DC of the int16 I and Q streams (exact integer sums)
__global__ void __launch_bounds__(kTrackThreads) track_mean_kernel(TrackArgs a, double* __restrict__ mean) {
    __shared__ long long sh[2][kTrackThreads / 32];
    const gnssacq_channel c = a.ch[blockIdx.x];
    const int16_t* p = (const int16_t*)a.raw + 2 * c.sample_offset;
    long long si = 0, sq = 0;
    for (int n = threadIdx.x; n < c.num_samples; n += kTrackThreads) { si += p[2 * n]; sq += p[2 * n + 1]; }
    for (int off = 16; off; off >>= 1) { si += __shfl_down_sync(0xffffffffu, si, off); sq += __shfl_down_sync(0xffffffffu, sq, off); }
    if ((threadIdx.x & 31) == 0) { sh[0][threadIdx.x >> 5] = si; sh[1][threadIdx.x >> 5] = sq; }
    __syncthreads();
    if (threadIdx.x == 0) {
        si = sq = 0;
        for (int w = 0; w < kTrackThreads / 32; ++w) { si += sh[0][w]; sq += sh[1][w]; }
        mean[2 * blockIdx.x] = (double)si / (double)c.num_samples;
        mean[2 * blockIdx.x + 1] = (double)sq / (double)c.num_samples;
    }
}

// grid (chunk, channel, tap group of 8)
__global__ void __launch_bounds__(kTrackThreads) correlate_kernel(TrackArgs a) {
    __shared__ double sh[kTrackThreads / 32][2 * kTrackTapsPerThread];
    const int cidx = blockIdx.y, tap0 = blockIdx.z * kTrackTapsPerThread;
    const gnssacq_channel c = a.ch[cidx];
    const int per = (c.num_samples + kTrackChunks - 1) / kTrackChunks;
    const int n_begin = blockIdx.x * per, n_end = min(n_begin + per, c.num_samples);
    const double step = c.code_hz / a.fs_hz;
    const double mi = a.mean ? a.mean[2 * cidx] : 0.0, mq = a.mean ? a.mean[2 * cidx + 1] : 0.0;
    const int8_t* ca = a.ca + (size_t)(c.prn - 1) * 1023;
    double off[kTrackTapsPerThread], acc_i[kTrackTapsPerThread], acc_q[kTrackTapsPerThread];
#pragma unroll
    for (int t = 0; t < kTrackTapsPerThread; ++t) {
        off[t] = (0.0 + (tap0 + t < a.n_taps ? a.spacing[tap0 + t] : 0.0)) + c.rem_chip;     // (0 + Spacing + remChip), :96
        acc_i[t] = acc_q[t] = 0.0;
    }
    for (int n = n_begin + threadIdx.x; n < n_end; n += kTrackThreads) {
        double xr, xi;
        track_sample(a, c.sample_offset + n, mi, mq, xr, xi);
        // (explicit roundings: no FMA contraction, so every intermediate is the double the reference forms)
        const double wave = __dadd_rn(__dmul_rn(2.0 * 3.14159265358979323846, __dmul_rn(c.carrier_hz, (double)n / a.fs_hz)), c.rem_phase);   // :103-104
        double sn, cs;
        sincos(wave, &sn, &cs);
        const double inph = xr * sn + xi * cs;       // imag(x * exp(i wave))
        const double quad = xr * cs - xi * sn;       // real(...)
#pragma unroll
        for (int t = 0; t < kTrackTapsPerThread; ++t) {
            const double tt = __dadd_rn(off[t], __dmul_rn(step, (double)n));
            long long k = (long long)ceil(tt) - 1;                  // Code(ceil(t)+1) of [Code(end) Code Code(1)] = CA[(ceil(t)-1) mod 1023]
            k %= 1023;
            if (k < 0) k += 1023;
            const double chip = (double)ca[k];
            acc_i[t] += chip * inph;
            acc_q[t] += chip * quad;
        }
    }
#pragma unroll
    for (int t = 0; t < kTrackTapsPerThread; ++t) {
        for (int o = 16; o; o >>= 1) {
            acc_i[t] += __shfl_down_sync(0xffffffffu, acc_i[t], o);
            acc_q[t] += __shfl_down_sync(0xffffffffu, acc_q[t], o);
        }
        if ((threadIdx.x & 31) == 0) { sh[threadIdx.x >> 5][2 * t] = acc_i[t]; sh[threadIdx.x >> 5][2 * t + 1] = acc_q[t]; }
    }
    __syncthreads();
    if (threadIdx.x < 2 * kTrackTapsPerThread) {
        const int t = tap0 + threadIdx.x / 2;
        if (t < a.n_taps) {
            double v = 0.0;
            for (int w = 0; w < kTrackThreads / 32; ++w) v += sh[w][threadIdx.x];
            a.partial[(((size_t)cidx * kTrackChunks + blockIdx.x) * a.n_taps + t) * 2 + (threadIdx.x & 1)] = v;
        }
    }
}

// fixed-order sum of the chunk partials (deterministic), out[channel][tap][I,Q]
__global__ void correlate_finish_kernel(const double* __restrict__ partial, int n_taps, int n_elems, double* __restrict__ out) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;           // channel * n_taps*2 + tap*2 + iq
    if (e >= n_elems) return;
    const int per = n_taps * 2, c = e / per, r = e - c * per;
    double v = 0.0;
    for (int k = 0; k < kTrackChunks; ++k) v += partial[((size_t)c * kTrackChunks + k) * per + r];
    out[e] = v;
}

// trackingCT.m:70-172 closed on the device.  One cluster of kLoopCtas CTAs per channel; every thread carries an
// identical copy of the channel state (all updates are the same float64 instruction sequence on the same
// reduced sums), so one cluster barrier per period is the only synchronisation: per-CTA sums go to a
// double-buffered shared-memory slot, the barrier publishes them, every CTA adds the slots in rank order.
constexpr int kLoopCtas = 8, kLoopThreads = 512;

struct LoopArgs {
    const void* raw;
    long long total_samples;
    int data_type, precision;
    double fs_hz, code_basis_hz;
    const gnssacq_channel* start;
    const int8_t* ca;
    gnssacq_loop_params lp;
    int n_periods;
    gnssacq_track_record* out;
    int* status;              // != 0: some channel ran out of samples
};

__device__ __forceinline__ double round_half_away(double v) { return v < 0.0 ? -floor(-v + 0.5) : floor(v + 0.5); }

__global__ void __launch_bounds__(kLoopThreads, 1) track_loop_kernel(LoopArgs a) {
    namespace cgx = cooperative_groups;
    cgx::cluster_group cluster = cgx::this_cluster();
    __shared__ double slot[2][8];                       // [parity][E_i E_q P_i P_q L_i L_q sumI sumQ]
    __shared__ double wsum[kLoopThreads / 32][8];
    __shared__ double total[2][6];                      // cluster-wide sums of the period (same in every CTA)
    const int rank = (int)cluster.block_rank(), cidx = blockIdx.x / kLoopCtas;
    const int gtid = rank * kLoopThreads + threadIdx.x, gthreads = kLoopCtas * kLoopThreads;
    const gnssacq_channel c0 = a.start[cidx];
    const int8_t* ca = a.ca + (size_t)(c0.prn - 1) * 1023;
    // calcLoopCoef.m:41-45
    const double wn_c = a.lp.dll_bw * 8 * a.lp.dll_damp / (4 * a.lp.dll_damp * a.lp.dll_damp + 1);
    const double tau1c = a.lp.dll_gain / (wn_c * wn_c), tau2c = 2.0 * a.lp.dll_damp / wn_c;
    const double wn_p = a.lp.pll_bw * 8 * a.lp.pll_damp / (4 * a.lp.pll_damp * a.lp.pll_damp + 1);
    const double tau1p = a.lp.pll_gain / (wn_p * wn_p), tau2p = 2.0 * a.lp.pll_damp / wn_p;
    const double sp[3] = {-a.lp.spacing_chips, 0.0, a.lp.spacing_chips};              // :24
    // The channel state lives in shared memory; thread 0 of EVERY CTA advances it (the same float64 instruction
    // sequence on the same sums in all eight CTAs -- identical results, no exchange), the other threads only read
    // it: the scalar loop math (divisions, sqrt, atan, fmod) would otherwise be executed 4096 times per period.
    struct State { double rem_chip, rem_phase, code_hz, carrier_hz, step; long long pos; int ns; int stop; };
    __shared__ State state[2];
    const double carrier_basis = c0.carrier_hz;
    double code_out_last = 0.0, dll_last = 0.0, carr_out_last = 0.0, pll_last = 0.0;          // (thread 0 only)
    const double two_pi = 2.0 * 3.14159265358979323846;
    auto publish = [&](State& st, double rem_chip, double rem_phase, double code_hz, double carrier_hz, long long pos) {
        st.rem_chip = rem_chip; st.rem_phase = rem_phase; st.code_hz = code_hz; st.carrier_hz = carrier_hz; st.pos = pos;
        st.step = code_hz / a.fs_hz;
        st.ns = (int)round_half_away((1023.0 - rem_chip) / st.step);                  // :78 (pdi = 1)
        st.stop = (st.ns < 1 || pos + st.ns > a.total_samples) ? 1 : 0;               // :107-111
    };
    if (threadIdx.x == 0) publish(state[0], c0.rem_chip, c0.rem_phase, c0.code_hz, c0.carrier_hz, c0.sample_offset);
    __syncthreads();

    for (int period = 0; period < a.n_periods; ++period) {
        const int par = period & 1;
        const double rem_chip = state[par].rem_chip, rem_phase = state[par].rem_phase, carrier_hz = state[par].carrier_hz,
                     code_hz = state[par].code_hz, step = state[par].step;
        const long long pos = state[par].pos;
        const int ns = state[par].ns;
        if (state[par].stop) {                                                        // uniform over the cluster
            if (gtid == 0) atomicExch(a.status, 1);
            break;
        }
        double mi = 0.0, mq = 0.0;
        if (a.precision == 2) {                                                       // :90-92 per-period DC of I and Q
            const int16_t* p = (const int16_t*)a.raw + 2 * pos;
            long long si = 0, sq = 0;
            for (int n = gtid; n < ns; n += gthreads) { si += p[2 * n]; sq += p[2 * n + 1]; }
            for (int o = 16; o; o >>= 1) { si += __shfl_down_sync(0xffffffffu, si, o); sq += __shfl_down_sync(0xffffffffu, sq, o); }
            if ((threadIdx.x & 31) == 0) { wsum[threadIdx.x >> 5][6] = (double)si; wsum[threadIdx.x >> 5][7] = (double)sq; }
            __syncthreads();
            if (threadIdx.x == 0) {
                double ti = 0.0, tq = 0.0;                                            // exact: integer-valued, < 2^53
                for (int w = 0; w < kLoopThreads / 32; ++w) { ti += wsum[w][6]; tq += wsum[w][7]; }
                slot[par][6] = ti; slot[par][7] = tq;
            }
            cluster.sync();
            double ti = 0.0, tq = 0.0;
            for (int r = 0; r < kLoopCtas; ++r) {
                const double* o = cluster.map_shared_rank(&slot[par][0], r);
                ti += o[6]; tq += o[7];
            }
            mi = ti / (double)ns; mq = tq / (double)ns;
            cluster.sync();                                                           // slots free for the correlator sums
        }
        double acc[6] = {0, 0, 0, 0, 0, 0};
        const double off0 = (0.0 + sp[0]) + rem_chip, off1 = (0.0 + sp[1]) + rem_chip, off2 = (0.0 + sp[2]) + rem_chip;
        // Carrier replica (:103-106): this thread's samples are n = gtid + j*gthreads, so its phasor advances by a
        // constant rotation per step -- two sincos per period instead of one per sample (the rotation's rounding
        // grows by ~1e-16 per step over <= 15 steps; gnssacq_correlate keeps the per-sample form).
        double cs, sn, rc, rs;
        sincos(__dadd_rn(__dmul_rn(two_pi, __dmul_rn(carrier_hz, (double)gtid / a.fs_hz)), rem_phase), &sn, &cs);
        sincos(two_pi * (carrier_hz * ((double)gthreads / a.fs_hz)), &rs, &rc);
        constexpr int kBatch = 16;                       // samples per thread fetched before any is used: the loads
        for (int n0 = gtid; n0 < ns; n0 += kBatch * gthreads) {          // overlap instead of paying 15 L2/HBM latencies in a row
            float fr[kBatch], fi[kBatch];                // (int8 / int16 values are exact in float)
#pragma unroll
            for (int j = 0; j < kBatch; ++j) {
                const int n = n0 + j * gthreads;
                fr[j] = fi[j] = 0.f;
                if (n < ns) {
                    const long long idx = pos + n;
                    if (a.precision == 2) { const short2 v = ((const short2*)a.raw)[idx]; fr[j] = (float)v.x; fi[j] = (float)v.y; }
                    else if (a.data_type == 2) { const char2 v = ((const char2*)a.raw)[idx]; fr[j] = (float)v.x; fi[j] = (float)v.y; }
                    else fr[j] = (float)((const int8_t*)a.raw)[idx];
                }
            }
#pragma unroll
            for (int j = 0; j < kBatch; ++j) {
                const int n = n0 + j * gthreads;
                if (n < ns) {
                    const double xr = (double)fr[j] - mi, xi = (a.data_type == 2 || a.precision == 2) ? (double)fi[j] - mq : 0.0;
                    const double inph = xr * sn + xi * cs, quad = xr * cs - xi * sn;          // :112-113
                    const double cn = cs * rc - sn * rs;
                    sn = sn * rc + cs * rs;
                    cs = cn;
                    const double sn_d = __dmul_rn(step, (double)n);
                    const double offs[3] = {off0, off1, off2};
#pragma unroll
                    for (int t = 0; t < 3; ++t) {
                        int k = (int)ceil(__dadd_rn(offs[t], sn_d)) - 1;                      // :96-101; |t| < 2^31 chips by far
                        k %= 1023;
                        if (k < 0) k += 1023;
                        const double chip = (double)ca[k];
                        acc[2 * t] += chip * inph;
                        acc[2 * t + 1] += chip * quad;
                    }
                }
            }
        }
#pragma unroll
        for (int t = 0; t < 6; ++t) {
            for (int o = 16; o; o >>= 1) acc[t] += __shfl_down_sync(0xffffffffu, acc[t], o);
            if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5][t] = acc[t];
        }
        __syncthreads();
        if (threadIdx.x < 6) {
            double v = 0.0;
            for (int w = 0; w < kLoopThreads / 32; ++w) v += wsum[w][threadIdx.x];
            slot[par][threadIdx.x] = v;
        }
        cluster.sync();                                                               // release/acquire: all slots visible
        if (threadIdx.x < 6) {                                                        // six threads pull the eight slots
            double v = 0.0;
            for (int r = 0; r < kLoopCtas; ++r) v += cluster.map_shared_rank(&slot[par][0], r)[threadIdx.x];
            total[par][threadIdx.x] = v;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            const double E_i = total[par][0], E_q = total[par][1], P_i = total[par][2], P_q = total[par][3],
                         L_i = total[par][4], L_q = total[par][5];
            // :102, :105 (with this period's NCO values), then the loops :135-150
            const double n_rem_chip = __dadd_rn(__dadd_rn(__dadd_rn(off1, __dmul_rn(step, (double)(ns - 1))), step), -__dmul_rn(a.code_basis_hz, 1e-3));
            const double n_rem_phase = fmod(__dadd_rn(__dmul_rn(two_pi, __dmul_rn(carrier_hz, (double)ns / a.fs_hz)), rem_phase), two_pi);
            const double E = sqrt(E_i * E_i + E_q * E_q), L = sqrt(L_i * L_i + L_q * L_q);
            const double dll = 0.5 * (E - L) / (E + L);
            const double code_out = code_out_last + (tau2c / tau1c) * (dll - dll_last) + dll * (0.001 / tau1c);
            dll_last = dll; code_out_last = code_out;
            const double n_code_hz = a.code_basis_hz - code_out;
            const double pll = atan(P_q / P_i) / two_pi;
            const double carr_out = carr_out_last + (tau2p / tau1p) * (pll - pll_last) + pll * (0.001 / tau1p);
            carr_out_last = carr_out; pll_last = pll;
            const double n_carrier_hz = carrier_basis + carr_out;
            publish(state[par ^ 1], n_rem_chip, n_rem_phase, n_code_hz, n_carrier_hz, pos + ns);
            if (rank == 0) {
                gnssacq_track_record r;
                r.P_i = P_i; r.P_q = P_q; r.E_i = E_i; r.E_q = E_q; r.L_i = L_i; r.L_q = L_q;
                r.pll_discri = pll; r.dll_discri = dll;
                r.rem_chip = n_rem_chip; r.code_hz = n_code_hz; r.carrier_hz = n_carrier_hz; r.rem_phase = n_rem_phase;
                r.sample_end = pos + ns; r.num_samples = ns; r.reserved = 0;
                a.out[(size_t)cidx * a.n_periods + period] = r;
            }
        }
        __syncthreads();                                   // state[par ^ 1] is complete
        // (the next period writes slot[par ^ 1]; slot[par] is rewritten two cluster barriers from now)
        (void)code_hz;
    }
    cluster.sync();                                        // nobody exits while its slots may still be read
}

// ---------------------------------------------------------------- handle
struct gnssacq_handle {
    gnssacq_config cfg;
    const VariantOps* ops = nullptr;
    int device = 0;
    int N = 0, P = 0, B = 0, K = 0, M = 0;
    int w = 0;
    size_t if_bytes = 0;
    std::vector<int> bin_base, bin_shift;
    std::vector<double> base_freq;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    // device buffers
    void* d_if = nullptr;
    int8_t* d_scode = nullptr;
    cf* d_cc = nullptr;
    cf* d_x = nullptr;
    int *d_bin_base = nullptr, *d_bin_shift = nullptr, *d_prn = nullptr;
    double* d_base_freq = nullptr;
    double* d_base_w = nullptr;            // (IF + doppler) / Fs per base, cycles per sample (K1 v2)
    unsigned char* d_comb = nullptr;       // [K*M ms][16][comb_pitch] re-ordered IF block (K1 v2), nullptr: K1 v1
    int comb_pitch = 0;
    Candidate* d_cand = nullptr;
    gnssacq_result* d_res = nullptr;
    float* d_surface = nullptr;
    cf* d_scratch = nullptr;
    int l2x_clusters = 0;          // > 0: use the L2-exchange persistent search kernel with this many clusters
    int coop_groups = 0;           // > 0: use the cluster-free cooperative kernel with this many CTA groups
    unsigned* d_group_ctr = nullptr;
    int bin0 = 0, B_full = 0;      // this handle's bins are [bin0, bin0 + B) of the B_full-bin grid
    int row0 = 0, n_rows = 0;      // ... and of that P x B grid (row = bin * P + prn index) it searches rows [row0, row0 + n_rows)
    // multi-GPU exchange (gnssacq_xchg_*)
    struct Xchg {
        bool on = false, is_root = false;
        gnssacq_shard sh{};
        unsigned char* block = nullptr;        // root: the exchange block (cudaMalloc); others: the mapped root block
        bool ipc_opened = false;
        unsigned char* if_buf = nullptr;       // root's IF buffer
        Candidate* cand_all = nullptr;         // root's [n_prn_total][freq_num_total]
        unsigned* flags = nullptr;             // [0] IF ready, [1 + r] shard r done, [63] timeout
        int* d_prn_all = nullptr;              // root
        gnssacq_result* d_res_all = nullptr;   // root
        gnssacq_result* h_res_all = nullptr;   // root, pinned
        unsigned epoch = 0;
        cudaEvent_t ev_a = nullptr, ev_b = nullptr, ev_c = nullptr, ev_d = nullptr;
    } xc;
    const gnssacq_result* d_last_rows = nullptr;   // where the last enqueued search wrote its rows (d_res or the caller's buffer)
    Candidate* d_row_slots = nullptr;
    float* d_partial = nullptr;    // cooperative kernel: accumulators of row parts handed between groups
    long long* d_sums = nullptr;
    double* d_means = nullptr;
    cf *d_fft_in = nullptr, *d_fft_out = nullptr;
    // fine-frequency stage scratch, kept between calls (re-made only when L changes)
    int fine_L = 0;
    void* d_fine_raw = nullptr;
    uint16_t* d_fine_chip = nullptr;
    cf* d_fine_u = nullptr;
    int8_t* d_fine_ca = nullptr;
    int* d_fine_start = nullptr;
    unsigned long long* d_fine_best = nullptr;
    // re-acquisition sweep (gnssacq_sweep): second staging pair, copy stream, per-buffer events, result slab
    void* d_if2 = nullptr;
    void* h_if2 = nullptr;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_copied[2] = {}, ev_consumed[2] = {};
    gnssacq_result* d_res_sweep = nullptr;
    int sweep_cap = 0;
    // tracking correlators (gnssacq_track_load / gnssacq_correlate): resident recording segment, C/A table,
    // per-call channel table and partial sums
    void* d_trk_raw = nullptr;
    size_t trk_bytes = 0, trk_cap = 0;
    int8_t* d_trk_ca = nullptr;            // [GNSSACQ_TRACK_MAX_PRN][1023]
    void* d_trk_ch = nullptr;              // [kTrackMaxChannels] gnssacq_channel
    double* d_trk_spacing = nullptr;       // [kTrackMaxTaps]
    double* d_trk_partial = nullptr;       // [channels][chunks][taps][2]
    double* d_trk_out = nullptr;           // [channels][taps][2]
    double* d_trk_mean = nullptr;          // [channels][2] int16 path
    double* h_trk_out = nullptr;           // pinned
    gnssacq_track_record* d_trk_rec = nullptr;   // [channels][periods] of the last gnssacq_track
    size_t trk_rec_cap = 0;
    int* d_trk_status = nullptr;
    // pinned host
    void* h_if = nullptr;
    gnssacq_result* h_res = nullptr;
    cudaEvent_t ev[6] = {};
    cudaEvent_t ev_upload = nullptr;       // last DMA out of the pinned staging buffer h_if (stage_and_upload)
    bool have_h2d = false;
    int launches = 0;
    std::string err;
};

namespace {

int fail(gnssacq_handle* h, int code, const std::string& msg) {
    if (h) h->err = msg;
    g_create_error = msg;
    return code;
}
#define CU(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess)                                                                          \
            return fail(h, GNSSACQ_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));       \
    } while (0)

const VariantOps* pick_variant(int Q, int R, int T) {
    int n = 0;
    const VariantOps* v = nullptr;
    if (Q == 3) v = gnss_variants_q3(&n);
    else if (Q == 13) v = gnss_variants_q13(&n);
    else if (Q == 29) v = gnss_variants_q29(&n);
    if (!v) return nullptr;
    for (int i = 0; i < n; ++i)
        if ((R == 0 || v[i].R == R) && (T == 0 || v[i].T == T)) return &v[i];
    return nullptr;
}

// Doppler bins -> (base transform, shift in FFT bins): f_b = f_base + s * (Fs/N)   (SURVEY A.7)
void plan_bins(gnssacq_handle* h) {
    const gnssacq_config& c = h->cfg;
    const double df = c.fs_hz / (double)c.samples_per_ms;
    h->bin_base.assign(h->B, 0);
    h->bin_shift.assign(h->B, 0);
    h->base_freq.clear();
    for (int b = 0; b < h->B; ++b) {
        const double f = c.if_hz + (c.freq_min_hz + c.freq_step_hz * (double)b);     // acquisition.m:42-43
        int found = -1, shift = 0;
        for (size_t i = 0; i < h->base_freq.size(); ++i) {
            const double r = (f - h->base_freq[i]) / df;
            const double rr = std::nearbyint(r);
            if (std::fabs(r - rr) * df < 1e-6 && std::fabs(rr) < (double)(c.samples_per_ms / 2)) {
                found = (int)i;
                shift = (int)rr;
                break;
            }
        }
        if (found < 0) {
            h->base_freq.push_back(f);
            found = (int)h->base_freq.size() - 1;
            shift = 0;
        }
        h->bin_base[b] = found;
        h->bin_shift[b] = shift;
    }
}

int validate(const gnssacq_config* c, std::string& why) {
    if (!c) { why = "cfg is NULL"; return GNSSACQ_ERR_INVALID_ARG; }
    if (!(c->fs_hz > 0) || !(c->code_hz > 0)) { why = "fs_hz and code_hz must be positive"; return GNSSACQ_ERR_INVALID_ARG; }
    if (c->data_type != 1 && c->data_type != 2) { why = "data_type must be 1 (real) or 2 (I/Q)"; return GNSSACQ_ERR_INVALID_ARG; }
    if (c->data_precision != 1 && c->data_precision != 2) { why = "data_precision must be 1 (int8) or 2 (int16)"; return GNSSACQ_ERR_INVALID_ARG; }
    if (c->data_precision == 2 && c->data_type != 2) { why = "int16 input is always I/Q (acquisition.m:29-32)"; return GNSSACQ_ERR_INVALID_ARG; }
    if (c->freq_num < 1 || c->noncoh_blocks < 1 || c->coh_ms < 1) { why = "freq_num, noncoh_blocks, coh_ms must be >= 1"; return GNSSACQ_ERR_INVALID_ARG; }
    if (c->n_prn < 1 || c->n_prn > GNSSACQ_MAX_PRN) { why = "n_prn must be 1..64"; return GNSSACQ_ERR_INVALID_ARG; }
    for (int i = 0; i < c->n_prn; ++i)
        if (c->prn[i] < 1 || c->prn[i] > 51) { why = "PRN outside 1..51"; return GNSSACQ_ERR_INVALID_ARG; }
    if (c->bin_count < 0 || c->bin_first < 0 || (c->bin_count > 0 && c->bin_first + c->bin_count > c->freq_num) ||
        (c->bin_count == 0 && c->bin_first != 0)) { why = "bin_first / bin_count outside the freq_num grid"; return GNSSACQ_ERR_INVALID_ARG; }
    {
        const long long grid = (long long)c->n_prn * (c->bin_count > 0 ? c->bin_count : c->freq_num);
        if (c->row_first < 0 || c->row_count < 0 || (long long)c->row_first + c->row_count > grid || (c->row_count == 0 && c->row_first != 0)) {
            why = "row_first / row_count outside the n_prn x bins grid"; return GNSSACQ_ERR_INVALID_ARG;
        }
    }
    if (c->work_split < 0 || c->work_split > 2) { why = "work_split must be 0 (auto), 1 (whole rows) or 2 (block-granular tail)"; return GNSSACQ_ERR_INVALID_ARG; }
    if (c->exchange < 0 || c->exchange > 3) { why = "exchange must be 0 (auto), 1 (DSMEM), 2 (L2 + clusters) or 3 (L2 + cooperative groups)"; return GNSSACQ_ERR_INVALID_ARG; }
    if (c->samples_per_ms <= 0 || c->samples_per_ms % 2000 != 0) {
        why = "samples_per_ms must be 2000*Q (built: Q = 3, 13, 29 -> 6000, 26000, 58000)";
        return GNSSACQ_ERR_UNSUPPORTED_N;
    }
    return GNSSACQ_OK;
}

}  // namespace

// ---------------------------------------------------------------- C ABI
extern "C" {

const char* gnssacq_version(void) { return GNSSACQ_VERSION_STR; }

int gnssacq_config_default(gnssacq_config* c) {
    if (!c) return GNSSACQ_ERR_INVALID_ARG;
    std::memset(c, 0, sizeof(*c));
    c->fs_hz = 58e6;                 // initParameters.m:42
    c->if_hz = 4.58e6;               // :41
    c->code_hz = 1.023e6;            // :44
    c->samples_per_ms = 58000;       // :46
    c->data_type = 2;                // :37
    c->data_precision = 1;           // :38
    c->freq_min_hz = -10000.0;       // :52
    c->freq_step_hz = 500.0;         // :51
    c->freq_num = 41;                // :53
    c->noncoh_blocks = 20;           // :54
    c->coh_ms = 1;
    c->n_prn = 32;                   // acquisition.m:47
    for (int i = 0; i < 32; ++i) c->prn[i] = i + 1;
    c->snr_threshold_db = 12.0;      // acquisition.m:70
    c->device = -1;
    return GNSSACQ_OK;
}

size_t gnssacq_if_bytes(const gnssacq_config* c) {
    if (!c) return 0;
    return (size_t)c->samples_per_ms * (size_t)c->data_type * (size_t)c->data_precision *
           (size_t)c->noncoh_blocks * (size_t)c->coh_ms;
}

int gnssacq_ca_code(int32_t prn, int8_t out[1023]) {
    if (!out || prn < 1 || prn > 51) return GNSSACQ_ERR_INVALID_ARG;
    ca_chips(prn, out);
    return GNSSACQ_OK;
}

int gnssacq_code_replica(const gnssacq_config* c, int32_t prn, int8_t* out) {
    if (!c || !out || prn < 1 || prn > 51 || c->samples_per_ms <= 0 || !(c->fs_hz > 0)) return GNSSACQ_ERR_INVALID_ARG;
    code_replica(*c, prn, out);
    return GNSSACQ_OK;
}

const char* gnssacq_last_error(const gnssacq_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int gnssacq_destroy(gnssacq_handle* h) {
    if (!h) return GNSSACQ_ERR_INVALID_ARG;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    cudaFree(h->d_if); cudaFree(h->d_scode); cudaFree(h->d_cc); cudaFree(h->d_x);
    cudaFree(h->d_bin_base); cudaFree(h->d_bin_shift); cudaFree(h->d_prn); cudaFree(h->d_base_freq); cudaFree(h->d_base_w); cudaFree(h->d_comb);
    cudaFree(h->d_cand); cudaFree(h->d_res); cudaFree(h->d_surface); cudaFree(h->d_scratch); cudaFree(h->d_group_ctr); cudaFree(h->d_row_slots); cudaFree(h->d_partial); cudaFree(h->d_if2); cudaFree(h->d_res_sweep);
    if (h->xc.on) {
        if (h->xc.is_root) { cudaFree(h->xc.block); cudaFree(h->xc.d_prn_all); cudaFree(h->xc.d_res_all); if (h->xc.h_res_all) cudaFreeHost(h->xc.h_res_all); }
        else if (h->xc.ipc_opened) cudaIpcCloseMemHandle(h->xc.block);
        for (cudaEvent_t e : {h->xc.ev_a, h->xc.ev_b, h->xc.ev_c, h->xc.ev_d}) if (e) cudaEventDestroy(e);
    }
    if (h->ev_upload) cudaEventDestroy(h->ev_upload);
    if (h->h_if2) cudaFreeHost(h->h_if2);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    for (auto& e : h->ev_copied) if (e) cudaEventDestroy(e);
    for (auto& e : h->ev_consumed) if (e) cudaEventDestroy(e);
    cudaFree(h->d_sums); cudaFree(h->d_means);
    cudaFree(h->d_trk_raw); cudaFree(h->d_trk_ca); cudaFree(h->d_trk_ch); cudaFree(h->d_trk_spacing); cudaFree(h->d_trk_partial);
    cudaFree(h->d_trk_out); cudaFree(h->d_trk_mean); cudaFree(h->d_trk_rec); cudaFree(h->d_trk_status);
    if (h->h_trk_out) cudaFreeHost(h->h_trk_out);
    cudaFree(h->d_fft_in); cudaFree(h->d_fft_out);
    cudaFree(h->d_fine_raw); cudaFree(h->d_fine_chip); cudaFree(h->d_fine_u); cudaFree(h->d_fine_ca); cudaFree(h->d_fine_start); cudaFree(h->d_fine_best);
    if (h->h_if) cudaFreeHost(h->h_if);
    if (h->h_res) cudaFreeHost(h->h_res);
    for (auto& e : h->ev) if (e) cudaEventDestroy(e);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;
    return GNSSACQ_OK;
}

int gnssacq_create(const gnssacq_config* cfg, gnssacq_handle** out) {
    gnssacq_handle* h = nullptr;
    if (!out) return fail(nullptr, GNSSACQ_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    std::string why;
    int rc = validate(cfg, why);
    if (rc != GNSSACQ_OK) return fail(nullptr, rc, why);

    const int Q = cfg->samples_per_ms / 2000;
    const VariantOps* ops = pick_variant(Q, cfg->cluster_ctas, cfg->threads);
    if (!ops) {
        char buf[200];
        std::snprintf(buf, sizeof buf, "no engine variant for samples_per_ms=%d (Q=%d) cluster_ctas=%d threads=%d",
                      cfg->samples_per_ms, Q, cfg->cluster_ctas, cfg->threads);
        return fail(nullptr, GNSSACQ_ERR_UNSUPPORTED_N, buf);
    }

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(nullptr, GNSSACQ_ERR_NO_DEVICE, "no CUDA device: libgnssacq has no CPU fallback");
    }
    int dev = cfg->device;
    if (dev < 0) { if (cudaGetDevice(&dev) != cudaSuccess) dev = 0; }
    if (dev >= ndev) return fail(nullptr, GNSSACQ_ERR_NO_DEVICE, "device ordinal out of range");
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess) return fail(nullptr, GNSSACQ_ERR_NO_DEVICE, "cannot query device");
    if (prop.major != 10) {
        char buf[160];
        std::snprintf(buf, sizeof buf, "device %d is sm_%d%d; libgnssacq is built for sm_100a only", dev, prop.major, prop.minor);
        return fail(nullptr, GNSSACQ_ERR_NO_DEVICE, buf);
    }

    h = new (std::nothrow) gnssacq_handle();
    if (!h) return fail(nullptr, GNSSACQ_ERR_NOMEM, "out of host memory");
    h->cfg = *cfg;
    h->ops = ops;
    h->device = dev;
    h->N = cfg->samples_per_ms;
    h->P = cfg->n_prn;
    h->B = cfg->freq_num;
    h->K = cfg->noncoh_blocks;
    h->M = cfg->coh_ms;
    h->w = (int)std::ceil(cfg->fs_hz / cfg->code_hz);          // acquisition.m:66
    h->if_bytes = gnssacq_if_bytes(cfg);
    plan_bins(h);                                               // on the FULL grid: same bases for every bin range
    h->B_full = cfg->freq_num;
    if (cfg->bin_count > 0) {                                   // validate() has checked the range
        h->bin0 = cfg->bin_first;
        h->B = cfg->bin_count;
        const std::vector<int> bb(h->bin_base.begin() + h->bin0, h->bin_base.begin() + h->bin0 + h->B);
        const std::vector<int> bs(h->bin_shift.begin() + h->bin0, h->bin_shift.begin() + h->bin0 + h->B);
        h->bin_base = bb;
        h->bin_shift = bs;
    }
    h->row0 = cfg->row_count > 0 ? cfg->row_first : 0;
    h->n_rows = cfg->row_count > 0 ? cfg->row_count : h->P * h->B;
    const size_t N = (size_t)h->N;
    const size_t nb = h->base_freq.size();

#define CUC(call)                                                                                        \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess) {                                                                        \
            std::string m__ = std::string(#call) + ": " + cudaGetErrorString(e__);                       \
            gnssacq_destroy(h);                                                                          \
            return fail(nullptr, e__ == cudaErrorMemoryAllocation ? GNSSACQ_ERR_NOMEM : GNSSACQ_ERR_CUDA, m__); \
        }                                                                                                \
    } while (0)

    CUC(cudaSetDevice(dev));
    CUC(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    h->stream = h->own_stream;
    for (auto& e : h->ev) CUC(cudaEventCreate(&e));
    CUC(ops->prepare());
    CUC(cudaMalloc(&h->d_if, h->if_bytes));
    CUC(cudaMalloc(&h->d_scode, (size_t)h->P * N));
    CUC(cudaMalloc(&h->d_cc, (size_t)h->P * N * sizeof(cf)));
    CUC(cudaMalloc(&h->d_x, nb * (size_t)h->K * (N / (N / 2000) * (2 * (N / 2000) - 1)) * sizeof(cf)));   // c-extended: N*(2Q-1)/Q
    CUC(cudaMalloc(&h->d_bin_base, h->B * sizeof(int)));
    CUC(cudaMalloc(&h->d_bin_shift, h->B * sizeof(int)));
    CUC(cudaMalloc(&h->d_prn, h->P * sizeof(int)));
    CUC(cudaMalloc(&h->d_base_freq, nb * sizeof(double)));
    CUC(cudaMalloc(&h->d_cand, (size_t)h->P * h->B * sizeof(Candidate)));
    CUC(cudaMalloc(&h->d_res, h->P * sizeof(gnssacq_result)));
    CUC(cudaMalloc(&h->d_sums, 2 * sizeof(long long)));
    CUC(cudaMalloc(&h->d_means, 2 * sizeof(double)));
    // exchange: 1 = DSMEM clusters, 2 = L2 buffer + clusters, 3 = L2 buffer + cooperative groups (no clusters).
    // auto: cooperative groups for the two real front ends (fastest measured, profiles/r01), DSMEM for tiny N.
    const int xmode = cfg->exchange ? cfg->exchange : (Q >= 13 ? 3 : 1);
    if (xmode == 2 || xmode == 3) {
        int n = xmode == 3 ? ops->max_groups_coop() : ops->max_clusters_l2x();
        // the cooperative kernel deals out single blocks of a row (work_split 0) or whole rows (1); the
        // clustered one whole rows
        // Block-granular tail (see search_kernel_coop): needs K-1 power planes per group (150 MB at the
        // reference's sizes) -- not possible above 2 GiB or beyond the kernel's 32-bit unit arithmetic.  It
        // costs 0.15-0.4 row times (publishing and adding the planes), so work_split 0 (auto) uses it only
        // where whole rows would leave >= 4 % of the last round's group-time idle (measured r01: pays for
        // <= 8 PRNs at N = 26 000, <= 4 PRNs at N = 58 000, not for 32).  Results are identical either way.
        bool by_blocks = xmode == 3 && cfg->work_split != 1 && h->K > 1 && (unsigned long long)n * n * h->K < (1ull << 32) &&
                         (unsigned long long)n * (h->K - 1) * ops->partial_bytes_per_group <= (2ull << 30);
        if (by_blocks && cfg->work_split == 0) {
            const long long rows = h->n_rows, rounds = (rows + n - 1) / n;
            by_blocks = (double)(rounds * n - rows) >= 0.04 * (double)(rounds * n);
        }
        const long long max_useful = by_blocks ? (long long)h->n_rows * h->K : (long long)h->n_rows;
        if (n > max_useful) n = (int)max_useful;
        if (n <= 0) {
            gnssacq_destroy(h);
            return fail(nullptr, GNSSACQ_ERR_CUDA, "persistent search kernel cannot be made resident on this device");
        }
        if (xmode == 3) h->coop_groups = n; else h->l2x_clusters = n;
        CUC(cudaMalloc(&h->d_scratch, (size_t)n * ops->scratch_bytes_per_cluster));
        // the padding columns of the exchange layout are never written: they must read as exact zeros
        CUC(cudaMemsetAsync(h->d_scratch, 0, (size_t)n * ops->scratch_bytes_per_cluster, h->stream));
        CUC(cudaMalloc(&h->d_group_ctr, (size_t)n * (2 + ops->R) * sizeof(unsigned)));     // group barriers + hand-over counters + row tickets
        if (by_blocks) CUC(cudaMalloc(&h->d_partial, (size_t)n * (h->K - 1) * ops->partial_bytes_per_group));
        CUC(cudaMalloc(&h->d_row_slots, (size_t)n * ops->R * sizeof(Candidate)));
    }
    if (cfg->keep_surface) {
        CUC(cudaMalloc(&h->d_surface, (size_t)h->P * h->B * N * sizeof(float)));
        if (h->n_rows < h->P * h->B) CUC(cudaMemset(h->d_surface, 0, (size_t)h->P * h->B * N * sizeof(float)));   // rows it never searches read as zeros
    }
    CUC(cudaMallocHost(&h->h_if, h->if_bytes));
    CUC(cudaMallocHost(&h->h_res, h->P * sizeof(gnssacq_result)));
    // Every create-time copy goes on the handle's own (non-blocking) stream: a synchronous cudaMemcpy from
    // pageable memory returns once the data is STAGED, and its DMA on the legacy stream is not ordered with
    // kernels on a non-blocking stream (seen once in r01 as one PRN's code spectrum built from a half-copied
    // replica table).
    CUC(cudaMemcpyAsync(h->d_bin_base, h->bin_base.data(), h->B * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CUC(cudaMemcpyAsync(h->d_bin_shift, h->bin_shift.data(), h->B * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CUC(cudaMemcpyAsync(h->d_prn, cfg->prn, h->P * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CUC(cudaMemcpyAsync(h->d_base_freq, h->base_freq.data(), nb * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    if (h->n_rows < h->P * h->B) {
        // a row range: the cells of the handle's own table that it never writes must not win K4's maximum
        std::vector<Candidate> none((size_t)h->P * h->B, Candidate{-1.f, 0, 0.0, 0.0});
        CUC(cudaMemcpyAsync(h->d_cand, none.data(), none.size() * sizeof(Candidate), cudaMemcpyHostToDevice, h->stream));
        CUC(cudaStreamSynchronize(h->stream));
    }
    {
        // K1 v2 (comb rows + cp.async staging) whenever its shared memory fits; otherwise the v1 gather kernel
        const int bps = h->cfg.data_type * h->cfg.data_precision;
        const int pitch = ((N / 16) * bps + 15) / 16 * 16;
        if (ops->smem_wipe2(pitch, h->M) <= (size_t)227 * 1024) {
            std::vector<double> bw(nb);
            for (size_t i = 0; i < nb; ++i) bw[i] = h->base_freq[i] / h->cfg.fs_hz;
            CUC(cudaMalloc(&h->d_base_w, nb * sizeof(double)));
            CUC(cudaMemcpy(h->d_base_w, bw.data(), nb * sizeof(double), cudaMemcpyHostToDevice));
            h->comb_pitch = pitch;
            CUC(cudaMalloc(&h->d_comb, (size_t)h->K * h->M * 16 * pitch));
            CUC(cudaMemset(h->d_comb, 0, (size_t)h->K * h->M * 16 * pitch));
        }
    }

    // code tables -> HBM, then K0 fills the conj-spectrum cache
    {
        std::vector<int8_t> sc((size_t)h->P * N);
        for (int p = 0; p < h->P; ++p) code_replica(*cfg, cfg->prn[p], sc.data() + (size_t)p * N);
        CUC(cudaMemcpyAsync(h->d_scode, sc.data(), sc.size(), cudaMemcpyHostToDevice, h->stream));
        CodeArgs a{h->d_scode, h->d_cc};
        CUC(ops->launch_code(a, h->P, h->stream));
        CUC(cudaStreamSynchronize(h->stream));
    }
#undef CUC
    *out = h;
    return GNSSACQ_OK;
}

int gnssacq_set_stream(gnssacq_handle* h, void* s) {
    if (!h) return GNSSACQ_ERR_INVALID_ARG;
    h->stream = (s == GNSSACQ_OWN_STREAM) ? h->own_stream : (cudaStream_t)s;
    return GNSSACQ_OK;
}

#ifdef GNSS_TIMELINE
static unsigned long long* g_timeline = nullptr;
extern "C" int gnssacq_debug_timeline(unsigned long long* out /*[16*16*32]*/) {
    return cudaMemcpy(out, g_timeline, 16 * 16 * 32 * sizeof(unsigned long long), cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : -4;
}
#endif
// Pageable caller memory -> HBM through the handle's pinned staging buffer, in chunks: the host copy of chunk i+1
// overlaps the DMA of chunk i (one chunk of latency instead of the sum of both copies).  The caller's buffer is
// free again when this returns.
// Host copy into the pinned staging buffer with non-temporal stores: the destination is only ever read by the DMA
// engine, so it should neither be fetched into the cache first (read-for-ownership) nor evict the caller's data.
static void copy_to_staging(unsigned char* dst, const unsigned char* src, size_t n) {
#if defined(__x86_64__) && !defined(GNSS_EXPERIMENT_PLAIN_MEMCPY)
    if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
        size_t i = 0;
        for (; i + 64 <= n; i += 64) {
            const __m128i a = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + i));
            const __m128i b = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + i + 16));
            const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + i + 32));
            const __m128i d = _mm_loadu_si128(reinterpret_cast<const __m128i*>(src + i + 48));
            _mm_stream_si128(reinterpret_cast<__m128i*>(dst + i), a);
            _mm_stream_si128(reinterpret_cast<__m128i*>(dst + i + 16), b);
            _mm_stream_si128(reinterpret_cast<__m128i*>(dst + i + 32), c);
            _mm_stream_si128(reinterpret_cast<__m128i*>(dst + i + 48), d);
        }
        if (i < n) std::memcpy(dst + i, src + i, n - i);
        _mm_sfence();                                    // the streamed lines are globally visible before the DMA is queued
        return;
    }
#endif
    std::memcpy(dst, src, n);
}
static int stage_and_upload(gnssacq_handle* h, void* d_dst, const void* host_src, cudaStream_t s) {
    // (Helper threads for the host copy were built and measured in r02: three helpers claiming 128 kB pieces next to the
    // caller's thread made the upload of the 2.32 MB block SLOWER, 0.30 ms against 0.185 ms, on the 16-core host of the
    // GPU box -- waking sleeping threads costs more than the 0.1 ms they could save.  profiles/r02/time_e2e_staging_helpers_v16.txt)
    constexpr size_t kChunk = 512 << 10;
    const unsigned char* src = static_cast<const unsigned char*>(host_src);
    unsigned char* pin = static_cast<unsigned char*>(h->h_if);
    if (h->ev_upload) CU(cudaEventSynchronize(h->ev_upload));      // an earlier (asynchronous) upload still reads h_if
    else CU(cudaEventCreateWithFlags(&h->ev_upload, cudaEventDisableTiming));
    for (size_t off = 0; off < h->if_bytes; off += kChunk) {
        const size_t n = std::min(kChunk, h->if_bytes - off);
        copy_to_staging(pin + off, src + off, n);
        CU(cudaMemcpyAsync(static_cast<unsigned char*>(d_dst) + off, pin + off, n, cudaMemcpyHostToDevice, s));
    }
    CU(cudaEventRecord(h->ev_upload, s));
    return GNSSACQ_OK;
}

static int enqueue(gnssacq_handle* h, const void* d_if, gnssacq_result* d_out = nullptr, bool xchg = false) {
    cudaStream_t s = h->stream;
    h->launches = 0;
    auto& xc = h->xc;
    if (xchg && !h->d_comb) return fail(h, GNSSACQ_ERR_STATE, "the multi-GPU exchange needs the comb-row K1 (shared memory too small for this shape)");
    CU(cudaEventRecord(h->ev[1], s));
    // int16 (acquisition.m:30-32): per-component means of the N*K*M samples, from `scan` (I, Q) pairs at `src`
    const double* means = h->cfg.data_precision == 2 ? h->d_means : nullptr;
    auto launch_means = [&](const void* src, long long scan) -> int {
        CU(cudaMemsetAsync(h->d_sums, 0, 2 * sizeof(long long), s));
        sum_int16_kernel<<<296, 256, 0, s>>>((const int16_t*)src, scan, h->d_sums);
        means_kernel<<<1, 1, 0, s>>>(h->d_sums, (long long)h->N * h->K * h->M, h->d_means);
        CU(cudaGetLastError());
        h->launches += 2;
        return GNSSACQ_OK;
    };
    if (h->d_comb) {
        const int bps = h->cfg.data_type * h->cfg.data_precision;
        const int rows = h->N / 16, tiles = (rows + kCombTM - 1) / kCombTM;
        if (xchg) CU(cudaEventRecord(xc.ev_a, s));
        comb_kernel<<<h->K * h->M * tiles, 256, (size_t)kCombTM * (4 * bps + 1) * 4, s>>>(
            (const unsigned char*)d_if, h->d_comb, rows, bps, h->comb_pitch, tiles,
            (xchg && xc.is_root) ? xc.flags : nullptr, (xchg && !xc.is_root) ? xc.flags : nullptr, xc.epoch,
            xchg ? xc.flags + 63 : nullptr);
        CU(cudaGetLastError());
        if (xchg) CU(cudaEventRecord(xc.ev_b, s));
        // from the comb copy, not `d_if`: on a non-root shard that is the root's buffer (see comb_kernel).
        // [K*M*16 rows][pitch bytes], one (I, Q) pair per 4 bytes; the pad bytes are zero (memset at create, never written)
        if (means) {
            if (int rc = launch_means(h->d_comb, (long long)h->K * h->M * 16 * h->comb_pitch / 4)) return rc;
        }
        Wipe2Args w2;
        w2.comb = h->d_comb;
        w2.pitch = h->comb_pitch;
        w2.bps = bps;
        w2.coh_ms = h->M;
        w2.K = h->K;
        w2.base_w = h->d_base_w;
        w2.means = means;
        w2.x = h->d_x;
        CU(h->ops->launch_wipe2(w2, (int)h->base_freq.size() * h->K, s));
        h->launches += 2;
    } else {
        // (K1 v1 is never used by the multi-GPU exchange: `d_if` is this handle's own, complete block)
        if (means) {
            if (int rc = launch_means(d_if, (long long)h->N * h->K * h->M)) return rc;
        }
        WipeArgs wa;
        wa.raw = d_if;
        wa.data_type = h->cfg.data_type;
        wa.precision = h->cfg.data_precision;
        wa.coh_ms = h->M;
        wa.K = h->K;
        wa.block_bytes = (size_t)h->N * h->M * h->cfg.data_type * h->cfg.data_precision;
        wa.base_freq_hz = h->d_base_freq;
        wa.fs_hz = h->cfg.fs_hz;
        wa.means = means;
        wa.x = h->d_x;
        CU(h->ops->launch_wipe(wa, (int)h->base_freq.size() * h->K, s));
        h->launches += 1;
    }
    CU(cudaEventRecord(h->ev[2], s));
    SearchArgs sa;
    sa.cc = h->d_cc;
    sa.x = h->d_x;
    sa.bin_base = h->d_bin_base;
    sa.bin_shift = h->d_bin_shift;
    sa.P = h->P; sa.B = h->B; sa.K = h->K;
    sa.row_first = h->row0; sa.n_rows = h->n_rows;
    sa.w = h->w;
    sa.cand = xchg ? xc.cand_all + (size_t)xc.sh.prn_first * xc.sh.freq_num_total + xc.sh.bin_first : h->d_cand;
    sa.cand_stride = xchg ? xc.sh.freq_num_total : h->B;
    sa.surface = h->d_surface;
    sa.scratch = h->d_scratch;
    sa.group_ctr = h->d_group_ctr;
    sa.row_slots = h->d_row_slots;
    sa.partial = h->d_partial;
    sa.part_ctr = h->d_group_ctr ? h->d_group_ctr + h->coop_groups : nullptr;
    sa.row_ticket = h->d_group_ctr ? h->d_group_ctr + (size_t)h->coop_groups * (1 + h->ops->R) : nullptr;
    sa.row_granular = h->d_partial ? 0 : 1;
#ifdef GNSS_TIMELINE
    static unsigned long long* d_timeline = nullptr;
    if (!d_timeline) { CU(cudaMalloc(&d_timeline, 16 * 16 * 32 * sizeof(unsigned long long))); }
    CU(cudaMemsetAsync(d_timeline, 0, 16 * 16 * 32 * sizeof(unsigned long long), s));
    sa.timeline = d_timeline;
    g_timeline = d_timeline;
#endif
    if (h->coop_groups > 0) {
        CU(cudaMemsetAsync(h->d_group_ctr, 0, (size_t)h->coop_groups * (2 + h->ops->R) * sizeof(unsigned), s));
        CU(h->ops->launch_search_coop(sa, h->coop_groups, s));
    } else if (h->l2x_clusters > 0) {
        CU(h->ops->launch_search_l2x(sa, h->l2x_clusters, s));
    } else {
        CU(h->ops->launch_search(sa, h->n_rows, s));
    }
    h->launches += 1;
    CU(cudaEventRecord(h->ev[3], s));
    if (xchg) {
        // candidates went straight into the root's table; a non-root shard now raises its "done" flag there,
        // the root runs K4 over the full table in gnssacq_xchg_finish
        if (!xc.is_root) {
            xchg_done_kernel<<<1, 1, 0, s>>>(xc.flags + 1 + xc.sh.rank, xc.epoch);
            CU(cudaGetLastError());
            h->launches += 1;
        }
        CU(cudaEventRecord(h->ev[4], s));
        return GNSSACQ_OK;
    }
    finalize_kernel<<<(h->P + 63) / 64, 64, 0, s>>>(h->d_cand, h->P, h->B, h->N, h->w, h->cfg.freq_min_hz,
                                                    h->cfg.freq_step_hz, h->cfg.snr_threshold_db, h->d_prn,
                                                    d_out ? d_out : h->d_res, h->B, h->bin0);
    CU(cudaGetLastError());
    h->d_last_rows = d_out ? d_out : h->d_res;
    h->launches += 1;
    CU(cudaEventRecord(h->ev[4], s));
    return GNSSACQ_OK;
}

int gnssacq_enqueue_device(gnssacq_handle* h, const void* d_if, size_t nbytes) {
    if (!h || !d_if) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    if (nbytes < h->if_bytes) return fail(h, GNSSACQ_ERR_SHORT_BUFFER, "IF block shorter than noncoh_blocks*coh_ms ms");
    CU(cudaSetDevice(h->device));
    h->have_h2d = false;
    CU(cudaEventRecord(h->ev[0], h->stream));
    return enqueue(h, d_if);
}

int gnssacq_enqueue_device_out(gnssacq_handle* h, const void* d_if, size_t nbytes, void* d_out_rows) {
    if (!h || !d_if || !d_out_rows) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    if (nbytes < h->if_bytes) return fail(h, GNSSACQ_ERR_SHORT_BUFFER, "IF block shorter than noncoh_blocks*coh_ms ms");
    CU(cudaSetDevice(h->device));
    h->have_h2d = false;
    CU(cudaEventRecord(h->ev[0], h->stream));
    return enqueue(h, d_if, (gnssacq_result*)d_out_rows);
}

int gnssacq_fetch_results(gnssacq_handle* h, gnssacq_result* out, gnssacq_stats* st) {
    if (!h || (!out && !st)) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    if (!h->d_last_rows) return fail(h, GNSSACQ_ERR_STATE, "no search has been enqueued on this handle");
    CU(cudaSetDevice(h->device));
    // rows of the LAST enqueued search, wherever it wrote them (its own table, or the caller's device buffer of
    // gnssacq_enqueue_device_out); out == NULL: timings only
    if (out) CU(cudaMemcpyAsync(h->h_res, h->d_last_rows, h->P * sizeof(gnssacq_result), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaEventRecord(h->ev[5], h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (out) std::memcpy(out, h->h_res, h->P * sizeof(gnssacq_result));
    if (st) {
        std::memset(st, 0, sizeof(*st));
        if (h->have_h2d) cudaEventElapsedTime(&st->h2d_ms, h->ev[0], h->ev[1]);
        cudaEventElapsedTime(&st->wipeoff_fft_ms, h->ev[1], h->ev[2]);
        cudaEventElapsedTime(&st->search_ms, h->ev[2], h->ev[3]);
        cudaEventElapsedTime(&st->finalize_ms, h->ev[3], h->ev[4]);
        cudaEventElapsedTime(&st->d2h_ms, h->ev[4], h->ev[5]);
        cudaEventElapsedTime(&st->total_ms, h->ev[0], h->ev[5]);
        st->kernel_launches = h->launches;
        st->n_bases = (int)h->base_freq.size();
        st->cluster_ctas = h->ops->R;
        st->threads = h->ops->T;
        st->exchange = h->coop_groups > 0 ? 3 : (h->l2x_clusters > 0 ? 2 : 1);
        st->resident_clusters = h->coop_groups > 0 ? h->coop_groups : h->l2x_clusters;
        st->work_split = h->d_partial ? 2 : 1;
    }
    return GNSSACQ_OK;
}

// ---------------------------------------------------------------- multi-GPU exchange through peer memory
int gnssacq_shard_plan(const gnssacq_config* full, int32_t rank, int32_t world, gnssacq_config* mine, gnssacq_shard* sh) {
    std::string why;
    if (!full || !mine || !sh || world < 1 || world > 62 || rank < 0 || rank >= world) return GNSSACQ_ERR_INVALID_ARG;
    if (int rc = validate(full, why)) return fail(nullptr, rc, why);
    if (full->bin_count != 0) return fail(nullptr, GNSSACQ_ERR_INVALID_ARG, "shard_plan wants the full grid (bin_count = 0)");
    std::memset(sh, 0, sizeof *sh);
    sh->rank = rank;
    sh->world = world;
    sh->n_prn_total = full->n_prn;
    for (int i = 0; i < full->n_prn; ++i) sh->prn_total[i] = full->prn[i];
    sh->freq_num_total = full->freq_num;
    if (full->n_prn >= world) {            // whole PRNs per shard (SURVEY 8e): the per-PRN work never leaves a GPU
        sh->prn_first = (int32_t)((long long)rank * full->n_prn / world);
        sh->prn_count = (int32_t)((long long)(rank + 1) * full->n_prn / world) - sh->prn_first;
        sh->bin_first = 0;
        sh->bin_count = full->freq_num;
    } else {                               // fewer PRNs than GPUs: every shard takes all PRNs and a range of bins
        sh->prn_first = 0;
        sh->prn_count = full->n_prn;
        const int q = full->freq_num / world, rem = full->freq_num % world;   // the first `rem` shards take one bin more,
        sh->bin_first = rank * q + (rank < rem ? rank : rem);                  // so the root always owns rows
        sh->bin_count = q + (rank < rem ? 1 : 0);
    }
    *mine = *full;
    mine->n_prn = sh->prn_count;
    for (int i = 0; i < GNSSACQ_MAX_PRN; ++i) mine->prn[i] = i < sh->prn_count ? full->prn[sh->prn_first + i] : 0;
    mine->bin_first = sh->bin_first;
    mine->bin_count = sh->bin_count;       // (== freq_num in the PRN-major case: the whole grid)
    return GNSSACQ_OK;                     // bin_count == 0 (more shards than bins): that shard has no rows and no handle
}

// rows [first, first + count) of shard `rank` under the row-granular plan: the root's share is (1000 + extra) / 1000
// of the others'; what is left goes to the others in equal parts, the first few taking one row more
static void plan_rows_range(long long total, int rank, int world, int extra_permille, long long& first, long long& count) {
    if (world == 1) { first = 0; count = total; return; }
    const long long wr = 1000 + extra_permille, wo = 1000;
    long long root = (total * wr + (wr + (world - 1) * wo) / 2) / (wr + (world - 1) * wo);
    if (root > total) root = total;
    if (root < 1 && total > 0) root = 1;                     // the root always owns rows (it runs K4)
    const long long rest = total - root, q = rest / (world - 1), rem = rest % (world - 1);
    if (rank == 0) { first = 0; count = root; return; }
    const long long r = rank - 1;
    first = root + r * q + (r < rem ? r : rem);
    count = q + (r < rem ? 1 : 0);
}
int gnssacq_shard_plan_rows(const gnssacq_config* full, int32_t rank, int32_t world, int32_t root_extra_permille,
                            gnssacq_config* mine, gnssacq_shard* sh) {
    std::string why;
    if (!full || !mine || !sh || world < 1 || world > 62 || rank < 0 || rank >= world) return GNSSACQ_ERR_INVALID_ARG;
    if (root_extra_permille <= -1000 || root_extra_permille > 100000) return fail(nullptr, GNSSACQ_ERR_INVALID_ARG, "root_extra_permille out of range");
    if (int rc = validate(full, why)) return fail(nullptr, rc, why);
    if (full->bin_count != 0 || full->row_count != 0) return fail(nullptr, GNSSACQ_ERR_INVALID_ARG, "shard_plan_rows wants the full grid (bin_count = row_count = 0)");
    std::memset(sh, 0, sizeof *sh);
    sh->rank = rank;
    sh->world = world;
    sh->n_prn_total = full->n_prn;
    for (int i = 0; i < full->n_prn; ++i) sh->prn_total[i] = full->prn[i];
    sh->freq_num_total = full->freq_num;
    sh->prn_first = 0;
    sh->prn_count = full->n_prn;
    sh->bin_first = 0;
    sh->bin_count = full->freq_num;
    sh->plan_rows = 1;
    sh->root_extra_permille = root_extra_permille;
    long long first, count;
    plan_rows_range((long long)full->n_prn * full->freq_num, rank, world, root_extra_permille, first, count);
    sh->row_first = (int32_t)first;
    sh->row_count = (int32_t)count;          // 0 (more shards than rows): that shard has no rows and no handle
    *mine = *full;
    mine->row_first = count > 0 ? sh->row_first : 0;
    mine->row_count = sh->row_count;
    return GNSSACQ_OK;
}

static int xchg_common(gnssacq_handle* h, const gnssacq_shard* sh) {
    if (!h || !sh) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    if (h->xc.on) return fail(h, GNSSACQ_ERR_STATE, "exchange already set up on this handle");
    if (sh->prn_count != h->P || sh->bin_count != h->B || sh->bin_first != h->bin0 || sh->freq_num_total != h->B_full ||
        (sh->plan_rows ? (sh->row_first != h->row0 || sh->row_count != h->n_rows) : (h->n_rows != h->P * h->B)))
        return fail(h, GNSSACQ_ERR_INVALID_ARG, "shard does not describe this handle (use gnssacq_shard_plan's config)");
    if (!h->d_comb) return fail(h, GNSSACQ_ERR_STATE, "the multi-GPU exchange needs the comb-row K1");
    CU(cudaSetDevice(h->device));
    h->xc.sh = *sh;
    for (cudaEvent_t* e : {&h->xc.ev_a, &h->xc.ev_b, &h->xc.ev_c, &h->xc.ev_d}) CU(cudaEventCreate(e));
    return GNSSACQ_OK;
}
static size_t xchg_if_span(const gnssacq_handle* h) { return (h->if_bytes + 255) / 256 * 256; }
static size_t xchg_cand_span(const gnssacq_shard* sh) {
    return ((size_t)sh->n_prn_total * sh->freq_num_total * sizeof(Candidate) + 255) / 256 * 256;
}
static void xchg_map(gnssacq_handle* h, unsigned char* block) {
    h->xc.block = block;
    h->xc.if_buf = block;
    h->xc.cand_all = reinterpret_cast<Candidate*>(block + xchg_if_span(h));
    h->xc.flags = reinterpret_cast<unsigned*>(block + xchg_if_span(h) + xchg_cand_span(&h->xc.sh));
    h->xc.on = true;
}

int gnssacq_xchg_root(gnssacq_handle* h, const gnssacq_shard* sh, void* ipc_out) {
    if (int rc = xchg_common(h, sh)) return rc;
    if (sh->rank != 0) return fail(h, GNSSACQ_ERR_INVALID_ARG, "the root is shard 0");
    unsigned char* block = nullptr;
    const size_t bytes = xchg_if_span(h) + xchg_cand_span(sh) + 64 * sizeof(unsigned);
    CU(cudaMalloc(&block, bytes));
    CU(cudaMemset(block, 0, bytes));
    h->xc.is_root = true;
    xchg_map(h, block);
    CU(cudaMalloc(&h->xc.d_prn_all, sh->n_prn_total * sizeof(int)));
    CU(cudaMemcpy(h->xc.d_prn_all, sh->prn_total, sh->n_prn_total * sizeof(int), cudaMemcpyHostToDevice));
    CU(cudaMalloc(&h->xc.d_res_all, sh->n_prn_total * sizeof(gnssacq_result)));
    CU(cudaMallocHost(&h->xc.h_res_all, sh->n_prn_total * sizeof(gnssacq_result)));
    if (ipc_out) {
        static_assert(sizeof(cudaIpcMemHandle_t) <= GNSSACQ_IPC_BYTES, "IPC handle size");
        cudaIpcMemHandle_t ih;
        CU(cudaIpcGetMemHandle(&ih, block));
        std::memset(ipc_out, 0, GNSSACQ_IPC_BYTES);
        std::memcpy(ipc_out, &ih, sizeof ih);
    }
    return GNSSACQ_OK;
}

int gnssacq_xchg_attach(gnssacq_handle* h, const gnssacq_shard* sh, const void* root_ipc) {
    if (!root_ipc) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    if (int rc = xchg_common(h, sh)) return rc;
    if (sh->rank == 0) return fail(h, GNSSACQ_ERR_INVALID_ARG, "shard 0 is the root (gnssacq_xchg_root)");
    cudaIpcMemHandle_t ih;
    std::memcpy(&ih, root_ipc, sizeof ih);
    void* p = nullptr;
    CU(cudaIpcOpenMemHandle(&p, ih, cudaIpcMemLazyEnablePeerAccess));      // the root's block, reachable over NVLink
    h->xc.ipc_opened = true;
    xchg_map(h, static_cast<unsigned char*>(p));
    return GNSSACQ_OK;
}

int gnssacq_xchg_attach_local(gnssacq_handle* h, const gnssacq_shard* sh, gnssacq_handle* root) {
    if (!root || !root->xc.on || !root->xc.is_root) return fail(h, GNSSACQ_ERR_INVALID_ARG, "root has no exchange block");
    if (int rc = xchg_common(h, sh)) return rc;
    if (sh->rank == 0) return fail(h, GNSSACQ_ERR_INVALID_ARG, "shard 0 is the root (gnssacq_xchg_root)");
    if (h->device != root->device) {
        int can = 0;
        CU(cudaDeviceCanAccessPeer(&can, h->device, root->device));
        if (!can) return fail(h, GNSSACQ_ERR_CUDA, "no peer access to the root's GPU");
        const cudaError_t e = cudaDeviceEnablePeerAccess(root->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CU(e);
        cudaGetLastError();
    }
    xchg_map(h, root->xc.block);
    return GNSSACQ_OK;
}

void* gnssacq_xchg_if_buffer(gnssacq_handle* h) { return (h && h->xc.on && h->xc.is_root) ? h->xc.if_buf : nullptr; }

int gnssacq_xchg_enqueue(gnssacq_handle* h, const void* host_if, size_t nbytes) {
    if (!h || !h->xc.on) return fail(h, GNSSACQ_ERR_STATE, "no exchange set up on this handle");
    if (host_if && !h->xc.is_root) return fail(h, GNSSACQ_ERR_INVALID_ARG, "only the root takes the IF block");
    if (host_if && nbytes < h->if_bytes) return fail(h, GNSSACQ_ERR_SHORT_BUFFER, "IF block shorter than noncoh_blocks*coh_ms ms");
    CU(cudaSetDevice(h->device));
    ++h->xc.epoch;
    CU(cudaEventRecord(h->ev[0], h->stream));
    h->have_h2d = false;
    if (host_if) {
        // page-locked caller memory goes to HBM as it is (the caller keeps it unchanged until gnssacq_xchg_fetch);
        // pageable memory is staged through the library's pinned buffer first (free again on return)
        cudaPointerAttributes pa{};
        const bool pinned = cudaPointerGetAttributes(&pa, host_if) == cudaSuccess && pa.type == cudaMemoryTypeHost;
        cudaGetLastError();
        if (pinned) CU(cudaMemcpyAsync(h->xc.if_buf, host_if, h->if_bytes, cudaMemcpyHostToDevice, h->stream));
        else if (int rc = stage_and_upload(h, h->xc.if_buf, host_if, h->stream)) return rc;
        h->have_h2d = true;
    }
    return enqueue(h, h->xc.if_buf, nullptr, true);       // non-root: a peer pointer -- K1a pulls it over NVLink
}

int gnssacq_xchg_finish(gnssacq_handle* h) {
    if (!h || !h->xc.on || !h->xc.is_root) return fail(h, GNSSACQ_ERR_STATE, "not the root of an exchange");
    CU(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    auto& xc = h->xc;
    CU(cudaEventRecord(xc.ev_c, s));
    if (xc.sh.world > 1) {
        unsigned long long has_rows = 0;
        for (int r = 1; r < xc.sh.world; ++r) {
            bool has;
            if (xc.sh.plan_rows) {
                long long first, count;
                plan_rows_range((long long)xc.sh.n_prn_total * xc.sh.freq_num_total, r, xc.sh.world, xc.sh.root_extra_permille, first, count);
                has = count > 0;
            } else {
                has = xc.sh.n_prn_total >= xc.sh.world || xc.sh.freq_num_total / xc.sh.world > 0 || r < xc.sh.freq_num_total % xc.sh.world;
            }
            if (has) has_rows |= 1ull << r;
        }
        xchg_wait_kernel<<<1, 64, 0, s>>>(xc.flags + 1, xc.sh.world, has_rows, xc.epoch, xc.flags + 63);
        CU(cudaGetLastError());
        h->launches += 1;
    }
    CU(cudaEventRecord(xc.ev_d, s));
    finalize_kernel<<<(xc.sh.n_prn_total + 63) / 64, 64, 0, s>>>(xc.cand_all, xc.sh.n_prn_total, xc.sh.freq_num_total, h->N, h->w,
                                                               h->cfg.freq_min_hz, h->cfg.freq_step_hz, h->cfg.snr_threshold_db,
                                                               xc.d_prn_all, xc.d_res_all, xc.sh.freq_num_total, 0);
    CU(cudaGetLastError());
    h->launches += 1;
    CU(cudaEventRecord(h->ev[4], s));
    return GNSSACQ_OK;
}

int gnssacq_xchg_fetch(gnssacq_handle* h, gnssacq_result* out, gnssacq_stats* st) {
    if (!h || !h->xc.on) return fail(h, GNSSACQ_ERR_STATE, "no exchange set up on this handle");
    if (out && !h->xc.is_root) return fail(h, GNSSACQ_ERR_INVALID_ARG, "rows are on the root");
    CU(cudaSetDevice(h->device));
    auto& xc = h->xc;
    const int n = xc.sh.n_prn_total;
    unsigned timed_out = 0;
    if (xc.is_root && out) CU(cudaMemcpyAsync(xc.h_res_all, xc.d_res_all, n * sizeof(gnssacq_result), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaEventRecord(h->ev[5], h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (xc.is_root) {
        CU(cudaMemcpy(&timed_out, xc.flags + 63, sizeof timed_out, cudaMemcpyDeviceToHost));
        if (timed_out) return fail(h, GNSSACQ_ERR_STATE, "a shard of the exchange did not answer within the time-out");
        if (out) std::memcpy(out, xc.h_res_all, n * sizeof(gnssacq_result));
    }
    if (st) {
        std::memset(st, 0, sizeof(*st));
        if (h->have_h2d) cudaEventElapsedTime(&st->h2d_ms, h->ev[0], h->ev[1]);
        cudaEventElapsedTime(&st->wipeoff_fft_ms, h->ev[1], h->ev[2]);
        cudaEventElapsedTime(&st->search_ms, h->ev[2], h->ev[3]);
        if (xc.is_root) {
            // (before gnssacq_xchg_finish these events are unrecorded: the queries fail and leave zeros)
            if (cudaEventElapsedTime(&st->gather_wait_ms, xc.ev_c, xc.ev_d) != cudaSuccess) st->gather_wait_ms = 0.f;
            if (cudaEventElapsedTime(&st->finalize_ms, xc.ev_d, h->ev[4]) != cudaSuccess) st->finalize_ms = 0.f;
            cudaEventElapsedTime(&st->d2h_ms, h->ev[4], h->ev[5]);
        } else {
            cudaEventElapsedTime(&st->if_pull_ms, xc.ev_a, xc.ev_b);
        }
        cudaEventElapsedTime(&st->total_ms, h->ev[0], h->ev[5]);
        cudaGetLastError();                    // a failed timing query must not surface at somebody's next launch check
        st->kernel_launches = h->launches;
        st->n_bases = (int)h->base_freq.size();
        st->cluster_ctas = h->ops->R;
        st->threads = h->ops->T;
        st->exchange = h->coop_groups > 0 ? 3 : (h->l2x_clusters > 0 ? 2 : 1);
        st->resident_clusters = h->coop_groups > 0 ? h->coop_groups : h->l2x_clusters;
        st->work_split = h->d_partial ? 2 : 1;
    }
    return GNSSACQ_OK;
}

int gnssacq_search_device(gnssacq_handle* h, const void* d_if, size_t nbytes, gnssacq_result* out, gnssacq_stats* st) {
    int rc = gnssacq_enqueue_device(h, d_if, nbytes);
    if (rc != GNSSACQ_OK) return rc;
    return gnssacq_fetch_results(h, out, st);
}

int gnssacq_search(gnssacq_handle* h, const void* if_samples, size_t nbytes, gnssacq_result* out, gnssacq_stats* st) {
    if (!h || !if_samples || !out) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    if (nbytes < h->if_bytes) return fail(h, GNSSACQ_ERR_SHORT_BUFFER, "IF block shorter than noncoh_blocks*coh_ms ms");
    CU(cudaSetDevice(h->device));
    CU(cudaEventRecord(h->ev[0], h->stream));
    if (int rc = stage_and_upload(h, h->d_if, if_samples, h->stream)) return rc;    // caller's buffer is free again after this
    h->have_h2d = true;
    int rc = enqueue(h, h->d_if);
    if (rc != GNSSACQ_OK) return rc;
    return gnssacq_fetch_results(h, out, st);
}

int gnssacq_search_multi(gnssacq_handle* const* hs, int32_t n, const void* if_samples, size_t nbytes, gnssacq_result* out) {
    if (!hs || n < 1 || !if_samples || !out) return GNSSACQ_ERR_INVALID_ARG;
    for (int i = 0; i < n; ++i) {
        gnssacq_handle* h = hs[i];
        if (!h) return GNSSACQ_ERR_INVALID_ARG;
        if (nbytes < h->if_bytes) return fail(h, GNSSACQ_ERR_SHORT_BUFFER, "IF block shorter than noncoh_blocks*coh_ms ms");
        CU(cudaSetDevice(h->device));
        CU(cudaEventRecord(h->ev[0], h->stream));
        if (int rc = stage_and_upload(h, h->d_if, if_samples, h->stream)) return rc;
        h->have_h2d = true;
        int rc = enqueue(h, h->d_if);
        if (rc != GNSSACQ_OK) return rc;
    }
    size_t off = 0;
    for (int i = 0; i < n; ++i) {
        int rc = gnssacq_fetch_results(hs[i], out + off, nullptr);
        if (rc != GNSSACQ_OK) return rc;
        off += (size_t)hs[i]->P;
    }
    return GNSSACQ_OK;
}

// BASELINE config 4 (periodic re-acquisition over a long recording) / SURVEY 8f-3 (IF ingest): n_windows
// independent searches.  Window i+1 is staged (host memcpy into pinned memory) and copied to HBM on a copy
// stream while window i is searched; two staging pairs, events in both directions, one D2H of all rows at the
// end.  Rows of window i are out[i*n_prn .. (i+1)*n_prn) and equal what gnssacq_search returns for that window.
// `fill(i, dst)` puts window i (if_bytes bytes) into pinned staging memory: a memcpy from the caller's window
// (gnssacq_sweep) or an fseek + fread straight from the recording (gnssacq_sweep_file).
extern "C++" {
template <class Fill>
static int sweep_impl(gnssacq_handle* h, int32_t n_windows, gnssacq_result* out, gnssacq_stats* st, Fill&& fill) {
    if (n_windows == 0) return GNSSACQ_OK;
    CU(cudaSetDevice(h->device));
    if (!h->copy_stream) {
        CU(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        CU(cudaMalloc(&h->d_if2, h->if_bytes));
        CU(cudaMallocHost(&h->h_if2, h->if_bytes));
        for (auto& e : h->ev_copied) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (auto& e : h->ev_consumed) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    if (h->sweep_cap < n_windows) {
        CU(cudaStreamSynchronize(h->stream));
        cudaFree(h->d_res_sweep);
        h->d_res_sweep = nullptr;
        h->sweep_cap = 0;
        CU(cudaMalloc(&h->d_res_sweep, (size_t)n_windows * h->P * sizeof(gnssacq_result)));
        h->sweep_cap = n_windows;
    }
    void* d_buf[2] = {h->d_if, h->d_if2};
    void* h_buf[2] = {h->h_if, h->h_if2};
    const auto t0 = std::chrono::steady_clock::now();
    int launches = 0;
    for (int i = 0; i < n_windows; ++i) {
        const int b = i & 1;
        if (i >= 2) CU(cudaEventSynchronize(h->ev_copied[b]));              // pinned buffer b has left for HBM
        { const int rc = fill(i, h_buf[b]); if (rc != GNSSACQ_OK) { cudaStreamSynchronize(h->stream); cudaStreamSynchronize(h->copy_stream); return rc; } }
        if (i >= 2) CU(cudaStreamWaitEvent(h->copy_stream, h->ev_consumed[b], 0));   // search i-2 is done with d_buf[b]
        else if (i == 0) CU(cudaStreamWaitEvent(h->copy_stream, h->ev[4], 0));      // d_if: after whatever this handle ran last
        // (i == 1: d_if2 / h_if2 are touched by sweeps only, and every sweep ends with a stream sync: no wait, so
        //  the copy of window 1 overlaps the search of window 0)
        CU(cudaMemcpyAsync(d_buf[b], h_buf[b], h->if_bytes, cudaMemcpyHostToDevice, h->copy_stream));
        CU(cudaEventRecord(h->ev_copied[b], h->copy_stream));
        CU(cudaStreamWaitEvent(h->stream, h->ev_copied[b], 0));
        h->have_h2d = false;
        CU(cudaEventRecord(h->ev[0], h->stream));
        int rc = enqueue(h, d_buf[b], h->d_res_sweep + (size_t)i * h->P);
        if (rc != GNSSACQ_OK) return rc;
        launches += h->launches;
        CU(cudaEventRecord(h->ev_consumed[b], h->stream));
    }
    CU(cudaMemcpyAsync(out, h->d_res_sweep, (size_t)n_windows * h->P * sizeof(gnssacq_result), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaEventRecord(h->ev[5], h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (st) {
        std::memset(st, 0, sizeof(*st));
        st->total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
        cudaEventElapsedTime(&st->wipeoff_fft_ms, h->ev[1], h->ev[2]);      // (of the last window)
        cudaEventElapsedTime(&st->search_ms, h->ev[2], h->ev[3]);
        cudaEventElapsedTime(&st->finalize_ms, h->ev[3], h->ev[4]);
        st->kernel_launches = launches;
        st->n_bases = (int)h->base_freq.size();
        st->cluster_ctas = h->ops->R;
        st->threads = h->ops->T;
        st->exchange = h->coop_groups > 0 ? 3 : (h->l2x_clusters > 0 ? 2 : 1);
        st->resident_clusters = h->coop_groups > 0 ? h->coop_groups : h->l2x_clusters;
        st->work_split = h->d_partial ? 2 : 1;
    }
    return GNSSACQ_OK;
}

}  // extern "C++"

int gnssacq_sweep(gnssacq_handle* h, const void* const* windows, int32_t n_windows, size_t nbytes_each,
                  gnssacq_result* out, gnssacq_stats* st) {
    if (!h || !windows || !out || n_windows < 0) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    if (nbytes_each < h->if_bytes) return fail(h, GNSSACQ_ERR_SHORT_BUFFER, "window shorter than noncoh_blocks*coh_ms ms");
    for (int i = 0; i < n_windows; ++i)
        if (!windows[i]) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL window");
    return sweep_impl(h, n_windows, out, st, [&](int i, void* dst) {
        std::memcpy(dst, windows[i], h->if_bytes);
        return (int)GNSSACQ_OK;
    });
}

// The same sweep straight from a recording: window j is what acquisition.m:27-34 reads with
// file.skip = skip_ms + j*epoch_ms, i.e. noncoh_blocks*coh_ms ms starting at byte
// (skip_ms + j*epoch_ms) * samples_per_ms * dataPrecision * dataType (SDR_main.m:17-23 run once per epoch).
// fseeko + fread go directly into the pinned staging buffers, overlapped with the previous window's search.
int gnssacq_sweep_file(gnssacq_handle* h, const char* path, int64_t skip_ms, int32_t epoch_ms, int32_t n_windows,
                       gnssacq_result* out, gnssacq_stats* st) {
    if (!h || !path || !out || n_windows < 0 || skip_ms < 0 || epoch_ms < 0) return fail(h, GNSSACQ_ERR_INVALID_ARG, "bad argument");
    FILE* f = std::fopen(path, "rb");
    if (!f) return fail(h, GNSSACQ_ERR_INVALID_ARG, "cannot open the recording");
    const long long ms_bytes = (long long)h->N * h->cfg.data_precision * h->cfg.data_type;
    const int rc = sweep_impl(h, n_windows, out, st, [&](int i, void* dst) {
        const long long off = (skip_ms + (long long)i * epoch_ms) * ms_bytes;               // acquisition.m:27
        if (fseeko(f, (off_t)off, SEEK_SET) != 0) return fail(h, GNSSACQ_ERR_SHORT_BUFFER, "seek past the end of the recording");
        if (std::fread(dst, 1, h->if_bytes, f) != h->if_bytes)                             // acquisition.m:28/34
            return fail(h, GNSSACQ_ERR_SHORT_BUFFER, "recording ends inside a window");
        return (int)GNSSACQ_OK;
    });
    std::fclose(f);
    return rc;
}

// Tracking correlators, SURVEY 8f-2.  gnssacq_track_load keeps a segment of the recording resident in HBM;
// gnssacq_correlate then runs one integration period for a batch of channels against it.
int gnssacq_track_load(gnssacq_handle* h, const void* if_samples, size_t nbytes) {
    if (!h || !if_samples || nbytes == 0) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    if (h->trk_cap < nbytes) {
        cudaFree(h->d_trk_raw);
        h->d_trk_raw = nullptr;
        h->trk_cap = h->trk_bytes = 0;
        if (cudaMalloc(&h->d_trk_raw, nbytes) != cudaSuccess) { cudaGetLastError(); return fail(h, GNSSACQ_ERR_NOMEM, "recording segment does not fit in HBM"); }
        h->trk_cap = nbytes;
    }
    if (!h->d_trk_ca) {
        std::vector<int8_t> ca((size_t)GNSSACQ_TRACK_MAX_PRN * 1023);
        for (int p = 1; p <= GNSSACQ_TRACK_MAX_PRN; ++p) ca_chips(p, ca.data() + (size_t)(p - 1) * 1023);
        CU(cudaMalloc(&h->d_trk_ca, ca.size()));
        CU(cudaMalloc(&h->d_trk_ch, kTrackMaxChannels * sizeof(gnssacq_channel)));
        CU(cudaMalloc(&h->d_trk_spacing, kTrackMaxTaps * sizeof(double)));
        CU(cudaMalloc(&h->d_trk_partial, (size_t)kTrackMaxChannels * kTrackChunks * kTrackMaxTaps * 2 * sizeof(double)));
        CU(cudaMalloc(&h->d_trk_out, (size_t)kTrackMaxChannels * kTrackMaxTaps * 2 * sizeof(double)));
        CU(cudaMalloc(&h->d_trk_mean, (size_t)kTrackMaxChannels * 2 * sizeof(double)));
        CU(cudaMallocHost(&h->h_trk_out, (size_t)kTrackMaxChannels * kTrackMaxTaps * 2 * sizeof(double)));
        CU(cudaMemcpyAsync(h->d_trk_ca, ca.data(), ca.size(), cudaMemcpyHostToDevice, h->stream));
        CU(cudaStreamSynchronize(h->stream));                        // `ca` is a temporary
    }
    CU(cudaMemcpyAsync(h->d_trk_raw, if_samples, nbytes, cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    h->trk_bytes = nbytes;
    return GNSSACQ_OK;
}

int gnssacq_correlate(gnssacq_handle* h, int32_t n_channels, const gnssacq_channel* ch, int32_t n_taps,
                      const double* spacing_chips, double* out_i, double* out_q) {
    if (!h || !ch || !spacing_chips || !out_i || !out_q) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    if (!h->d_trk_raw || !h->trk_bytes) return fail(h, GNSSACQ_ERR_STATE, "gnssacq_track_load first");
    if (n_channels < 1 || n_channels > kTrackMaxChannels || n_taps < 1 || n_taps > kTrackMaxTaps)
        return fail(h, GNSSACQ_ERR_INVALID_ARG, "1..64 channels, 1..32 taps");
    const gnssacq_config& c = h->cfg;
    const size_t bps = (size_t)c.data_type * c.data_precision;
    for (int i = 0; i < n_channels; ++i) {
        if (ch[i].prn < 1 || ch[i].prn > GNSSACQ_TRACK_MAX_PRN) return fail(h, GNSSACQ_ERR_INVALID_ARG, "PRN out of range");
        if (ch[i].num_samples < 1 || ch[i].sample_offset < 0 ||
            ((size_t)ch[i].sample_offset + (size_t)ch[i].num_samples) * bps > h->trk_bytes)
            return fail(h, GNSSACQ_ERR_SHORT_BUFFER, "Not enough raw data (trackingCT.m:107-111)");
        if (!(ch[i].code_hz > 0.0)) return fail(h, GNSSACQ_ERR_INVALID_ARG, "code_hz must be positive");
    }
    CU(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    CU(cudaMemcpyAsync(h->d_trk_ch, ch, n_channels * sizeof(gnssacq_channel), cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(h->d_trk_spacing, spacing_chips, n_taps * sizeof(double), cudaMemcpyHostToDevice, s));
    TrackArgs a;
    a.raw = h->d_trk_raw;
    a.data_type = c.data_type;
    a.precision = c.data_precision;
    a.fs_hz = c.fs_hz;
    a.ch = (const gnssacq_channel*)h->d_trk_ch;
    a.n_taps = n_taps;
    a.spacing = h->d_trk_spacing;
    a.ca = h->d_trk_ca;
    a.mean = nullptr;
    a.partial = h->d_trk_partial;
    if (c.data_precision == 2) {
        track_mean_kernel<<<n_channels, kTrackThreads, 0, s>>>(a, h->d_trk_mean);
        a.mean = h->d_trk_mean;
    }
    const dim3 grid(kTrackChunks, (unsigned)n_channels, (unsigned)((n_taps + kTrackTapsPerThread - 1) / kTrackTapsPerThread));
    correlate_kernel<<<grid, kTrackThreads, 0, s>>>(a);
    const int n_elems = n_channels * n_taps * 2;
    correlate_finish_kernel<<<(n_elems + 127) / 128, 128, 0, s>>>(h->d_trk_partial, n_taps, n_elems, h->d_trk_out);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h->h_trk_out, h->d_trk_out, n_elems * sizeof(double), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    for (int i = 0; i < n_channels * n_taps; ++i) { out_i[i] = h->h_trk_out[2 * i]; out_q[i] = h->h_trk_out[2 * i + 1]; }
    return GNSSACQ_OK;
}

int gnssacq_loop_params_default(gnssacq_loop_params* p) {
    if (!p) return GNSSACQ_ERR_INVALID_ARG;
    p->dll_bw = 2.0; p->dll_damp = 0.707; p->dll_gain = 0.1;        // initParameters.m:60-62
    p->pll_bw = 15.0; p->pll_damp = 0.707; p->pll_gain = 0.25;      // initParameters.m:63-65
    p->spacing_chips = 0.5;                                          // initParameters.m:59
    return GNSSACQ_OK;
}

int gnssacq_track(gnssacq_handle* h, int32_t n_channels, const gnssacq_channel* start, const gnssacq_loop_params* loops,
                  int32_t n_periods, gnssacq_track_record* out) {
    if (!h || !start || !loops || !out) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    if (!h->d_trk_raw || !h->trk_bytes) return fail(h, GNSSACQ_ERR_STATE, "gnssacq_track_load first");
    if (n_channels < 1 || n_channels > kTrackMaxChannels || n_periods < 1)
        return fail(h, GNSSACQ_ERR_INVALID_ARG, "1..64 channels, at least one period");
    if (!(loops->dll_bw > 0 && loops->dll_damp > 0 && loops->dll_gain > 0 && loops->pll_bw > 0 && loops->pll_damp > 0 &&
          loops->pll_gain > 0 && loops->spacing_chips > 0 && loops->spacing_chips < 1.0))
        return fail(h, GNSSACQ_ERR_INVALID_ARG, "loop parameters must be positive, spacing inside one chip");
    const gnssacq_config& c = h->cfg;
    const size_t bps = (size_t)c.data_type * c.data_precision;
    const long long total = (long long)(h->trk_bytes / bps);
    for (int i = 0; i < n_channels; ++i) {
        if (start[i].prn < 1 || start[i].prn > GNSSACQ_TRACK_MAX_PRN) return fail(h, GNSSACQ_ERR_INVALID_ARG, "PRN out of range");
        if (start[i].sample_offset < 0 || start[i].sample_offset >= total) return fail(h, GNSSACQ_ERR_SHORT_BUFFER, "channel starts outside the loaded segment");
        if (!(start[i].code_hz > 0.0)) return fail(h, GNSSACQ_ERR_INVALID_ARG, "code_hz must be positive");
    }
    CU(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const size_t n_rec = (size_t)n_channels * n_periods;
    if (h->trk_rec_cap < n_rec) {
        CU(cudaStreamSynchronize(s));
        cudaFree(h->d_trk_rec);
        h->d_trk_rec = nullptr;
        h->trk_rec_cap = 0;
        CU(cudaMalloc(&h->d_trk_rec, n_rec * sizeof(gnssacq_track_record)));
        h->trk_rec_cap = n_rec;
    }
    if (!h->d_trk_status) CU(cudaMalloc(&h->d_trk_status, sizeof(int)));
    CU(cudaMemsetAsync(h->d_trk_status, 0, sizeof(int), s));
    CU(cudaMemsetAsync(h->d_trk_rec, 0, n_rec * sizeof(gnssacq_track_record), s));
    CU(cudaMemcpyAsync(h->d_trk_ch, start, n_channels * sizeof(gnssacq_channel), cudaMemcpyHostToDevice, s));
    LoopArgs a;
    a.raw = h->d_trk_raw;
    a.total_samples = total;
    a.data_type = c.data_type;
    a.precision = c.data_precision;
    a.fs_hz = c.fs_hz;
    a.code_basis_hz = c.code_hz;
    a.start = (const gnssacq_channel*)h->d_trk_ch;
    a.ca = h->d_trk_ca;
    a.lp = *loops;
    a.n_periods = n_periods;
    a.out = h->d_trk_rec;
    a.status = h->d_trk_status;
    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3((unsigned)(n_channels * kLoopCtas), 1, 1);
    lc.blockDim = dim3(kLoopThreads, 1, 1);
    lc.dynamicSmemBytes = 0;
    lc.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = kLoopCtas;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    lc.attrs = attr;
    lc.numAttrs = 1;
    CU(cudaLaunchKernelEx(&lc, track_loop_kernel, a));
    int status = 0;
    CU(cudaMemcpyAsync(out, h->d_trk_rec, n_rec * sizeof(gnssacq_track_record), cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(&status, h->d_trk_status, sizeof(int), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    if (status) return fail(h, GNSSACQ_ERR_SHORT_BUFFER, "Not enough raw data (trackingCT.m:107-111): a channel ran past the loaded segment");
    return GNSSACQ_OK;
}

int gnssacq_read_surface(gnssacq_handle* h, int32_t prn_index, float* out) {
    if (!h || !out || prn_index < 0 || prn_index >= h->P) return fail(h, GNSSACQ_ERR_INVALID_ARG, "bad argument");
    if (!h->d_surface) return fail(h, GNSSACQ_ERR_STATE, "handle was created without keep_surface");
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    const size_t n = (size_t)h->B * h->N;
    CU(cudaMemcpy(out, h->d_surface + (size_t)prn_index * n, n * sizeof(float), cudaMemcpyDeviceToHost));
    return GNSSACQ_OK;
}

int gnssacq_fine_frequency(gnssacq_handle* h, const void* if_long, size_t nbytes, int32_t L, int32_t n_sv,
                           const int32_t* prn, const int32_t* code_phase, double* out_hz) {
    if (!h || !if_long || !prn || !code_phase || !out_hz) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    if (n_sv == 0) return GNSSACQ_OK;
    if (L < 1 || L > 16 || n_sv < 0) return fail(h, GNSSACQ_ERR_INVALID_ARG, "L must be 1..16, n_sv >= 0");
    const gnssacq_config& c = h->cfg;
    const size_t bps = (size_t)c.data_type * c.data_precision;
    const size_t need = (size_t)(L + 1) * h->N * bps;
    if (nbytes < need) return fail(h, GNSSACQ_ERR_SHORT_BUFFER, "fine-frequency stage needs (L+1) ms of IF (acquisition.m:91/96)");
    for (int i = 0; i < n_sv; ++i)
        if (prn[i] < 1 || prn[i] > 51 || code_phase[i] < 0 || code_phase[i] >= h->N)
            return fail(h, GNSSACQ_ERR_INVALID_ARG, "PRN or code phase out of range");
    CU(cudaSetDevice(h->device));
    cudaStream_t s = h->stream;
    const int N = h->N, K = h->K;
    const long long LN = (long long)L * N, F = LN * K;                          // acquisition.m:108
    if (F > 0xFFFFFFFFll) return fail(h, GNSSACQ_ERR_INVALID_ARG, "fftlength exceeds 2^32");

    constexpr int kChunk = 4;                                                   // SVs per pass (scratch ~0.4 GB at N = 58 000)
    auto cleanup = [&]() {};
#define CUF(call)                                                                                        \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess) { cleanup(); return fail(h, GNSSACQ_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); } \
    } while (0)
    if (h->fine_L != L) {
        // (re)build the per-L scratch: chip index of sample t (acquisition.m:104-105, same double arithmetic)
        cudaFree(h->d_fine_raw); cudaFree(h->d_fine_chip); cudaFree(h->d_fine_u); cudaFree(h->d_fine_ca);
        cudaFree(h->d_fine_start); cudaFree(h->d_fine_best);
        h->d_fine_raw = nullptr; h->d_fine_chip = nullptr; h->d_fine_u = nullptr; h->d_fine_ca = nullptr;
        h->d_fine_start = nullptr; h->d_fine_best = nullptr;
        h->fine_L = 0;
        std::vector<uint16_t> chip((size_t)LN);
        const double inv_fs = 1.0 / c.fs_hz, inv_fc = 1.0 / c.code_hz;
        const double codelength = c.code_hz * 1e-3;                             // initParameters.m:47
        for (long long t = 1; t <= LN; ++t) {
            const double idx = std::floor((inv_fs * (double)t) / inv_fc);
            chip[(size_t)(t - 1)] = (uint16_t)std::fmod(idx, codelength);       // rem(.)+1, 0-based here
        }
        CUF(cudaMalloc(&h->d_fine_raw, need));
        CUF(cudaMalloc(&h->d_fine_chip, chip.size() * sizeof(uint16_t)));
        CUF(cudaMalloc(&h->d_fine_ca, (size_t)GNSSACQ_MAX_PRN * 1023));
        CUF(cudaMalloc(&h->d_fine_start, GNSSACQ_MAX_PRN * sizeof(int)));
        CUF(cudaMalloc(&h->d_fine_best, GNSSACQ_MAX_PRN * sizeof(unsigned long long)));
        CUF(cudaMalloc(&h->d_fine_u, (size_t)kChunk * K * L * N * sizeof(cf)));
        CUF(cudaMemcpyAsync(h->d_fine_chip, chip.data(), chip.size() * sizeof(uint16_t), cudaMemcpyHostToDevice, s));
        CUF(cudaStreamSynchronize(s));                                          // `chip` is a temporary
        h->fine_L = L;
    }
    if (n_sv > GNSSACQ_MAX_PRN) return fail(h, GNSSACQ_ERR_INVALID_ARG, "too many SVs");
    void* d_raw = h->d_fine_raw; uint16_t* d_chip = h->d_fine_chip; int8_t* d_ca = h->d_fine_ca; int* d_start = h->d_fine_start;
    cf* d_u = h->d_fine_u; unsigned long long* d_best = h->d_fine_best;
    std::vector<int8_t> ca((size_t)n_sv * 1023);
    std::vector<int> start(n_sv);
    for (int i = 0; i < n_sv; ++i) {
        ca_chips(prn[i], ca.data() + (size_t)i * 1023);
        start[i] = N - code_phase[i] - 1;                                       // acquisition.m:106 (1-based N-codedelay)
    }
    const int chunk = n_sv < kChunk ? n_sv : kChunk;
    CUF(cudaMemcpyAsync(d_raw, if_long, need, cudaMemcpyHostToDevice, s));
    CUF(cudaMemcpyAsync(d_ca, ca.data(), ca.size(), cudaMemcpyHostToDevice, s));
    CUF(cudaMemcpyAsync(d_start, start.data(), n_sv * sizeof(int), cudaMemcpyHostToDevice, s));
    CUF(cudaMemsetAsync(d_best, 0, n_sv * sizeof(unsigned long long), s));
    const double* means = nullptr;
    if (c.data_precision == 2) {                                                // acquisition.m:92-94
        const long long pairs = (long long)(L + 1) * N;
        CUF(cudaMemsetAsync(h->d_sums, 0, 2 * sizeof(long long), s));
        sum_int16_kernel<<<296, 256, 0, s>>>((const int16_t*)d_raw, pairs, h->d_sums);
        means_kernel<<<1, 1, 0, s>>>(h->d_sums, pairs, h->d_means);
        CUF(cudaGetLastError());
        means = h->d_means;
    }
    for (int first = 0; first < n_sv; first += chunk) {
        const int n = (n_sv - first) < chunk ? (n_sv - first) : chunk;
        FineArgs fa;
        fa.raw = d_raw; fa.chip = d_chip; fa.ca = d_ca + (size_t)first * 1023; fa.start = d_start + first;
        fa.means = means; fa.data_type = c.data_type; fa.precision = c.data_precision;
        fa.L = L; fa.K = K; fa.F = F; fa.u = d_u;
        CUF(h->ops->launch_fine(fa, n * K * L, s));
        dim3 grid((unsigned)((N + 255) / 256), (unsigned)K, (unsigned)n);
        fine_combine_kernel<<<grid, 256, 0, s>>>(d_u, K, L, N, F, c.data_type == 2 ? 1 : 0, d_best + first);
        CUF(cudaGetLastError());
    }
    std::vector<unsigned long long> best(n_sv);
    CUF(cudaMemcpyAsync(best.data(), d_best, n_sv * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    CUF(cudaStreamSynchronize(s));
#undef CUF
    for (int i = 0; i < n_sv; ++i) {
        const double idx = (double)(0xFFFFFFFFu - (unsigned)(best[i] & 0xFFFFFFFFull)) + 1.0;   // 1-based FreqPeakIndex (:116)
        double fine = idx * (c.fs_hz / (double)F);                                                // :117
        if (c.data_type == 2) fine = -idx * (c.fs_hz / (double)F) + c.fs_hz / 2.0;                // :119
        out_hz[i] = fine;
    }
    return GNSSACQ_OK;
}

int gnssacq_fp32_peak_tflops(int32_t device, double* out_tflops) {
    gnssacq_handle* h = nullptr;
    if (!out_tflops) return GNSSACQ_ERR_INVALID_ARG;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail(nullptr, GNSSACQ_ERR_NO_DEVICE, "no CUDA device"); }
    if (device < 0) cudaGetDevice(&device);
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    float* d = nullptr;
    CU(cudaMalloc(&d, 4));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    const int blocks = prop.multiProcessorCount * 8, iters = 4096;
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        CU(cudaEventRecord(e0, 0));
        fma_peak_kernel<<<blocks, 256>>>(d, iters, 1.0000001f, 1e-7f);
        CU(cudaEventRecord(e1, 0));
        CU(cudaEventSynchronize(e1));
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, e0, e1));
        const double flops = 2.0 * 16.0 * 8.0 * (double)iters * 256.0 * (double)blocks;
        if (rep > 0 && ms > 0.f) best = std::max(best, flops / (ms * 1e-3) * 1e-12);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d);
    *out_tflops = best;
    return GNSSACQ_OK;
}

int gnssacq_fft_forward(gnssacq_handle* h, const float* in, float* out) {
    if (!h || !in || !out) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    CU(cudaSetDevice(h->device));
    const size_t bytes = (size_t)h->N * sizeof(cf);
    if (!h->d_fft_in) {
        CU(cudaMalloc(&h->d_fft_in, bytes));
        CU(cudaMalloc(&h->d_fft_out, bytes));
    }
    CU(cudaMemcpyAsync(h->d_fft_in, in, bytes, cudaMemcpyHostToDevice, h->stream));
    NaturalArgs a{h->d_fft_in, h->d_fft_out};
    CU(h->ops->launch_natural(a, 1, h->stream));
    CU(cudaMemcpyAsync(out, h->d_fft_out, bytes, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return GNSSACQ_OK;
}

}  // extern "C"
