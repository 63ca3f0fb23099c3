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
#if defined(__x86_64__)
#include <emmintrin.h>
#endif

#include "gnss_host.h"

using namespace gnss;

#define GNSSACQ_VERSION_STR "gnssacq 0.2.0 (sm_100a)"

namespace {

thread_local std::string g_create_error;

// ---------------------------------------------------------------- C/A code (generateCAcode.m)
const int kG2Delay[51] = {5,   6,   7,   8,   17,  18,  139, 140, 141, 251, 252, 254, 255, 256, 257, 258, 469,
                          470, 471, 472, 473, 474, 509, 512, 513, 514, 515, 516, 859, 860, 861, 862, 145, 175,
                          52,  21,  237, 235, 886, 657, 634, 762, 355, 1012, 176, 603, 130, 359, 595, 68,  386};

// K1a (r02): re-order the raw IF block (acquisition.m:27-38's bytes, as read) into 16 comb rows per millisecond:
// out[ms][rho][m] = sample 16*m + rho of that ms (see Wipe2Args).  Input is read with 16-byte vector loads
// (8 packed int8 I/Q samples per load, fully coalesced) -- `raw` may be a PEER pointer: on ranks > 0 of a
// multi-GPU search this kernel is what pulls the IF block out of rank 0's HBM over NVLink, so no separate
// broadcast is needed.  Until the root's "IF ready" flag, which this kernel waits for, that buffer holds whatever it
// held before (the previous block, a half-finished upload), so nothing else on such a rank reads `raw`: the int16
// means are summed from the comb copy.  A CTA handles TM consecutive m of one ms (TM*16 samples, contiguous in the input).
constexpr int kCombTM = 256;
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

namespace gnss {

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


int fail(gnssacq_handle* h, int code, const std::string& msg) {
    if (h) h->err = msg;
    g_create_error = msg;
    return code;
}

int cuda_fail(gnssacq_handle* h, cudaError_t e, const char* call, int oom_code) {
    cudaGetLastError();                    // the error must not surface at the next launch check
    return fail(h, e == cudaErrorMemoryAllocation ? oom_code : GNSSACQ_ERR_CUDA, std::string(call) + ": " + cudaGetErrorString(e));
}

void fill_engine_stats(const gnssacq_handle* h, gnssacq_stats* st) {
    st->n_bases = (int)h->base_freq.size();
    st->cluster_ctas = h->ops->R;
    st->threads = h->ops->T;
    st->exchange = h->xmode;
    st->resident_clusters = h->used_groups;
    st->work_split = h->used_split;
}

// How the persistent search kernels (exchange 2 / 3) deal out one row set: the resident groups, and whether the
// cooperative kernel hands the tail out block by block.  Chosen per row set: at create for the handle's own rows, and
// again for every set of Doppler windows (160 rows on 37 groups want the block tail where 1 312 rows do not).
struct Schedule { int groups = 0; bool by_blocks = false; };

// Exchange 2 / 3: `n` groups made resident, but never more than there is work for.  The cooperative kernel deals out
// single blocks of a row (block-granular tail) or whole rows; the clustered one whole rows.
// Block-granular tail (see search_kernel_coop): needs K-1 power planes per group (150 MB at the reference's sizes) --
// not possible above 2 GiB or beyond the kernel's 32-bit unit arithmetic.  It costs 0.15-0.4 row times (publishing and
// adding the planes), so work_split 0 (auto) uses it only where whole rows would leave >= 4 % of the last round's
// group-time idle (measured r01: pays for <= 8 PRNs at N = 26 000, <= 4 PRNs at N = 58 000, not for 32).  Results are
// identical either way.  rows == 0: nothing to launch.
int plan_schedule(gnssacq_handle* h, long long rows, Schedule& sc) {
    sc = Schedule{};
    if (h->xmode == 1 || rows == 0) return GNSSACQ_OK;
    const VariantOps* ops = h->ops;
    const int split = h->cfg.work_split;
    int n = h->xmode == 3 ? ops->max_groups_coop() : ops->max_clusters_l2x();
    bool by_blocks = h->xmode == 3 && split != 1 && h->K > 1 && (unsigned long long)n * n * h->K < (1ull << 32) &&
                     (unsigned long long)n * (h->K - 1) * ops->partial_bytes_per_group <= (2ull << 30);
    if (by_blocks && split == 0) {
        const long long rounds = (rows + n - 1) / n;
        by_blocks = (double)(rounds * n - rows) >= 0.04 * (double)(rounds * n);
    }
    const long long max_useful = by_blocks ? rows * h->K : rows;
    if (n > max_useful) n = (int)max_useful;
    if (n <= 0) return fail(h, GNSSACQ_ERR_CUDA, "persistent search kernel cannot be made resident on this device");
    sc.groups = n;
    sc.by_blocks = by_blocks;
    return GNSSACQ_OK;
}

// Makes `sc` the handle's schedule.  Per-group buffers are only ever grown, and the hand-over planes are built the
// first time a schedule asks for the block-granular tail; what is built goes into the handle only once every call
// has succeeded, so a failure leaves the previous schedule whole.  Any search still using the old buffers must have
// finished (create: none yet; gnssacq_set_doppler_windows waits for the stream).
int use_schedule(gnssacq_handle* h, const Schedule& sc) {
    const VariantOps* ops = h->ops;
    const size_t n = (size_t)sc.groups;
    DevPtr<cf> scratch;
    DevPtr<unsigned> ctr;
    DevPtr<Candidate> slots;
    DevPtr<float> partial;
    const bool grow = sc.groups > h->group_cap;
    if (grow) {
        CU(alloc(scratch, n * ops->scratch_bytes_per_cluster), GNSSACQ_ERR_NOMEM);
        // the padding columns of the exchange layout are never written: they must read as exact zeros
        CU(cudaMemsetAsync(scratch.get(), 0, n * ops->scratch_bytes_per_cluster, h->stream), GNSSACQ_ERR_NOMEM);
        CU(alloc(ctr, n * (2 + ops->R) * sizeof(unsigned)), GNSSACQ_ERR_NOMEM);     // group barriers + hand-over counters + row tickets
        CU(alloc(slots, n * ops->R * sizeof(Candidate)), GNSSACQ_ERR_NOMEM);
    }
    const bool planes = sc.by_blocks && sc.groups > h->partial_groups;
    if (planes) CU(alloc(partial, n * (h->K - 1) * ops->partial_bytes_per_group), GNSSACQ_ERR_NOMEM);
    if (grow) {
        h->d_scratch = std::move(scratch);
        h->d_group_ctr = std::move(ctr);
        h->d_row_slots = std::move(slots);
        h->group_cap = sc.groups;
    }
    if (planes) {
        h->d_partial = std::move(partial);
        h->partial_groups = sc.groups;
    }
    h->coop_groups = h->xmode == 3 ? sc.groups : 0;
    h->l2x_clusters = h->xmode == 2 ? sc.groups : 0;
    h->by_blocks = sc.by_blocks;
    return GNSSACQ_OK;
}

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

// Doppler bins -> (base transform, shift in FFT bins): f_b = f_base + s * (Fs/NF)   (SURVEY A.7)
// A padded shape (N < NF) with an M-ms fold also needs f_b - f_base to be a whole number of Fs/N: the carrier
// advances by (f_b - f_base)*N/Fs cycles from one ms of the fold to the next, and only a whole number of cycles
// leaves the folded block a plain shift of the base's (for N = NF both conditions are the same).
void plan_bins(gnssacq_handle* h) {
    const gnssacq_config& c = h->cfg;
    const double df = c.fs_hz / (double)h->NF, dms = c.fs_hz / (double)h->N;
    const bool fold = h->M > 1 && h->NF != h->N;
    h->bin_base.assign(h->B, 0);
    h->bin_shift.assign(h->B, 0);
    h->base_freq.clear();
    for (int b = 0; b < h->B; ++b) {
        const double f = c.if_hz + (c.freq_min_hz + c.freq_step_hz * (double)b);     // acquisition.m:42-43
        int found = -1, shift = 0;
        for (size_t i = 0; i < h->base_freq.size(); ++i) {
            const double r = (f - h->base_freq[i]) / df;
            const double rr = std::nearbyint(r);
            const double q = (f - h->base_freq[i]) / dms;
            if (std::fabs(r - rr) * df < 1e-6 && std::fabs(rr) < (double)(h->NF / 2) &&
                (!fold || std::fabs(q - std::nearbyint(q)) * dms < 1e-6)) {
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

// For a handle that does not search all of its P x B rows: the cells of its candidate table that no search writes must
// not win K4's maximum (peak -1 never does), and the rows of the kept surface that it never searches read as zeros.
// Synchronous (the sentinel table is a temporary).
int clear_unsearched(gnssacq_handle* h) {
    std::vector<Candidate> none((size_t)h->P * h->B, Candidate{-1.f, 0, 0.0, 0.0});
    CU(cudaMemcpyAsync(h->d_cand.get(), none.data(), none.size() * sizeof(Candidate), cudaMemcpyHostToDevice, h->stream), GNSSACQ_ERR_NOMEM);
    if (h->d_surface) CU(cudaMemsetAsync(h->d_surface.get(), 0, (size_t)h->P * h->B * h->N * sizeof(float), h->stream), GNSSACQ_ERR_NOMEM);
    CU(cudaStreamSynchronize(h->stream), GNSSACQ_ERR_NOMEM);
    return GNSSACQ_OK;
}

// The transform length NF for N samples per ms: N itself when it is a built 2000*Q, otherwise the smallest built
// length >= 2N - 1, into which each ms is zero-padded (the circular correlation of N lags then never wraps).
// 0: neither (N > 29 000 and not built).
int transform_length(int n) {
    static const int kBuilt[] = {6000, 26000, 58000};         // 2000*Q, Q = 3, 13, 29 (gnss_q*.cu)
    if (n <= 0) return 0;
    for (int b : kBuilt)
        if (n == b) return n;
    for (int b : kBuilt)
        if ((long long)b >= 2ll * n - 1) return b;
    return 0;
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
    if (transform_length(c->samples_per_ms) == 0) {
        why = "samples_per_ms must be a built transform length (6000, 26000, 58000) or at most 29000 "
              "(zero-padded into the smallest built length >= 2*samples_per_ms - 1)";
        return GNSSACQ_ERR_UNSUPPORTED_N;
    }
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

int stage_and_upload(gnssacq_handle* h, void* d_dst, const void* host_src, cudaStream_t s) {
    // (Helper threads for the host copy were built and measured in r02: three helpers claiming 128 kB pieces next to the
    // caller's thread made the upload of the 2.32 MB block SLOWER, 0.30 ms against 0.185 ms, on the 16-core host of the
    // GPU box -- waking sleeping threads costs more than the 0.1 ms they could save.  profiles/r02/time_e2e_staging_helpers_v16.txt)
    constexpr size_t kChunk = 512 << 10;
    const unsigned char* src = static_cast<const unsigned char*>(host_src);
    unsigned char* pin = static_cast<unsigned char*>(h->h_if.get());
    if (h->ev_upload) CU(cudaEventSynchronize(h->ev_upload.get()));      // an earlier (asynchronous) upload still reads h_if
    else CU(create(h->ev_upload, cudaEventDisableTiming));
    for (size_t off = 0; off < h->if_bytes; off += kChunk) {
        const size_t n = std::min(kChunk, h->if_bytes - off);
        copy_to_staging(pin + off, src + off, n);
        CU(cudaMemcpyAsync(static_cast<unsigned char*>(d_dst) + off, pin + off, n, cudaMemcpyHostToDevice, s));
    }
    CU(cudaEventRecord(h->ev_upload.get(), s));
    return GNSSACQ_OK;
}

// int16 per-component means of n_pairs samples into h->d_means, summed over the `scan` (I, Q) pairs at `src`
// (two launches)
static int launch_means(gnssacq_handle* h, const void* src, long long scan, long long n_pairs, cudaStream_t s) {
    CU(cudaMemsetAsync(h->d_sums.get(), 0, 2 * sizeof(long long), s));
    sum_int16_kernel<<<296, 256, 0, s>>>((const int16_t*)src, scan, h->d_sums.get());
    means_kernel<<<1, 1, 0, s>>>(h->d_sums.get(), n_pairs, h->d_means.get());
    CU(cudaGetLastError());
    return GNSSACQ_OK;
}

int enqueue(gnssacq_handle* h, const void* d_if, gnssacq_result* d_out, bool xchg) {
    cudaStream_t s = h->stream;
    h->launches = 0;
    auto& xc = h->xc;
    if (xchg && !h->d_comb) return fail(h, GNSSACQ_ERR_STATE, "the multi-GPU exchange needs the comb-row K1 (shared memory too small for this shape)");
    CU(cudaEventRecord(h->ev[1].get(), s));
    // int16 (acquisition.m:30-32): per-component means of the N*K*M samples
    const double* means = h->cfg.data_precision == 2 ? h->d_means.get() : nullptr;
    const long long n_pairs = (long long)h->N * h->K * h->M;
    if (h->d_comb) {
        const int bps = h->cfg.data_type * h->cfg.data_precision;
        const int rows = h->N / 16, tiles = (rows + kCombTM - 1) / kCombTM;
        if (xchg) CU(cudaEventRecord(xc.ev_a.get(), s));
        comb_kernel<<<h->K * h->M * tiles, 256, (size_t)kCombTM * (4 * bps + 1) * 4, s>>>(
            (const unsigned char*)d_if, h->d_comb.get(), rows, bps, h->comb_pitch, tiles,
            (xchg && xc.is_root) ? xc.flags : nullptr, (xchg && !xc.is_root) ? xc.flags : nullptr, xc.epoch,
            xchg ? xc.flags + 63 : nullptr);
        CU(cudaGetLastError());
        if (xchg) CU(cudaEventRecord(xc.ev_b.get(), s));
        // from the comb copy, not `d_if`: on a non-root shard that is the root's buffer (see comb_kernel).
        // [K*M*16 rows][pitch bytes], one (I, Q) pair per 4 bytes; the pad bytes are zero (memset at create, never written)
        if (means) {
            if (int rc = launch_means(h, h->d_comb.get(), (long long)h->K * h->M * 16 * h->comb_pitch / 4, n_pairs, s)) return rc;
            h->launches += 2;
        }
        Wipe2Args w2;
        w2.comb = h->d_comb.get();
        w2.pitch = h->comb_pitch;
        w2.bps = bps;
        w2.coh_ms = h->M;
        w2.K = h->K;
        w2.base_w = h->d_base_w.get();
        w2.means = means;
        w2.x = h->d_x.get();
        CU(h->ops->launch_wipe2(w2, (int)h->base_freq.size() * h->K, s));
        h->launches += 2;
    } else {
        // (K1 v1 is never used by the multi-GPU exchange: `d_if` is this handle's own, complete block)
        if (means) {
            if (int rc = launch_means(h, d_if, n_pairs, n_pairs, s)) return rc;
            h->launches += 2;
        }
        WipeArgs wa;
        wa.raw = d_if;
        wa.data_type = h->cfg.data_type;
        wa.precision = h->cfg.data_precision;
        wa.coh_ms = h->M;
        wa.K = h->K;
        wa.block_bytes = (size_t)h->N * h->M * h->cfg.data_type * h->cfg.data_precision;
        wa.n_ms = h->N;
        wa.base_freq_hz = h->d_base_freq.get();
        wa.fs_hz = h->cfg.fs_hz;
        wa.means = means;
        wa.x = h->d_x.get();
        CU(h->ops->launch_wipe(wa, (int)h->base_freq.size() * h->K, s));
        h->launches += 1;
    }
    CU(cudaEventRecord(h->ev[2].get(), s));
    SearchArgs sa;
    sa.cc = h->d_cc.get();
    sa.x = h->d_x.get();
    sa.bin_base = h->d_bin_base.get();
    sa.bin_shift = h->d_bin_shift.get();
    sa.P = h->P; sa.B = h->B; sa.K = h->K;
    sa.row_first = h->row0; sa.n_rows = h->n_rows;
    sa.rows = h->windows ? h->d_rows.get() : nullptr;
    sa.w = h->w;
    sa.n_lags = h->N;
    sa.cand = xchg ? xc.cand_all + (size_t)xc.sh.prn_first * xc.sh.freq_num_total + xc.sh.bin_first : h->d_cand.get();
    sa.cand_stride = xchg ? xc.sh.freq_num_total : h->B;
    sa.surface = h->d_surface.get();
    sa.scratch = h->d_scratch.get();
    sa.group_ctr = h->d_group_ctr.get();
    sa.row_slots = h->d_row_slots.get();
    sa.partial = h->d_partial.get();
    sa.part_ctr = h->d_group_ctr ? h->d_group_ctr.get() + h->coop_groups : nullptr;
    sa.row_ticket = h->d_group_ctr ? h->d_group_ctr.get() + (size_t)h->coop_groups * (1 + h->ops->R) : nullptr;
    sa.row_granular = h->by_blocks ? 0 : 1;
#ifdef GNSS_TIMELINE
    static unsigned long long* d_timeline = nullptr;
    if (!d_timeline) { CU(cudaMalloc(&d_timeline, 16 * 16 * 32 * sizeof(unsigned long long))); }
    CU(cudaMemsetAsync(d_timeline, 0, 16 * 16 * 32 * sizeof(unsigned long long), s));
    sa.timeline = d_timeline;
    g_timeline = d_timeline;
#endif
    h->used_groups = h->coop_groups + h->l2x_clusters;
    h->used_split = h->by_blocks ? 2 : 1;
    if (h->n_rows > 0) {                   // (0: Doppler windows that hold no bin; K4 reports every PRN as not searched)
        if (h->coop_groups > 0) {
            CU(cudaMemsetAsync(h->d_group_ctr.get(), 0, (size_t)h->coop_groups * (2 + h->ops->R) * sizeof(unsigned), s));
            CU(h->ops->launch_search_coop(sa, h->coop_groups, s));
        } else if (h->l2x_clusters > 0) {
            CU(h->ops->launch_search_l2x(sa, h->l2x_clusters, s));
        } else {
            CU(h->ops->launch_search(sa, h->n_rows, s));
        }
        h->launches += 1;
    }
    CU(cudaEventRecord(h->ev[3].get(), s));
    if (xchg) {
        // candidates went straight into the root's table; a non-root shard now raises its "done" flag there,
        // the root runs K4 over the full table in gnssacq_xchg_finish
        if (!xc.is_root) {
            xchg_done_kernel<<<1, 1, 0, s>>>(xc.flags + 1 + xc.sh.rank, xc.epoch);
            CU(cudaGetLastError());
            h->launches += 1;
        }
        CU(cudaEventRecord(h->ev[4].get(), s));
        return GNSSACQ_OK;
    }
    finalize_kernel<<<(h->P + 63) / 64, 64, 0, s>>>(h->d_cand.get(), h->P, h->B, h->N, h->w, h->cfg.freq_min_hz,
                                                    h->cfg.freq_step_hz, h->cfg.snr_threshold_db, h->d_prn.get(),
                                                    d_out ? d_out : h->d_res.get(), h->B, h->bin0);
    CU(cudaGetLastError());
    h->d_last_rows = d_out ? d_out : h->d_res.get();
    h->launches += 1;
    CU(cudaEventRecord(h->ev[4].get(), s));
    return GNSSACQ_OK;
}

// Upload of a pageable IF block to the handle's own IF buffer, timed from ev[0]; the search follows on the stream.
int upload_if(gnssacq_handle* h, const void* if_samples) {
    CU(cudaEventRecord(h->ev[0].get(), h->stream));
    if (int rc = stage_and_upload(h, h->d_if.get(), if_samples, h->stream)) return rc;    // caller's buffer is free again after this
    h->have_h2d = true;
    return GNSSACQ_OK;
}

// d_out == nullptr: the rows go to the handle's own table
int enqueue_device(gnssacq_handle* h, const void* d_if, size_t nbytes, gnssacq_result* d_out) {
    if (!h || !d_if) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    if (nbytes < h->if_bytes) return fail(h, GNSSACQ_ERR_SHORT_BUFFER, "IF block shorter than noncoh_blocks*coh_ms ms");
    CU(cudaSetDevice(h->device));
    h->have_h2d = false;
    CU(cudaEventRecord(h->ev[0].get(), h->stream));
    return enqueue(h, d_if, d_out);
}


// BASELINE config 4 (periodic re-acquisition over a long recording) / SURVEY 8f-3 (IF ingest): n_windows
// independent searches.  Window i+1 is staged (host memcpy into pinned memory) and copied to HBM on a copy
// stream while window i is searched; two staging pairs, events in both directions, one D2H of all rows at the
// end.  Rows of window i are out[i*n_prn .. (i+1)*n_prn) and equal what gnssacq_search returns for that window.
// `fill(i, dst)` puts window i (if_bytes bytes) into pinned staging memory: a memcpy from the caller's window
// (gnssacq_sweep) or an fseek + fread straight from the recording (gnssacq_sweep_file).
template <class Fill>
int sweep_impl(gnssacq_handle* h, int32_t n_windows, gnssacq_result* out, gnssacq_stats* st, Fill&& fill) {
    if (n_windows == 0) return GNSSACQ_OK;
    CU(cudaSetDevice(h->device));
    if (!h->sweep) {
        auto sw = std::make_unique<SweepState>();
        CU(create(sw->copy_stream, cudaStreamNonBlocking));
        CU(alloc(sw->d_if2, h->if_bytes));
        CU(alloc(sw->h_if2, h->if_bytes));
        for (auto& e : sw->copied) CU(create(e, cudaEventDisableTiming));
        for (auto& e : sw->consumed) CU(create(e, cudaEventDisableTiming));
        h->sweep = std::move(sw);
    }
    SweepState& sw = *h->sweep;
    if (sw.cap < n_windows) {
        CU(cudaStreamSynchronize(h->stream));
        sw.cap = 0;
        CU(alloc(sw.d_res, (size_t)n_windows * h->P * sizeof(gnssacq_result)));
        sw.cap = n_windows;
    }
    cudaStream_t cs = sw.copy_stream.get();
    void* d_buf[2] = {h->d_if.get(), sw.d_if2.get()};
    void* h_buf[2] = {h->h_if.get(), sw.h_if2.get()};
    const auto t0 = std::chrono::steady_clock::now();
    int launches = 0;
    for (int i = 0; i < n_windows; ++i) {
        const int b = i & 1;
        if (i >= 2) CU(cudaEventSynchronize(sw.copied[b].get()));              // pinned buffer b has left for HBM
        { const int rc = fill(i, h_buf[b]); if (rc != GNSSACQ_OK) { cudaStreamSynchronize(h->stream); cudaStreamSynchronize(cs); return rc; } }
        if (i >= 2) CU(cudaStreamWaitEvent(cs, sw.consumed[b].get(), 0));   // search i-2 is done with d_buf[b]
        else if (i == 0) CU(cudaStreamWaitEvent(cs, h->ev[4].get(), 0));      // d_if: after whatever this handle ran last
        // (i == 1: d_if2 / h_if2 are touched by sweeps only, and every sweep ends with a stream sync: no wait, so
        //  the copy of window 1 overlaps the search of window 0)
        CU(cudaMemcpyAsync(d_buf[b], h_buf[b], h->if_bytes, cudaMemcpyHostToDevice, cs));
        CU(cudaEventRecord(sw.copied[b].get(), cs));
        CU(cudaStreamWaitEvent(h->stream, sw.copied[b].get(), 0));
        h->have_h2d = false;
        CU(cudaEventRecord(h->ev[0].get(), h->stream));
        int rc = enqueue(h, d_buf[b], sw.d_res.get() + (size_t)i * h->P);
        if (rc != GNSSACQ_OK) return rc;
        launches += h->launches;
        CU(cudaEventRecord(sw.consumed[b].get(), h->stream));
    }
    CU(cudaMemcpyAsync(out, sw.d_res.get(), (size_t)n_windows * h->P * sizeof(gnssacq_result), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaEventRecord(h->ev[5].get(), h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (st) {
        std::memset(st, 0, sizeof(*st));
        st->total_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
        cudaEventElapsedTime(&st->wipeoff_fft_ms, h->ev[1].get(), h->ev[2].get());      // (of the last window)
        cudaEventElapsedTime(&st->search_ms, h->ev[2].get(), h->ev[3].get());
        cudaEventElapsedTime(&st->finalize_ms, h->ev[3].get(), h->ev[4].get());
        st->kernel_launches = launches;
        fill_engine_stats(h, st);
    }
    return GNSSACQ_OK;
}

}  // namespace gnss

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

int gnssacq_transform_size(const gnssacq_config* c, int32_t* n_out) {
    if (!c || !n_out) return fail(nullptr, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    const int nf = transform_length(c->samples_per_ms);
    if (nf == 0) return fail(nullptr, GNSSACQ_ERR_UNSUPPORTED_N, "samples_per_ms has no built transform length (> 29 000 and not 6000, 26000 or 58000)");
    *n_out = nf;
    return GNSSACQ_OK;
}

const char* gnssacq_last_error(const gnssacq_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int gnssacq_destroy(gnssacq_handle* h) {
    if (!h) return GNSSACQ_ERR_INVALID_ARG;
    delete h;
    return GNSSACQ_OK;
}

int gnssacq_create(const gnssacq_config* cfg, gnssacq_handle** out) {
    if (!out) return fail(nullptr, GNSSACQ_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    std::string why;
    int rc = validate(cfg, why);
    if (rc != GNSSACQ_OK) return fail(nullptr, rc, why);

    const int NF = transform_length(cfg->samples_per_ms);       // validate() has checked it is not 0
    const int Q = NF / 2000;
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

    // on any failure below, `owner` releases whatever has been made so far
    std::unique_ptr<gnssacq_handle> owner(new (std::nothrow) gnssacq_handle());
    gnssacq_handle* const h = owner.get();
    if (!h) return fail(nullptr, GNSSACQ_ERR_NOMEM, "out of host memory");
    h->cfg = *cfg;
    h->ops = ops;
    h->device = dev;
    h->N = cfg->samples_per_ms;
    h->NF = NF;
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
    const size_t N = (size_t)h->N, NFs = (size_t)NF;
    const size_t nb = h->base_freq.size();

    CU(cudaSetDevice(dev), GNSSACQ_ERR_NOMEM);
    CU(create(h->own_stream, cudaStreamNonBlocking), GNSSACQ_ERR_NOMEM);
    h->stream = h->own_stream.get();
    for (auto& e : h->ev) CU(create(e, cudaEventDefault), GNSSACQ_ERR_NOMEM);
    CU(ops->prepare(), GNSSACQ_ERR_NOMEM);
    CU(alloc(h->d_if, h->if_bytes), GNSSACQ_ERR_NOMEM);
    CU(alloc(h->d_scode, (size_t)h->P * NFs), GNSSACQ_ERR_NOMEM);
    CU(alloc(h->d_cc, (size_t)h->P * NFs * sizeof(cf)), GNSSACQ_ERR_NOMEM);
    CU(alloc(h->d_x, nb * (size_t)h->K * (NFs / Q * (2 * Q - 1)) * sizeof(cf)), GNSSACQ_ERR_NOMEM);   // c-extended: NF*(2Q-1)/Q
    CU(alloc(h->d_bin_base, h->B * sizeof(int)), GNSSACQ_ERR_NOMEM);
    CU(alloc(h->d_bin_shift, h->B * sizeof(int)), GNSSACQ_ERR_NOMEM);
    CU(alloc(h->d_prn, h->P * sizeof(int)), GNSSACQ_ERR_NOMEM);
    CU(alloc(h->d_base_freq, nb * sizeof(double)), GNSSACQ_ERR_NOMEM);
    CU(alloc(h->d_cand, (size_t)h->P * h->B * sizeof(Candidate)), GNSSACQ_ERR_NOMEM);
    CU(alloc(h->d_res, h->P * sizeof(gnssacq_result)), GNSSACQ_ERR_NOMEM);
    CU(alloc(h->d_sums, 2 * sizeof(long long)), GNSSACQ_ERR_NOMEM);
    CU(alloc(h->d_means, 2 * sizeof(double)), GNSSACQ_ERR_NOMEM);
    // exchange: 1 = DSMEM clusters, 2 = L2 buffer + clusters, 3 = L2 buffer + cooperative groups (no clusters).
    // auto: cooperative groups for the two real front ends (fastest measured, profiles/r01), DSMEM for tiny N.
    h->xmode = cfg->exchange ? cfg->exchange : (Q >= 13 ? 3 : 1);
    {
        Schedule sc;
        if (int rc = plan_schedule(h, h->n_rows, sc)) return rc;
        if (int rc = use_schedule(h, sc)) return rc;
    }
    if (cfg->keep_surface) {
        CU(alloc(h->d_surface, (size_t)h->P * h->B * N * sizeof(float)), GNSSACQ_ERR_NOMEM);
    }
    CU(alloc(h->h_if, h->if_bytes), GNSSACQ_ERR_NOMEM);
    CU(alloc(h->h_res, h->P * sizeof(gnssacq_result)), GNSSACQ_ERR_NOMEM);
    // Every create-time copy goes on the handle's own (non-blocking) stream: a synchronous cudaMemcpy from
    // pageable memory returns once the data is STAGED, and its DMA on the legacy stream is not ordered with
    // kernels on a non-blocking stream (seen once in r01 as one PRN's code spectrum built from a half-copied
    // replica table).
    CU(cudaMemcpyAsync(h->d_bin_base.get(), h->bin_base.data(), h->B * sizeof(int), cudaMemcpyHostToDevice, h->stream), GNSSACQ_ERR_NOMEM);
    CU(cudaMemcpyAsync(h->d_bin_shift.get(), h->bin_shift.data(), h->B * sizeof(int), cudaMemcpyHostToDevice, h->stream), GNSSACQ_ERR_NOMEM);
    CU(cudaMemcpyAsync(h->d_prn.get(), cfg->prn, h->P * sizeof(int), cudaMemcpyHostToDevice, h->stream), GNSSACQ_ERR_NOMEM);
    CU(cudaMemcpyAsync(h->d_base_freq.get(), h->base_freq.data(), nb * sizeof(double), cudaMemcpyHostToDevice, h->stream), GNSSACQ_ERR_NOMEM);
    if (h->n_rows < h->P * h->B) {                              // a row range
        if (int rc = clear_unsearched(h)) return rc;
    }
    std::vector<double> bw(nb);                                 // (read by a copy that the final sync waits for)
    {
        // K1 v2 (comb rows + cp.async staging) whenever its shared memory fits; otherwise, and for every padded shape
        // (its ms are not whole comb rows), the v1 gather kernel
        const int bps = h->cfg.data_type * h->cfg.data_precision;
        const int pitch = ((N / 16) * bps + 15) / 16 * 16;
        if (NF == h->N && ops->smem_wipe2(pitch, h->M) <= (size_t)227 * 1024) {
            for (size_t i = 0; i < nb; ++i) bw[i] = h->base_freq[i] / h->cfg.fs_hz;
            CU(alloc(h->d_base_w, nb * sizeof(double)), GNSSACQ_ERR_NOMEM);
            CU(cudaMemcpyAsync(h->d_base_w.get(), bw.data(), nb * sizeof(double), cudaMemcpyHostToDevice, h->stream), GNSSACQ_ERR_NOMEM);
            h->comb_pitch = pitch;
            CU(alloc(h->d_comb, (size_t)h->K * h->M * 16 * pitch), GNSSACQ_ERR_NOMEM);
            // the int16 means sum the pad bytes too: they must be zero, and no kernel ever writes them
            CU(cudaMemsetAsync(h->d_comb.get(), 0, (size_t)h->K * h->M * 16 * pitch, h->stream), GNSSACQ_ERR_NOMEM);
        }
    }

    // code tables -> HBM, then K0 fills the conj-spectrum cache with conj(fft(c2))/NF: c2[j] = c[j mod N] for
    // j <= 2N-2, 0 beyond (c2 = c for N = NF), so that lags m < N of the NF-point correlation never wrap
    std::vector<cf> chirp, hfilt;                                // (padded: read by copies that the final sync waits for)
    {
        std::vector<int8_t> sc((size_t)h->P * NFs, 0), one(N);
        for (int p = 0; p < h->P; ++p) {
            code_replica(*cfg, cfg->prn[p], one.data());
            int8_t* row = sc.data() + (size_t)p * NFs;
            for (size_t j = 0; j < NFs && j <= 2 * N - 2; ++j) row[j] = one[j % N];
        }
        CU(cudaMemcpyAsync(h->d_scode.get(), sc.data(), sc.size(), cudaMemcpyHostToDevice, h->stream), GNSSACQ_ERR_NOMEM);
        CodeArgs a{h->d_scode.get(), h->d_cc.get()};
        CU(ops->launch_code(a, h->P, h->stream), GNSSACQ_ERR_NOMEM);
    }
    if (NF != h->N) {
        // Bluestein tables of the N-point DFTs (fine stage, gnssacq_fft_forward): ch[n] = exp(i pi n^2 / N) with n^2 mod 2N
        // in integers (exact: 2N^2 < 2^31 for N <= 29 000), and H = FFT_NF of the chirp filter h[j] = ch[|j|], |j| < N
        chirp.resize(N);
        hfilt.assign(NFs, mk(0.f, 0.f));
        for (int n = 0; n < h->N; ++n) {
            const int e = (int)(((long long)n * n) % (2ll * h->N));
            const double ang = 3.14159265358979323846 * (double)e / (double)h->N;
            chirp[n] = mk((float)std::cos(ang), (float)std::sin(ang));
            hfilt[n] = chirp[n];
            if (n > 0) hfilt[NFs - n] = chirp[n];
        }
        CU(alloc(h->d_chirp, N * sizeof(cf)), GNSSACQ_ERR_NOMEM);
        CU(alloc(h->d_chirp_filt, NFs * sizeof(cf)), GNSSACQ_ERR_NOMEM);
        DevPtr<cf> tmp;
        CU(alloc(tmp, NFs * sizeof(cf)), GNSSACQ_ERR_NOMEM);
        CU(cudaMemcpyAsync(h->d_chirp.get(), chirp.data(), N * sizeof(cf), cudaMemcpyHostToDevice, h->stream), GNSSACQ_ERR_NOMEM);
        CU(cudaMemcpyAsync(tmp.get(), hfilt.data(), NFs * sizeof(cf), cudaMemcpyHostToDevice, h->stream), GNSSACQ_ERR_NOMEM);
        NaturalArgs na{tmp.get(), h->d_chirp_filt.get()};
        CU(ops->launch_natural(na, 1, h->stream), GNSSACQ_ERR_NOMEM);
        CU(cudaStreamSynchronize(h->stream), GNSSACQ_ERR_NOMEM);   // before `tmp` is freed
    }
    CU(cudaStreamSynchronize(h->stream), GNSSACQ_ERR_NOMEM);
    *out = owner.release();
    return GNSSACQ_OK;
}

int gnssacq_set_stream(gnssacq_handle* h, void* s) {
    if (!h) return GNSSACQ_ERR_INVALID_ARG;
    h->stream = (s == GNSSACQ_OWN_STREAM) ? h->own_stream.get() : (cudaStream_t)s;
    return GNSSACQ_OK;
}

// The windows only choose which rows of the full grid K2 walks: the forward spectra, K1 and the int16 means are the
// full grid's, so a windowed PRN's candidates are bit for bit those of the full search in its window's bins, and K4
// over a table whose other cells hold the peak -1 sentinel picks what a bin_first / bin_count handle would.
int gnssacq_set_doppler_windows(gnssacq_handle* h, const double* lo_hz, const double* hi_hz) {
    if (!h) return GNSSACQ_ERR_INVALID_ARG;
    if (!lo_hz != !hi_hz) return fail(h, GNSSACQ_ERR_INVALID_ARG, "lo_hz and hi_hz must both be given or both be NULL");
    if (lo_hz) {
        for (int i = 0; i < h->P; ++i)
            if (!(lo_hz[i] <= hi_hz[i])) return fail(h, GNSSACQ_ERR_INVALID_ARG, "a Doppler window has lo_hz > hi_hz or a NaN bound");
    }
    if (h->cfg.bin_count > 0 || h->cfg.row_count > 0) return fail(h, GNSSACQ_ERR_STATE, "Doppler windows need a handle over the full grid (bin_count = row_count = 0)");
    if (h->xc.on) return fail(h, GNSSACQ_ERR_STATE, "Doppler windows are not available in the multi-GPU exchange");
    // grid row ids, bin-major: the strided schedule then keeps the groups on neighbouring rows (the same forward spectra).
    // Cleared: all P*B rows, which the search kernels walk without the list.
    std::vector<int> rows;
    rows.reserve((size_t)h->P * h->B);
    for (int b = 0; b < h->B; ++b) {
        const double f = std::fma(h->cfg.freq_step_hz, (double)b, h->cfg.freq_min_hz);   // K4's doppler_hz (a fused multiply-add there)
        for (int p = 0; p < h->P; ++p)
            if (!lo_hz || (lo_hz[p] <= f && f <= hi_hz[p])) rows.push_back(b * h->P + p);
    }
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));                       // an enqueued search may still read the old tables
    if (lo_hz && !h->d_rows) CU(alloc(h->d_rows, (size_t)h->P * h->B * sizeof(int)), GNSSACQ_ERR_NOMEM);
    Schedule sc;
    if (int rc = plan_schedule(h, (long long)rows.size(), sc)) return rc;
    if (int rc = use_schedule(h, sc)) return rc;
    if (lo_hz) CU(cudaMemcpyAsync(h->d_rows.get(), rows.data(), rows.size() * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    if (int rc = clear_unsearched(h)) return rc;                // (synchronises: `rows` is a temporary)
    h->n_rows = (int)rows.size();
    h->windows = lo_hz != nullptr;
    return GNSSACQ_OK;
}



int gnssacq_enqueue_device(gnssacq_handle* h, const void* d_if, size_t nbytes) {
    return enqueue_device(h, d_if, nbytes, nullptr);
}

int gnssacq_enqueue_device_out(gnssacq_handle* h, const void* d_if, size_t nbytes, void* d_out_rows) {
    if (!d_out_rows) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    return enqueue_device(h, d_if, nbytes, (gnssacq_result*)d_out_rows);
}

int gnssacq_fetch_results(gnssacq_handle* h, gnssacq_result* out, gnssacq_stats* st) {
    if (!h || (!out && !st)) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    if (!h->d_last_rows) return fail(h, GNSSACQ_ERR_STATE, "no search has been enqueued on this handle");
    CU(cudaSetDevice(h->device));
    // rows of the LAST enqueued search, wherever it wrote them (its own table, or the caller's device buffer of
    // gnssacq_enqueue_device_out); out == NULL: timings only
    if (out) CU(cudaMemcpyAsync(h->h_res.get(), h->d_last_rows, h->P * sizeof(gnssacq_result), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaEventRecord(h->ev[5].get(), h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (out) std::memcpy(out, h->h_res.get(), h->P * sizeof(gnssacq_result));
    if (st) {
        std::memset(st, 0, sizeof(*st));
        if (h->have_h2d) cudaEventElapsedTime(&st->h2d_ms, h->ev[0].get(), h->ev[1].get());
        cudaEventElapsedTime(&st->wipeoff_fft_ms, h->ev[1].get(), h->ev[2].get());
        cudaEventElapsedTime(&st->search_ms, h->ev[2].get(), h->ev[3].get());
        cudaEventElapsedTime(&st->finalize_ms, h->ev[3].get(), h->ev[4].get());
        cudaEventElapsedTime(&st->d2h_ms, h->ev[4].get(), h->ev[5].get());
        cudaEventElapsedTime(&st->total_ms, h->ev[0].get(), h->ev[5].get());
        st->kernel_launches = h->launches;
        fill_engine_stats(h, st);
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
    if (int rc = upload_if(h, if_samples)) return rc;
    int rc = enqueue(h, h->d_if.get());
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
        if (int rc = upload_if(h, if_samples)) return rc;
        int rc = enqueue(h, h->d_if.get());
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

int gnssacq_read_surface(gnssacq_handle* h, int32_t prn_index, float* out) {
    if (!h || !out || prn_index < 0 || prn_index >= h->P) return fail(h, GNSSACQ_ERR_INVALID_ARG, "bad argument");
    if (!h->d_surface) return fail(h, GNSSACQ_ERR_STATE, "handle was created without keep_surface");
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    const size_t n = (size_t)h->B * h->N;
    CU(cudaMemcpy(out, h->d_surface.get() + (size_t)prn_index * n, n * sizeof(float), cudaMemcpyDeviceToHost));
    return GNSSACQ_OK;
}

int gnssacq_fine_frequency(gnssacq_handle* h, const void* if_long, size_t nbytes, int32_t L, int32_t n_sv,
                           const int32_t* prn, const int32_t* code_phase, double* out_hz) {
    if (!h || !if_long || !prn || !code_phase || !out_hz) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    if (n_sv == 0) return GNSSACQ_OK;
    if (L < 1 || L > 16 || n_sv < 0) return fail(h, GNSSACQ_ERR_INVALID_ARG, "L must be 1..16, n_sv >= 0");
    if (n_sv > GNSSACQ_MAX_PRN) return fail(h, GNSSACQ_ERR_INVALID_ARG, "too many SVs");
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

    constexpr int kChunk = 4;                                                   // SVs per pass (scratch ~0.4 GB at N = 58 000;
                                                                                // a padded shape adds K*L*NF per SV: ~0.37 GB at 16.368 MHz, L = 10, K = 20)
    const bool padded = h->NF != h->N;
    if (!h->fine || h->fine->L != L) {
        // (re)build the per-L scratch: chip index of sample t (acquisition.m:104-105, same double arithmetic)
        h->fine.reset();                                                        // the old scratch goes first
        std::vector<uint16_t> chip((size_t)LN);
        const double inv_fs = 1.0 / c.fs_hz, inv_fc = 1.0 / c.code_hz;
        const double codelength = c.code_hz * 1e-3;                             // initParameters.m:47
        for (long long t = 1; t <= LN; ++t) {
            const double idx = std::floor((inv_fs * (double)t) / inv_fc);
            chip[(size_t)(t - 1)] = (uint16_t)std::fmod(idx, codelength);       // rem(.)+1, 0-based here
        }
        auto fs = std::make_unique<FineState>();
        CU(alloc(fs->raw, need));
        CU(alloc(fs->chip, chip.size() * sizeof(uint16_t)));
        CU(alloc(fs->ca, (size_t)GNSSACQ_MAX_PRN * 1023));
        CU(alloc(fs->start, GNSSACQ_MAX_PRN * sizeof(int)));
        CU(alloc(fs->best, GNSSACQ_MAX_PRN * sizeof(unsigned long long)));
        CU(alloc(fs->u, (size_t)kChunk * K * L * N * sizeof(cf)));
        if (padded) CU(alloc(fs->v, (size_t)kChunk * K * L * h->NF * sizeof(cf)));
        CU(cudaMemcpyAsync(fs->chip.get(), chip.data(), chip.size() * sizeof(uint16_t), cudaMemcpyHostToDevice, s));
        CU(cudaStreamSynchronize(s));                                           // `chip` is a temporary
        fs->L = L;
        h->fine = std::move(fs);
    }
    void* d_raw = h->fine->raw.get(); uint16_t* d_chip = h->fine->chip.get(); int8_t* d_ca = h->fine->ca.get();
    int* d_start = h->fine->start.get(); cf* d_u = h->fine->u.get(); unsigned long long* d_best = h->fine->best.get();
    std::vector<int8_t> ca((size_t)n_sv * 1023);
    std::vector<int> start(n_sv);
    for (int i = 0; i < n_sv; ++i) {
        ca_chips(prn[i], ca.data() + (size_t)i * 1023);
        start[i] = N - code_phase[i] - 1;                                       // acquisition.m:106 (1-based N-codedelay)
    }
    const int chunk = n_sv < kChunk ? n_sv : kChunk;
    CU(cudaMemcpyAsync(d_raw, if_long, need, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(d_ca, ca.data(), ca.size(), cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(d_start, start.data(), n_sv * sizeof(int), cudaMemcpyHostToDevice, s));
    CU(cudaMemsetAsync(d_best, 0, n_sv * sizeof(unsigned long long), s));
    const double* means = nullptr;
    if (c.data_precision == 2) {                                                // acquisition.m:92-94
        const long long pairs = (long long)(L + 1) * N;
        if (int rc = launch_means(h, d_raw, pairs, pairs, s)) return rc;
        means = h->d_means.get();
    }
    for (int first = 0; first < n_sv; first += chunk) {
        const int n = (n_sv - first) < chunk ? (n_sv - first) : chunk;
        FineArgs fa;
        fa.raw = d_raw; fa.chip = d_chip; fa.ca = d_ca + (size_t)first * 1023; fa.start = d_start + first;
        fa.means = means; fa.data_type = c.data_type; fa.precision = c.data_precision;
        fa.L = L; fa.K = K; fa.F = F; fa.u = d_u;
        if (padded) {
            // the K*L N-point DFTs as Bluestein convolutions through the NF-point engine (see ChirpArgs)
            ChirpArgs ca{h->d_chirp.get(), h->d_chirp_filt.get(), N, nullptr, h->fine->v.get(), d_u};
            CU(h->ops->launch_fine_chirp(fa, ca, n * K * L, s));
            CU(h->ops->launch_chirp_out(ca, n * K * L, s));
        } else {
            CU(h->ops->launch_fine(fa, n * K * L, s));
        }
        dim3 grid((unsigned)((N + 255) / 256), (unsigned)K, (unsigned)n);
        fine_combine_kernel<<<grid, 256, 0, s>>>(d_u, K, L, N, F, c.data_type == 2 ? 1 : 0, d_best + first);
        CU(cudaGetLastError());
    }
    std::vector<unsigned long long> best(n_sv);
    CU(cudaMemcpyAsync(best.data(), d_best, n_sv * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
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
    DevPtr<float> d;
    CU(alloc(d, 4));
    Event e0, e1;
    CU(create(e0, cudaEventDefault));
    CU(create(e1, cudaEventDefault));
    const int blocks = prop.multiProcessorCount * 8, iters = 4096;
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        CU(cudaEventRecord(e0.get(), 0));
        fma_peak_kernel<<<blocks, 256>>>(d.get(), iters, 1.0000001f, 1e-7f);
        CU(cudaEventRecord(e1.get(), 0));
        CU(cudaEventSynchronize(e1.get()));
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, e0.get(), e1.get()));
        const double flops = 2.0 * 16.0 * 8.0 * (double)iters * 256.0 * (double)blocks;
        if (rep > 0 && ms > 0.f) best = std::max(best, flops / (ms * 1e-3) * 1e-12);
    }
    *out_tflops = best;
    return GNSSACQ_OK;
}

int gnssacq_fft_forward(gnssacq_handle* h, const float* in, float* out) {
    if (!h || !in || !out) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    CU(cudaSetDevice(h->device));
    const size_t bytes = (size_t)h->N * sizeof(cf);
    const bool padded = h->NF != h->N;
    if (!h->fft) {
        auto f = std::make_unique<FftState>();
        CU(alloc(f->in, bytes));
        CU(alloc(f->out, bytes));
        if (padded) CU(alloc(f->v, (size_t)h->NF * sizeof(cf)));
        h->fft = std::move(f);
    }
    CU(cudaMemcpyAsync(h->fft->in.get(), in, bytes, cudaMemcpyHostToDevice, h->stream));
    if (padded) {
        // the N-point DFT as a Bluestein convolution through the NF-point engine (the fine stage's path)
        ChirpArgs c{h->d_chirp.get(), h->d_chirp_filt.get(), h->N, h->fft->in.get(), h->fft->v.get(), h->fft->out.get()};
        CU(h->ops->launch_chirp_in(c, 1, h->stream));
        CU(h->ops->launch_chirp_out(c, 1, h->stream));
    } else {
        NaturalArgs a{h->fft->in.get(), h->fft->out.get()};
        CU(h->ops->launch_natural(a, 1, h->stream));
    }
    CU(cudaMemcpyAsync(out, h->fft->out.get(), bytes, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return GNSSACQ_OK;
}

}  // extern "C"
