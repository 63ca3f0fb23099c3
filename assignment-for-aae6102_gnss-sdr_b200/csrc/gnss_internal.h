// gnss_internal.h -- argument blocks shared by the kernels (per-Q translation units)
// and the C-ABI host code (gnssacq.cu).  Not part of the public interface.
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>
#include "gnss_engine.h"

namespace gnss {

// One (PRN, Doppler-bin) row's outcome, written by the search kernel (K2 + K3).
struct Candidate {
    float peak;        // max over lags of the non-coherent power (acquisition.m:63 restricted to the row)
    int lag;           // first lag attaining it (0-based)
    double sum_all;    // sum over all lags of power^2
    double sum_win;    // sum of power^2 over lags lag-(w-1) .. lag+(w-1), clipped to [0,N-1] (acquisition.m:67)
};

struct SearchArgs {
    const cf* cc;          // [P][N]   conj(fft(code))/N, G layout
    const cf* x;           // [n_bases][K][N] forward spectra of wiped-off blocks, G layout
    const int* bin_base;   // [B] which base a bin derives from
    const int* bin_shift;  // [B] shift in FFT bins relative to that base (SURVEY A.7)
    int P, B, K;
    int row_first, n_rows; // this launch searches rows [row_first, +n_rows) of the grid, row = b*P + p (all of them: 0, P*B) ...
    const int* rows;       // ... or, when not null, the n_rows grid rows listed here, bin-major (Doppler windows).  The
                           // contiguous range is computed, not looked up: a per-row table read on the path to the next
                           // row's first loads cost the default search kernels 1 % (B200, configs 1 and 2)
    int w;                 // ceil(Fs/fc) (acquisition.m:66)
    int n_lags;            // lags a row reports: samples per ms.  The transform length for a built N; less for a handle that
                           // zero-pads each ms into a longer transform, whose lags >= n_lags are not part of the correlation
    Candidate* cand;       // [P][cand_stride]: row (p, b) at cand[p*cand_stride + b].  A shard of a multi-GPU search
                           // points this straight into the ROOT GPU's table (peer memory, NVLink stores)
    int cand_stride;       // >= B (the full grid's bin count when the handle owns a bin sub-range)
    float* surface;        // optional [P][B][n_lags] (debug), lag order
    cf* scratch;           // L2-exchange variants: [groups][2][16][RS] (double-buffered finished rows)
    unsigned* group_ctr;   // coop variant: one arrival counter per CTA group (zeroed before the launch)
    Candidate* row_slots;  // coop variant: [groups][R] per-CTA partial row results
    float* partial;        // coop variant: [groups][K-1][R][ACC_ELEMS] power planes of tail-row blocks handed to the finishing group
    unsigned* part_ctr;    // coop variant: [groups][R] published planes (zeroed before the launch)
    unsigned* row_ticket;  // coop variant: [groups] row-end tickets: the last of a group's R CTAs to finish a row writes its candidate
    int row_granular;      // coop variant: deal out whole rows only (no hand-over; sums independent of the group count)
#ifdef GNSS_TIMELINE       // experiment builds only (profiles/timeline.py): clock64 stamps of one iteration of group 0
    unsigned long long* timeline;   // [R][warps][32]
#endif
};

struct WipeArgs {
    const void* raw;       // device IF block
    int data_type, precision, coh_ms, K;
    size_t block_bytes;    // bytes per coherent block
    int n_ms;              // samples per ms (the fold's stride); < N: wipe_pad_kernel zero-pads each ms to the transform length
    const double* base_freq_hz;   // [n_bases] IF + doppler of each base
    double fs_hz;
    const double* means;   // [2] int16 path (device), else nullptr
    cf* x;                 // [n_bases][K][N]
};

// K1 v2 (r02): the IF block is first re-ordered by `comb_kernel` into 16 "comb" rows per millisecond --
// row rho of ms t holds samples n = 16*m + rho, m = 0 .. N/16-1, contiguously (pitch bytes per row, a multiple
// of 16) -- because an a-row of the prime-factor array only ever reads samples of ONE residue n mod 16
// (n = a*M1 + b*M2 + c*M3 with M2, M3 multiples of 16).  wipe2_kernel then stages exactly its rows with
// cp.async (contiguous 16-byte chunks) instead of gathering single bytes scattered over the whole block.
struct Wipe2Args {
    const unsigned char* comb;    // [K*M ms][16][pitch] bytes
    int pitch;                    // bytes per comb row (multiple of 16)
    int bps;                      // bytes per sample: 1 int8 real, 2 int8 I/Q, 4 int16 I/Q
    int coh_ms, K;
    const double* base_w;         // [n_bases] (IF + doppler) / Fs of each base, cycles per sample
    const double* means;          // [2] int16 path (device), else nullptr
    cf* x;                        // [n_bases][K][NX]
};

struct CodeArgs {
    const int8_t* scode;   // [P][N] upsampled +-1 code replicas (acquisition.m:51)
    cf* cc;                // [P][N]
};

struct NaturalArgs {
    const cf* in;          // [units][N] natural order
    cf* out;               // [units][N] natural order
};

// fine-frequency stage (acquisition.m:83-127): K*L decimated N-point transforms per acquired SV
struct FineArgs {
    const void* raw;             // device copy of the (L+1) ms block
    const uint16_t* chip;        // [L*N]
    const int8_t* ca;            // [n_sv][1023]
    const int* start;            // [n_sv] N - codedelay - 1
    const double* means;         // [2] int16 path, else nullptr
    int data_type, precision, L, K;
    long long F;
    cf* u;                       // [n_sv][K][L][N] natural order
};

// Bluestein (chirp-z) N-point DFTs, for an N that is not a built transform length, through the built N'-point
// engine (N' >= 2N-1):  X[k] = conj(ch[k]) * (a (*) h)[k],  a[n] = x[n] conj(ch[n]) zero-padded to N',
// ch[n] = exp(i pi n^2 / N), h the chirp filter ch[j], |j| < N, wrapped mod N'.  The circular convolution is
// conj(FFT(conj(FFT(a) * H))) / N' with H = FFT(h), built once per handle.
struct ChirpArgs {
    const cf* chirp;       // [n] ch[n]
    const cf* filt;        // [N'] H, natural order
    int n;                 // DFT length N
    const cf* in;          // [units][n] natural-order input (chirp_in_kernel; the fine stage loads its own)
    cf* v;                 // [units][N'] FFT(a), natural order
    cf* out;               // [units][n] X, natural order
};

struct VariantOps {
    int Q, R, T;
    size_t smem_search, smem_transform;
    cudaError_t (*prepare)();
    cudaError_t (*launch_code)(const CodeArgs&, int units, cudaStream_t);
    cudaError_t (*launch_wipe)(const WipeArgs&, int units, cudaStream_t);
    cudaError_t (*launch_wipe2)(const Wipe2Args&, int units, cudaStream_t);
    size_t (*smem_wipe2)(int pitch, int coh_ms);
    cudaError_t (*launch_natural)(const NaturalArgs&, int units, cudaStream_t);
    cudaError_t (*launch_fine)(const FineArgs&, int units, cudaStream_t);
    cudaError_t (*launch_search)(const SearchArgs&, int rows, cudaStream_t);
    // L2-exchange persistent variant: `clusters` co-resident clusters loop over the rows
    cudaError_t (*launch_search_l2x)(const SearchArgs&, int clusters, cudaStream_t);
    int (*max_clusters_l2x)();             // co-resident clusters of search_kernel_l2x on the current device
    size_t scratch_bytes_per_cluster;
    // cluster-free cooperative persistent variant: groups of R CTAs, software barriers through L2
    cudaError_t (*launch_search_coop)(const SearchArgs&, int groups, cudaStream_t);
    int (*max_groups_coop)();              // co-resident CTA groups on the current device
    size_t partial_bytes_per_group;        // coop variant: one power plane (all R slices) of the tail hand-over
    // zero-padded shapes (samples per ms < N): K1 gather kernel, and the three stages of a Bluestein DFT
    cudaError_t (*launch_wipe_pad)(const WipeArgs&, int units, cudaStream_t);
    cudaError_t (*launch_chirp_in)(const ChirpArgs&, int units, cudaStream_t);       // ChirpArgs.in -> v
    cudaError_t (*launch_fine_chirp)(const FineArgs&, const ChirpArgs&, int units, cudaStream_t);   // fine samples -> v
    cudaError_t (*launch_chirp_out)(const ChirpArgs&, int units, cudaStream_t);      // v -> out
};

// defined in gnss_q3.cu / gnss_q13.cu / gnss_q29.cu
const VariantOps* gnss_variants_q3(int* count);
const VariantOps* gnss_variants_q13(int* count);
const VariantOps* gnss_variants_q29(int* count);

}  // namespace gnss
