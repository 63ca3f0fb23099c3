/* gnssacq.h -- C ABI of libgnssacq.so: B200-native GPS L1 C/A parallel code-phase acquisition.
 *
 * Drop-in boundary for ONE function of the reference receiver,
 *     Acquired = acquisition(file, signal, acq)
 *     (SDR_MATLAB-main/acqtckpos/acquisition.m:1, coarse search :19-80),
 * which has no FFI of its own (it is a MATLAB function).  The entry points below
 * are what a MEX gateway (matlab/gnssacq_mex.c) or a ctypes loader
 * (gnssacq/api.py) binds; INTEGRATION.md shows both stubs.
 *
 * Conventions: plain C, no C++ or torch types; every function returns 0 on
 * success or a negative gnssacq_status; no exceptions or exit() cross the ABI.
 * A handle is not re-entrant; distinct handles may be used from distinct
 * threads.  Caller owns `if_samples` and `out`; the library copies the input
 * into its own pinned staging before the call returns.  There is NO CPU
 * fallback: without a CUDA device (sm_100) gnssacq_create fails with
 * GNSSACQ_ERR_NO_DEVICE.
 */
#ifndef GNSSACQ_H_
#define GNSSACQ_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GNSSACQ_MAX_PRN 64

typedef enum gnssacq_status {
    GNSSACQ_OK = 0,
    GNSSACQ_ERR_INVALID_ARG = -1,    /* NULL pointer, non-positive count, PRN outside 1..51 ...        */
    GNSSACQ_ERR_UNSUPPORTED_N = -2,  /* samples_per_ms has no transform length: neither 2000*Q with Q
                                        built (6000, 26000, 58000) nor <= 29000 (gnssacq_transform_size) */
    GNSSACQ_ERR_SHORT_BUFFER = -3,   /* fewer IF bytes than noncoh_blocks*coh_ms ms                    */
    GNSSACQ_ERR_CUDA = -4,           /* a CUDA runtime call failed; see gnssacq_last_error             */
    GNSSACQ_ERR_NO_DEVICE = -5,      /* no CUDA device / wrong architecture                            */
    GNSSACQ_ERR_NOMEM = -6,
    GNSSACQ_ERR_STATE = -7           /* e.g. gnssacq_read_surface without keep_surface                 */
} gnssacq_status;

/* Mirrors exactly the fields acquisition.m reads (acquisition.m:24-43,53,66,70) plus the
 * extensions BASELINE.json's configs need (coh_ms, PRN shard, engine variant). */
typedef struct gnssacq_config {
    double fs_hz;             /* signal.Fs            (initParameters.m:42) */
    double if_hz;             /* signal.IF            (initParameters.m:41) */
    double code_hz;           /* signal.codeFreqBasis (initParameters.m:44) */
    int32_t samples_per_ms;   /* signal.Sample = ceil(Fs*1e-3) (initParameters.m:46).  Any value up to 29000
                                 (Fs <= 29 MHz), or 58000: a value that is not a built transform length is
                                 zero-padded each ms into one (gnssacq_transform_size) */
    int32_t data_type;        /* file.dataType: 1 real, 2 I/Q   (initParameters.m:37) */
    int32_t data_precision;   /* file.dataPrecision: 1 int8, 2 int16 (initParameters.m:38) */
    double freq_min_hz;       /* acq.freqMin  (initParameters.m:52) */
    double freq_step_hz;      /* acq.freqStep (initParameters.m:51) */
    int32_t freq_num;         /* acq.freqNum  (initParameters.m:53) */
    int32_t noncoh_blocks;    /* acq.datalen  (initParameters.m:54): K non-coherent blocks */
    int32_t coh_ms;           /* M, coherent ms per block; 1 in the reference (SURVEY A.8) */
    int32_t n_prn;            /* number of PRNs searched by THIS handle (a rank's shard) */
    int32_t prn[GNSSACQ_MAX_PRN]; /* reference: 1..32 (acquisition.m:47) */
    double snr_threshold_db;  /* 12 (acquisition.m:70) */
    int32_t device;           /* CUDA device ordinal; -1 = current device */
    int32_t cluster_ctas;     /* engine variant: CTAs per transform (0 = auto) */
    int32_t threads;          /* engine variant: threads per CTA (0 = auto) */
    int32_t keep_surface;     /* debug: also keep the freq_num x samples_per_ms power surface of
                                 every PRN in HBM for gnssacq_read_surface (costs HBM + bandwidth) */
    int32_t exchange;         /* engine variant: how the CTAs of a transform exchange rows before the last
                                 pass.  0 = auto, 1 = distributed shared memory (clusters), 2 = L2-resident
                                 buffer (persistent clusters), 3 = L2-resident buffer, cooperative CTA
                                 groups without clusters (uses every SM) */
    int32_t work_split;       /* exchange 3 only: how the (PRN, bin) rows are dealt out to the resident CTA groups.
                                 1 = whole rows.  2 = whole rows while there are enough for every group, the
                                 remaining rows block by block: consecutive groups share a row's noncoh_blocks and
                                 the finishing group adds their power planes in block order (bit-identical to 1;
                                 costs (noncoh_blocks - 1) planes of samples_per_ms floats per group of HBM).
                                 0 = auto: 2 where it pays -- a handle with few rows (one rank's shard at 8 GPUs,
                                 a single-PRN re-acquisition) --, else 1 */
    int32_t bin_first;        /* this handle searches Doppler bins [bin_first, bin_first + bin_count) of the grid */
    int32_t bin_count;        /* (a rank's shard when there are fewer PRNs than GPUs, SURVEY 8e); 0 = all freq_num
                                 bins.  The forward transforms are planned on the FULL grid, so a sub-range produces
                                 bit for bit the candidates the full search has for those bins */
    int32_t row_first;        /* this handle searches rows [row_first, row_first + row_count) of its n_prn x bins grid, */
    int32_t row_count;        /* rows counted bin-major (row = bin * n_prn + prn index: the order the search kernel walks
                                 them).  0 = all rows.  A shard of gnssacq_shard_plan_rows: any share of the grid, to the
                                 row -- a PRN whose bins are spread over several shards is finished on the root
                                 (gnssacq_xchg_*); used alone, such a handle reports the best of the rows it owns */
} gnssacq_config;

/* One PRN's coarse-search outcome (acquisition.m:62-74); returned for every PRN, acquired or not. */
typedef struct gnssacq_result {
    int32_t prn;
    int32_t acquired;         /* SNR >= threshold (acquisition.m:70) */
    int32_t code_phase;       /* codePhase-1, what Acquired.codedelay stores (acquisition.m:74) */
    int32_t doppler_bin;      /* fbin-1 */
    double doppler_hz;        /* acquisition.m:64 */
    double peak;              /* acquisition.m:63 */
    double noise_meansq;      /* denominator of acquisition.m:67-68 */
    double snr_db;            /* acquisition.m:67 */
    double fine_freq_hz;      /* NaN here; filled by gnssacq_fine_frequency (acquisition.m:83-127) */
} gnssacq_result;

/* Device-side timings of the last search (CUDA events on the handle's stream), milliseconds. */
typedef struct gnssacq_stats {
    float h2d_ms;             /* pinned host -> HBM copy of the IF block (0 for search_device) */
    float wipeoff_fft_ms;     /* K1: wipe-off (+fold) + forward FFT of every (base, block) */
    float search_ms;          /* K2: spectrum multiply + inverse transform + |.|^2 accumulate + row peak */
    float finalize_ms;        /* K4: per-PRN winner, noise floor, SNR, threshold */
    float d2h_ms;             /* result rows HBM -> host */
    float total_ms;           /* first event to last event */
    int32_t kernel_launches;  /* kernels launched by this search */
    int32_t n_bases;          /* distinct forward transforms per block after the bin-shift identity */
    int32_t cluster_ctas;     /* engine variant actually used */
    int32_t threads;
    int32_t exchange;         /* 1 = DSMEM, 2 = L2 + clusters, 3 = L2 + cooperative groups */
    int32_t resident_clusters;/* persistent clusters / CTA groups of the search kernel (0 for DSMEM) */
    int32_t work_split;       /* schedule actually used: 1 = whole rows, 2 = block-granular tail */
    float if_pull_ms;         /* multi-GPU exchange: K1a on a non-root shard = wait for the root's IF block + pull it over
                                 NVLink + re-order (0 on the root / single GPU, where it is part of wipeoff_fft_ms) */
    float gather_wait_ms;     /* multi-GPU exchange, root: waiting for the other shards' candidates after its own search */
} gnssacq_stats;

typedef struct gnssacq_handle gnssacq_handle;

const char* gnssacq_version(void);

/* Fill *cfg with initParameters.m's defaults (Opensky front end, 32 PRNs, 41 bins, 20 ms). */
int gnssacq_config_default(gnssacq_config* cfg);

/* Bytes of IF data one search consumes: samples_per_ms*data_type*data_precision*noncoh_blocks*coh_ms
 * (the fread count of acquisition.m:29/34 times the sample size). */
size_t gnssacq_if_bytes(const gnssacq_config* cfg);

/* Transform length the search of cfg->samples_per_ms = N runs on: N itself when N is a built 2000*Q (6000,
 * 26000, 58000), otherwise the smallest built length >= 2N-1, into which each ms is zero-padded (the same rows
 * as a circular N-point correlation, at the cost of the longer transform).  Host only, no device needed.
 * Returns GNSSACQ_ERR_UNSUPPORTED_N, as gnssacq_create does, when there is none (N > 29000, not built).
 * A handle whose N is padded cannot take part in the multi-GPU exchange (gnssacq_xchg_*: GNSSACQ_ERR_STATE). */
int gnssacq_transform_size(const gnssacq_config* cfg, int32_t* n_out);

/* Build a handle: validates cfg, selects the device, allocates HBM/pinned buffers and fills the
 * HBM-resident cache of conj(fft(code))/N for cfg->prn[] (replaces acquisition.m:49-51,58). */
int gnssacq_create(const gnssacq_config* cfg, gnssacq_handle** out);
int gnssacq_destroy(gnssacq_handle* h);

/* Last error text of a handle; with h == NULL, of the last failed gnssacq_create on this thread. */
const char* gnssacq_last_error(const gnssacq_handle* h);

/* Run kernels on this CUDA stream (a cudaStream_t passed as void*).  NULL is the CUDA legacy default
 * stream (what torch.cuda.current_stream().cuda_stream returns by default); GNSSACQ_OWN_STREAM
 * restores the non-blocking stream the handle created for itself (the initial setting). */
#define GNSSACQ_OWN_STREAM ((void*)(intptr_t)-1)
int gnssacq_set_stream(gnssacq_handle* h, void* cuda_stream);

/* The search (replaces acquisition.m:27-80 minus file I/O): `if_samples` is the byte block
 * acquisition.m:29/34 reads (host memory).  Writes cfg.n_prn rows to out[] in cfg.prn[] order. */
int gnssacq_search(gnssacq_handle* h, const void* if_samples, size_t nbytes,
                   gnssacq_result* out, gnssacq_stats* stats /* may be NULL */);

/* Same, with the IF block already resident in HBM (device pointer). */
int gnssacq_search_device(gnssacq_handle* h, const void* d_if_samples, size_t nbytes,
                          gnssacq_result* out, gnssacq_stats* stats /* may be NULL */);

/* Enqueue only (no host synchronisation, results stay in HBM): for back-to-back timing loops.
 * gnssacq_fetch_results() synchronises and copies the rows of the last enqueued search -- from wherever that
 * search wrote them (the handle's own table, or the device buffer given to gnssacq_enqueue_device_out).
 * out may be NULL when only the timings are wanted; GNSSACQ_ERR_STATE if nothing has been enqueued yet. */
int gnssacq_enqueue_device(gnssacq_handle* h, const void* d_if_samples, size_t nbytes);
int gnssacq_fetch_results(gnssacq_handle* h, gnssacq_result* out, gnssacq_stats* stats /* may be NULL */);
/* Enqueue only, and have K4 write the cfg.n_prn result rows straight into caller-owned HBM
 * (`d_out_rows`, n_prn * sizeof(gnssacq_result) bytes) -- e.g. the send buffer of the NCCL
 * all-gather that assembles the per-rank PRN shards.  Stream-ordered; no host synchronisation. */
int gnssacq_enqueue_device_out(gnssacq_handle* h, const void* d_if_samples, size_t nbytes, void* d_out_rows);

/* Single-process multi-GPU convenience (e.g. for the MEX gateway, which lives in one MATLAB process):
 * `hs[i]` are handles created on different devices (cfg.device) for disjoint PRN shards (cfg.prn[]); the IF
 * block is staged and copied to every device over its own PCIe link, all shards are enqueued, then fetched.
 * Rows land in out[] in handle order (sum of the handles' n_prn).  The one-process-per-GPU path
 * (gnssacq/dist.py: NCCL broadcast + all-gather over NVLink) is the one the benchmark uses. */
int gnssacq_search_multi(gnssacq_handle* const* hs, int32_t n_handles, const void* if_samples, size_t nbytes,
                         gnssacq_result* out);

/* Re-acquisition sweep (BASELINE.json config 4; replaces a loop of SDR_main.m:17-23 over file.skip; the IF
 * ingest of SURVEY 8f-3, acquisition.m:27-38).  `windows[i]` points to the i-th window's IF bytes in HOST memory
 * (what acquisition.m would fread after fseek to skip_i*Sample*dataPrecision*dataType), each at least
 * gnssacq_if_bytes long.  Window i+1 is staged in pinned memory and copied to HBM on a copy stream while window i
 * is searched; all rows come back in one transfer: out[i*n_prn + p] is what gnssacq_search returns for window i.
 * stats (may be NULL): total_ms = host wall time of the sweep, kernel_launches = all launches, kernel times of
 * the last window. */
int gnssacq_sweep(gnssacq_handle* h, const void* const* windows, int32_t n_windows, size_t nbytes_each,
                  gnssacq_result* out, gnssacq_stats* stats);

/* Assisted re-acquisition: per-PRN Doppler windows for every later search on this handle (gnssacq_search,
 * _search_device, _enqueue_device[_out], _search_multi, _sweep, _sweep_file) until cleared.  lo_hz[i] / hi_hz[i]
 * belong to cfg.prn[i]; PRN i is searched over the bins b of the handle's grid with
 * lo_hz[i] <= freq_min_hz + freq_step_hz*b <= hi_hz[i] (the doppler_hz K4 reports).  Only those rows are searched, so
 * the search time follows the number of bins in the windows, not freq_num.  A windowed PRN's row is byte-identical to
 * the row of a one-PRN handle with bin_first / bin_count set to its window's bins (doppler_bin / doppler_hz on this
 * handle's full grid); the int16 means stay those of the whole block.  A PRN whose window holds no bin is not searched:
 * its row has acquired = 0, snr_db = NaN, peak = -1.  lo_hz == hi_hz == NULL clears the windows (full grid again).
 * lo_hz > hi_hz, a NaN bound or exactly one NULL array: GNSSACQ_ERR_INVALID_ARG.  A handle made with bin_count or
 * row_count, or in the multi-GPU exchange: GNSSACQ_ERR_STATE (and gnssacq_xchg_root / _attach / _attach_local refuse
 * a handle with windows set).  Synchronous: waits for the handle's stream and returns once the tables are in HBM. */
int gnssacq_set_doppler_windows(gnssacq_handle* h, const double* lo_hz, const double* hi_hz);

/* ---- one acquisition sharded over several GPUs, exchange through peer memory (no NCCL in the step) -------------
 * SURVEY 8e.  The (PRN, Doppler bin) rows of ONE acquisition are dealt out to `world` handles, one per GPU
 * (processes or one process): whole PRNs per shard when n_prn >= world, otherwise every shard takes all PRNs and a
 * range of bins (gnssacq_shard_plan).  Shard 0 is the root.  Its exchange block -- IF buffer, candidate table of the
 * FULL grid [n_prn][freq_num], flags -- is mapped into the other shards (CUDA IPC between processes,
 * peer access inside one process).  One step:
 *   root   : [H2D of the IF block] -> K1a (publishes "IF ready") -> K1b -> K2 (candidates into its own table)
 *   others : K1a waits for "IF ready", PULLS the IF block out of the root's HBM over NVLink (16-byte vector loads)
 *            -> K1b -> K2, which STORES its row candidates straight into the root's table over NVLink -> "done" flag
 *   root   : waits for every "done" flag -> K4 over the full table (first bin / first code phase over ALL bins,
 *            acquisition.m:62-68) -> rows.
 * Because K4 sees exactly the candidates a single-GPU search computes, the rows are byte-identical for any world.
 * All calls are stream-ordered and return at once, except gnssacq_xchg_fetch.  Every shard must call
 * gnssacq_xchg_enqueue the same number of times (the flags carry a step counter). */
typedef struct gnssacq_shard {
    int32_t rank, world;
    int32_t n_prn_total;                  /* the whole acquisition */
    int32_t prn_total[GNSSACQ_MAX_PRN];
    int32_t freq_num_total;
    int32_t prn_first, prn_count;         /* this shard's rows: PRNs [prn_first, +prn_count) x bins [bin_first, +bin_count) */
    int32_t bin_first, bin_count;
    int32_t row_first, row_count;         /* gnssacq_shard_plan_rows: rows [row_first, +row_count) of that grid, bin-major
                                             (row_count = 0 with plan_rows = 0: the whole rectangle) */
    int32_t plan_rows;                    /* 1 = made by gnssacq_shard_plan_rows */
    int32_t root_extra_permille;          /* its weight argument (the root recomputes the other shards' shares from it) */
} gnssacq_shard;
#define GNSSACQ_IPC_BYTES 64
/* full config + (rank, world) -> this shard's config (`mine`: PRN subset and bin range filled in) and its place */
int gnssacq_shard_plan(const gnssacq_config* full, int32_t rank, int32_t world, gnssacq_config* mine, gnssacq_shard* shard);
/* Row-granular plan: the n_prn x freq_num rows, in the bin-major order the search kernel walks them, are cut into
 * `world` contiguous ranges; every shard keeps all PRNs (their code spectra are cached per handle) and computes only its
 * rows.  The root's range is (1000 + root_extra_permille) / 1000 times the others': the other shards start a step later
 * than the root by the time the IF block needs to reach them (gnssacq_stats.if_pull_ms), so equal shares leave the
 * root waiting at the end of every step (gnssacq_stats.gather_wait_ms); a few per cent more rows on the root level the
 * finish times.  root_extra_permille may be negative (> -1000).  Result rows do not depend on the plan. */
int gnssacq_shard_plan_rows(const gnssacq_config* full, int32_t rank, int32_t world, int32_t root_extra_permille,
                            gnssacq_config* mine, gnssacq_shard* shard);
/* root only: allocate the exchange block; ipc_out (GNSSACQ_IPC_BYTES, may be NULL) receives the handle other
 * PROCESSES open with gnssacq_xchg_attach */
int gnssacq_xchg_root(gnssacq_handle* root, const gnssacq_shard* shard, void* ipc_out);
int gnssacq_xchg_attach(gnssacq_handle* h, const gnssacq_shard* shard, const void* root_ipc);        /* other process */
int gnssacq_xchg_attach_local(gnssacq_handle* h, const gnssacq_shard* shard, gnssacq_handle* root); /* same process */
/* device pointer of the root's IF buffer (gnssacq_if_bytes): for callers whose samples are already in HBM */
void* gnssacq_xchg_if_buffer(gnssacq_handle* root);
/* one step of this shard.  host_if: root only -- NULL = the IF block is already in the exchange block's buffer,
 * else it is copied there first: pageable memory through the library's pinned staging buffer (the caller's
 * buffer is free on return), page-locked memory directly (keep it unchanged until gnssacq_xchg_fetch) */
int gnssacq_xchg_enqueue(gnssacq_handle* h, const void* host_if, size_t nbytes);
/* root only: wait for every shard, K4 over the full table (stream-ordered, no host sync) */
int gnssacq_xchg_finish(gnssacq_handle* root);
/* root only: host sync + the n_prn_total rows of the last finished step */
int gnssacq_xchg_fetch(gnssacq_handle* root, gnssacq_result* out, gnssacq_stats* stats /* may be NULL */);

/* The same sweep read straight from a recording file (BASELINE config 4: one acquisition every epoch_ms over a
 * 90 s recording = 900 windows).  Window j = the bytes acquisition.m:27-34 reads with file.skip = skip_ms +
 * j*epoch_ms: noncoh_blocks*coh_ms ms from byte (skip_ms + j*epoch_ms) * samples_per_ms * dataPrecision *
 * dataType (SDR_main.m:17-23 run once per epoch).  fseek + fread fill the library's pinned staging buffers
 * directly while the previous window is searched.  A window that runs past the end of the file:
 * GNSSACQ_ERR_SHORT_BUFFER (MATLAB's fread would return fewer samples and acquisition.m:56 would then fail). */
int gnssacq_sweep_file(gnssacq_handle* h, const char* path, int64_t skip_ms, int32_t epoch_ms, int32_t n_windows,
                       gnssacq_result* out, gnssacq_stats* stats);

/* Tracking correlators (SURVEY 8f-2; replaces trackingCT.m:85-118, and with 25 taps the correlator bank of
 * trackingCT_POS_updated_multicorrelator.m:207-260).  The loop filters stay with the caller (trackingCT.m:135-150).
 * gnssacq_track_load copies a segment of the recording (same sample format as the handle's config) to HBM once;
 * gnssacq_correlate then runs ONE integration period for a batch of channels against it, in float64:
 *   carr   = exp(i*(2*pi*carrier_hz*n/Fs + rem_phase)), n = 0..num_samples-1            (:103-106)
 *   I[tap] = sum(code_tap .* imag(x .* carr)),  Q[tap] = sum(code_tap .* real(x .* carr))  (:112-117)
 *   code_tap(n) = Code(ceil(spacing[tap] + rem_chip + n*code_hz/Fs) + 1), Code = [CA(end) CA CA(1)]  (:66,96-101)
 * with x the num_samples samples starting sample_offset samples into the loaded segment (int16 data: the
 * per-integration means of I and Q are removed, :90-92).  out_i / out_q: [n_channels][n_taps]. */
#define GNSSACQ_TRACK_MAX_PRN 37
typedef struct gnssacq_channel {
    int32_t prn;              /* Acquired.sv(svindex) */
    int32_t num_samples;      /* numSample (trackingCT.m:78) */
    int64_t sample_offset;    /* position of the integration in the loaded segment, in samples (ftell/(precision*type)) */
    double carrier_hz;        /* carrierFreq */
    double rem_phase;         /* remPhase */
    double code_hz;           /* codeFreq */
    double rem_chip;          /* remChip */
} gnssacq_channel;
int gnssacq_track_load(gnssacq_handle* h, const void* if_samples, size_t nbytes);
int gnssacq_correlate(gnssacq_handle* h, int32_t n_channels, const gnssacq_channel* channels, int32_t n_taps,
                      const double* spacing_chips, double* out_i, double* out_q);

/* The whole conventional tracking loop of trackingCT.m:70-172 on the device: n_periods integration periods of every
 * channel against the loaded segment, early/prompt/late correlators, DLL and PLL discriminators and loop filters
 * (calcLoopCoef.m:41-45, trackingCT.m:135-150) in float64, one thread-block cluster per channel, no host round
 * trip per millisecond.  start[c]: prn, sample_offset = Sample - AcqCodeDelay + 1 (+ skip*Sample) (trackingCT.m:60),
 * carrier_hz = Acquired.fineFreq (also the NCO basis), code_hz = codeFreqBasis, rem_chip = rem_phase = 0
 * (num_samples is ignored).  out[c*n_periods + i] holds the TckResultCT fields of period i (trackingCT.m:153-172).
 * Running out of samples ("Not enough raw data", :107-111) returns GNSSACQ_ERR_SHORT_BUFFER. */
typedef struct gnssacq_loop_params {
    double dll_bw, dll_damp, dll_gain;   /* track.DLLBW, DLLDamp, DLLGain   (initParameters.m:60-62) */
    double pll_bw, pll_damp, pll_gain;   /* track.PLLBW, PLLDamp, PLLGain   (initParameters.m:63-65) */
    double spacing_chips;                /* track.CorrelatorSpacing         (initParameters.m:59)    */
} gnssacq_loop_params;
typedef struct gnssacq_track_record {
    double P_i, P_q, E_i, E_q, L_i, L_q;  /* :115-117 */
    double pll_discri, dll_discri;        /* :146, :139 */
    double rem_chip, code_hz, carrier_hz, rem_phase;   /* values AFTER the period's update, as stored at :164-167 */
    int64_t sample_end;                   /* absoluteSample/(dataPrecision*dataType): position after the read (:171) */
    int32_t num_samples;                  /* :78 */
    int32_t reserved;
} gnssacq_track_record;
int gnssacq_loop_params_default(gnssacq_loop_params* p);
int gnssacq_track(gnssacq_handle* h, int32_t n_channels, const gnssacq_channel* start, const gnssacq_loop_params* loops,
                  int32_t n_periods, gnssacq_track_record* out);

/* Fine-frequency stage (replaces acquisition.m:89-121; SURVEY 8f-1).  `if_long` is the (L+1) ms block
 * acquisition.m:91/96 reads from the same file offset (host memory); for each of the n_sv acquired SVs
 * (prn[i], code_phase[i] = Acquired.codedelay) the code-stripped L ms are zero-padded to
 * fftlength = L*samples_per_ms*noncoh_blocks and the spectral peak gives out_hz[i] = Acquired.fineFreq
 * (absolute Hz; for I/Q data  -idx*(Fs/fftlength) + Fs/2  with the reference's 1-based idx). */
int gnssacq_fine_frequency(gnssacq_handle* h, const void* if_long, size_t nbytes, int32_t L, int32_t n_sv,
                           const int32_t* prn, const int32_t* code_phase, double* out_hz);

/* ---- table generators (host side, replace generateCAcode.m and acquisition.m:50-51) ---- */
int gnssacq_ca_code(int32_t prn, int8_t out_chips[1023]);
int gnssacq_code_replica(const gnssacq_config* cfg, int32_t prn, int8_t* out_samples /* samples_per_ms */);

/* ---- diagnostics used by the parity tests ---- */
/* Power surface of PRN index `prn_index` (row-major freq_num x samples_per_ms floats, lag order of
 * acquisition.m:59) from the last search; needs cfg.keep_surface = 1. */
int gnssacq_read_surface(gnssacq_handle* h, int32_t prn_index, float* out);
/* Measured FP32 FMA throughput of `device` in TFLOP/s (2 flops per FFMA; dependent-chain-free FFMA
 * loop on every SM, CUDA-event timed): the denominator of the FP32 roofline, since
 * MEASURED_PEAKS.json only records HBM and BF16 tensor peaks. */
int gnssacq_fp32_peak_tflops(int32_t device, double* out_tflops);
/* Forward DFT of samples_per_ms complex floats (interleaved re,im; host pointers) through the engine.  For a
 * padded samples_per_ms N the N-point DFT is a Bluestein (chirp-z) convolution through the engine's longer
 * transform, the same path as the fine-frequency stage's DFTs. */
int gnssacq_fft_forward(gnssacq_handle* h, const float* in, float* out);

#ifdef __cplusplus
}
#endif
#endif /* GNSSACQ_H_ */
