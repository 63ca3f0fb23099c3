/* gnssacq_mex.c -- MEX gateway from MATLAB to libgnssacq.so (include/gnssacq.h).
 *
 * The FIRST argument is always the mode, a char row; every mode is dispatched by comparing that string
 * (never by counting arguments):
 *   rows     = gnssacq_mex('search',     raw, cfg)                          coarse search (acquisition.m:41-80)
 *   fineFreq = gnssacq_mex('fine',       longraw, cfg, L, sv, codedelay)    fine-frequency stage (:83-127)
 *   rows3    = gnssacq_mex('sweep_file', path, cfg, skip_ms, epoch_ms, n)   n re-acquisitions straight from a recording
 *              gnssacq_mex('track_load', segment, cfg)                      recording segment -> HBM (tracking)
 *   [I, Q]   = gnssacq_mex('correlate',  channels, cfg, spacing)            one integration period, all channels
 *              channels: 7 x n double, rows [prn; numSample; sample_offset; carrierFreq; remPhase; codeFreq;
 *              remChip] (trackingCT.m:42-58,78); I, Q: n x numel(spacing) (trackingCT.m:115-117)
 *   rec      = gnssacq_mex('track',      channels, cfg, loops, n_periods)   closed DLL/PLL loop on the device
 *              loops: [DLLBW DLLDamp DLLGain PLLBW PLLDamp PLLGain CorrelatorSpacing]; rec: 14 x n_periods x n,
 *              rows [P_i P_q E_i E_q L_i L_q PLLdiscri DLLdiscri remChip codeFreq carrierFreq remPhase
 *              sample_end numSample] (trackingCT.m:153-172)
 *   [rec, I, Q] = gnssacq_mex('track', channels, cfg, loops, n_periods, spacing)   the same loop, and every period the
 *              correlator bank at spacing (1 x n_taps, trackingCT_POS_updated_multicorrelator.m:41,207-260); I, Q:
 *              n_taps x n_periods x n.  The bank only observes: rec is what the 5-argument form returns
 *              gnssacq_mex('close')                                         destroy the handles now
 *
 * `raw` is the block acquisition.m:29/34 reads, passed as int8 (or int16) WITHOUT conversion to
 * double; `cfg` is a scalar struct whose fields are named after gnssacq_config, plus
 *   cfg.n_gpus   (default 1)  number of GPUs the PRN list is sharded over (PRN-major, SURVEY 8e): the gateway
 *                             keeps one handle per GPU and 'search' goes through gnssacq_search_multi
 *   cfg.devices  (optional)   the CUDA device ordinals to use, numel >= n_gpus (default 0 .. n_gpus-1)
 *   cfg.doppler_lo_hz, cfg.doppler_hi_hz  (optional, 'search' and 'sweep_file', both or neither)  n_prn-element
 *                             per-PRN Doppler windows (gnssacq_set_doppler_windows): PRN cfg.prn(i) is searched only
 *                             over the grid bins with doppler_lo_hz(i) <= doppler_hz <= doppler_hi_hz(i); a PRN whose
 *                             window holds no bin comes back with acquired 0, snr_db NaN, peak -1.  Left out: the
 *                             full grid
 * 'search' returns an n_prn x 8 double matrix, one row per searched PRN, in the order of cfg.prn:
 *   [prn acquired code_phase doppler_bin doppler_hz peak noise_meansq snr_db]
 * ('sweep_file': n_prn x 8 x n).  The handles are kept in statics between calls (mexLock) and rebuilt only when
 * cfg changes; they are destroyed by mexAtExit.  Library errors become MATLAB errors gnssacq:e<code>.
 * Modes other than 'search' use the first handle (one GPU).
 *
 * SOURCE-ONLY DELIVERABLE: neither MATLAB nor Octave (mex.h) exists in the build image, so this
 * file is compile-checked against tests/stubs/mex.h only.  Build on a MATLAB host with
 *   mex -I<repo>/include gnssacq_mex.c -L<repo>/assignment-for-aae6102_gnss-sdr_b200/gnssacq -lgnssacq
 */
#include <stdint.h>
#include <string.h>
#include "mex.h"
#include "gnssacq.h"

#define MAX_GPUS 8
static gnssacq_handle* g_handle[MAX_GPUS];
static int g_n_handles = 0;
static gnssacq_config g_cfg;
static int g_gpus = 0, g_dev[MAX_GPUS];
static int g_have_cfg = 0, g_locked = 0, g_windows = 0;

static void close_all(void) {
    int i;
    for (i = 0; i < g_n_handles; ++i)
        if (g_handle[i]) { gnssacq_destroy(g_handle[i]); g_handle[i] = NULL; }
    g_n_handles = 0;
    g_have_cfg = 0;
    g_windows = 0;
}

static double field(const mxArray* s, const char* name, double dflt) {
    const mxArray* f = mxGetField(s, 0, name);
    return (f && mxGetNumberOfElements(f) >= 1) ? mxGetScalar(f) : dflt;
}

static void fail(int rc, const char* msg) {
    char id[32];
    sprintf(id, "gnssacq:e%d", -rc);
    mexErrMsgIdAndTxt(id, "%s", msg ? msg : "gnssacq error");
}

static void channels_from(const mxArray* a, gnssacq_channel* ch, int n_ch, int keep_num_samples) {
    const double* m = mxGetPr(a);
    int i;
    for (i = 0; i < n_ch; ++i) {
        ch[i].prn = (int32_t)m[7 * i];
        ch[i].num_samples = keep_num_samples ? (int32_t)m[7 * i + 1] : 0;
        ch[i].sample_offset = (int64_t)m[7 * i + 2];
        ch[i].carrier_hz = m[7 * i + 3];
        ch[i].rem_phase = m[7 * i + 4];
        ch[i].code_hz = m[7 * i + 5];
        ch[i].rem_chip = m[7 * i + 6];
    }
}

static void rows_to_matrix(const gnssacq_result* rows, int n, double* out) {
    int i;
    for (i = 0; i < n; ++i) {
        out[i + 0 * n] = rows[i].prn;
        out[i + 1 * n] = rows[i].acquired;
        out[i + 2 * n] = rows[i].code_phase;
        out[i + 3 * n] = rows[i].doppler_bin;
        out[i + 4 * n] = rows[i].doppler_hz;
        out[i + 5 * n] = rows[i].peak;
        out[i + 6 * n] = rows[i].noise_meansq;
        out[i + 7 * n] = rows[i].snr_db;
    }
}

/* cfg struct -> library config + GPU list; (re)build the handles when anything changed */
static void ensure_handles(const mxArray* cs, gnssacq_config* cfg_out) {
    gnssacq_config c;
    const mxArray *prn, *devs;
    int i, g, gpus, dev[MAX_GPUS], rc, same;
    gnssacq_config_default(&c);
    c.fs_hz = field(cs, "fs_hz", c.fs_hz);
    c.if_hz = field(cs, "if_hz", c.if_hz);
    c.code_hz = field(cs, "code_hz", c.code_hz);
    c.samples_per_ms = (int32_t)field(cs, "samples_per_ms", c.samples_per_ms);
    c.data_type = (int32_t)field(cs, "data_type", c.data_type);
    c.data_precision = (int32_t)field(cs, "data_precision", c.data_precision);
    c.freq_min_hz = field(cs, "freq_min_hz", c.freq_min_hz);
    c.freq_step_hz = field(cs, "freq_step_hz", c.freq_step_hz);
    c.freq_num = (int32_t)field(cs, "freq_num", c.freq_num);
    c.noncoh_blocks = (int32_t)field(cs, "noncoh_blocks", c.noncoh_blocks);
    c.coh_ms = (int32_t)field(cs, "coh_ms", c.coh_ms);
    c.snr_threshold_db = field(cs, "snr_threshold_db", c.snr_threshold_db);
    c.device = (int32_t)field(cs, "device", -1);
    prn = mxGetField(cs, 0, "prn");
    if (prn) {
        size_t n = mxGetNumberOfElements(prn);
        const double* p = mxGetPr(prn);
        if (n > GNSSACQ_MAX_PRN) fail(GNSSACQ_ERR_INVALID_ARG, "too many PRNs");
        c.n_prn = (int32_t)n;
        for (i = 0; i < GNSSACQ_MAX_PRN; ++i) c.prn[i] = (i < (int)n) ? (int32_t)p[i] : 0;
    }
    gpus = (int)field(cs, "n_gpus", 1);
    if (gpus < 1 || gpus > MAX_GPUS) fail(GNSSACQ_ERR_INVALID_ARG, "cfg.n_gpus must be 1..8");
    if (gpus > c.n_prn) gpus = c.n_prn;               /* whole PRNs per GPU (SURVEY 8e); bin splits: gnssacq_search_split */
    devs = mxGetField(cs, 0, "devices");
    if (devs && (int)mxGetNumberOfElements(devs) < gpus) fail(GNSSACQ_ERR_INVALID_ARG, "cfg.devices shorter than cfg.n_gpus");
    for (g = 0; g < gpus; ++g) dev[g] = devs ? (int)mxGetPr(devs)[g] : (gpus == 1 ? c.device : g);

    same = g_have_cfg && g_gpus == gpus && memcmp(&c, &g_cfg, sizeof c) == 0;
    for (g = 0; same && g < gpus; ++g) same = (dev[g] == g_dev[g]);
    if (!same) {
        close_all();
        for (g = 0; g < gpus; ++g) {                   /* PRN-major shard g: PRNs [lo, hi) of the list */
            gnssacq_config cg = c;
            const int lo = g * c.n_prn / gpus, hi = (g + 1) * c.n_prn / gpus;
            cg.n_prn = hi - lo;
            for (i = 0; i < GNSSACQ_MAX_PRN; ++i) cg.prn[i] = (i < hi - lo) ? c.prn[lo + i] : 0;
            cg.device = dev[g];
            rc = gnssacq_create(&cg, &g_handle[g]);
            if (rc != GNSSACQ_OK) { close_all(); fail(rc, gnssacq_last_error(NULL)); }
            g_n_handles = g + 1;
        }
        if (!g_locked) { mexLock(); mexAtExit(close_all); g_locked = 1; }
        g_cfg = c;
        g_gpus = gpus;
        for (g = 0; g < gpus; ++g) g_dev[g] = dev[g];
        g_have_cfg = 1;
    }
    *cfg_out = c;
}

/* cfg.doppler_lo_hz / cfg.doppler_hi_hz -> every handle's slice of the windows (PRN-major shards, as in
 * ensure_handles); neither field: clear windows an earlier call set */
static void apply_windows(const mxArray* cs, const gnssacq_config* c) {
    const mxArray* lo = mxGetField(cs, 0, "doppler_lo_hz");
    const mxArray* hi = mxGetField(cs, 0, "doppler_hi_hz");
    int g, rc;
    if (!lo && !hi) {
        for (g = 0; g_windows && g < g_n_handles; ++g) {
            rc = gnssacq_set_doppler_windows(g_handle[g], NULL, NULL);
            if (rc != GNSSACQ_OK) fail(rc, gnssacq_last_error(g_handle[g]));
        }
        g_windows = 0;
        return;
    }
    if (!lo || !hi || !mxIsDouble(lo) || !mxIsDouble(hi) || (int)mxGetNumberOfElements(lo) != c->n_prn ||
        (int)mxGetNumberOfElements(hi) != c->n_prn)
        fail(GNSSACQ_ERR_INVALID_ARG, "cfg.doppler_lo_hz and cfg.doppler_hi_hz must both be double with n_prn elements");
    g_windows = 1;
    for (g = 0; g < g_n_handles; ++g) {
        const int first = g * c->n_prn / g_n_handles;
        rc = gnssacq_set_doppler_windows(g_handle[g], mxGetPr(lo) + first, mxGetPr(hi) + first);
        if (rc != GNSSACQ_OK) fail(rc, gnssacq_last_error(g_handle[g]));
    }
}

void mexFunction(int nlhs, mxArray* plhs[], int nrhs, const mxArray* prhs[]) {
    static const char* usage =
        "usage: gnssacq_mex(mode, ...), mode = 'search' | 'fine' | 'sweep_file' | 'track_load' | 'correlate' | 'track' | 'close'"
        " ('search' and 'sweep_file' take optional per-PRN windows cfg.doppler_lo_hz / cfg.doppler_hi_hz)";
    char mode[24];
    gnssacq_config c;
    size_t nbytes;
    int rc, i;

    if (nrhs < 1 || !mxIsChar(prhs[0]) || mxGetString(prhs[0], mode, sizeof mode) != 0) fail(GNSSACQ_ERR_INVALID_ARG, usage);
    if (strcmp(mode, "close") == 0) { close_all(); return; }
    if (nrhs < 3 || !mxIsStruct(prhs[2])) fail(GNSSACQ_ERR_INVALID_ARG, usage);
    ensure_handles(prhs[2], &c);
    nbytes = mxGetNumberOfElements(prhs[1]) * mxGetElementSize(prhs[1]);

    if (strcmp(mode, "search") == 0) {                 /* acquisition.m:41-80 */
        gnssacq_result* rows;
        if (nrhs != 3 || !(mxIsInt8(prhs[1]) || mxIsInt16(prhs[1]))) fail(GNSSACQ_ERR_INVALID_ARG, "search: raw must be int8 or int16");
        apply_windows(prhs[2], &c);
        rows = (gnssacq_result*)mxMalloc(sizeof(gnssacq_result) * (size_t)c.n_prn);
        rc = (g_n_handles == 1) ? gnssacq_search(g_handle[0], mxGetData(prhs[1]), nbytes, rows, NULL)
                                : gnssacq_search_multi(g_handle, g_n_handles, mxGetData(prhs[1]), nbytes, rows);
        if (rc != GNSSACQ_OK) { mxFree(rows); fail(rc, gnssacq_last_error(g_handle[0])); }
        plhs[0] = mxCreateDoubleMatrix((mwSize)c.n_prn, 8, mxREAL);
        rows_to_matrix(rows, c.n_prn, mxGetPr(plhs[0]));
        mxFree(rows);
    } else if (strcmp(mode, "fine") == 0) {            /* acquisition.m:83-127 */
        int n_sv;
        const double *svd, *cdd;
        int32_t *sv, *cd;
        if (nrhs != 6 || !(mxIsInt8(prhs[1]) || mxIsInt16(prhs[1]))) fail(GNSSACQ_ERR_INVALID_ARG, "fine: (longraw, cfg, L, sv, codedelay)");
        n_sv = (int)mxGetNumberOfElements(prhs[4]);
        if ((int)mxGetNumberOfElements(prhs[5]) != n_sv) fail(GNSSACQ_ERR_INVALID_ARG, "sv and codedelay differ in length");
        svd = mxGetPr(prhs[4]);
        cdd = mxGetPr(prhs[5]);
        sv = (int32_t*)mxMalloc(sizeof(int32_t) * (size_t)(n_sv + 1));
        cd = (int32_t*)mxMalloc(sizeof(int32_t) * (size_t)(n_sv + 1));
        for (i = 0; i < n_sv; ++i) { sv[i] = (int32_t)svd[i]; cd[i] = (int32_t)cdd[i]; }
        plhs[0] = mxCreateDoubleMatrix(1, (mwSize)n_sv, mxREAL);
        rc = gnssacq_fine_frequency(g_handle[0], mxGetData(prhs[1]), nbytes, (int32_t)mxGetScalar(prhs[3]), n_sv,
                                    sv, cd, mxGetPr(plhs[0]));
        mxFree(sv);
        mxFree(cd);
        if (rc != GNSSACQ_OK) fail(rc, gnssacq_last_error(g_handle[0]));
    } else if (strcmp(mode, "sweep_file") == 0) {      /* SDR_main.m:17-23 once per epoch, read by the library */
        char path[1024];
        int n_win, w;
        gnssacq_result* rows;
        mwSize dims[3];
        if (nrhs != 6 || !mxIsChar(prhs[1]) || mxGetString(prhs[1], path, sizeof path) != 0)
            fail(GNSSACQ_ERR_INVALID_ARG, "sweep_file: (path, cfg, skip_ms, epoch_ms, n_windows)");
        n_win = (int)mxGetScalar(prhs[5]);
        if (n_win < 1) fail(GNSSACQ_ERR_INVALID_ARG, "sweep_file: n_windows >= 1");
        if (g_n_handles != 1) fail(GNSSACQ_ERR_INVALID_ARG, "sweep_file runs on one GPU (cfg.n_gpus = 1)");
        apply_windows(prhs[2], &c);
        rows = (gnssacq_result*)mxMalloc(sizeof(gnssacq_result) * (size_t)c.n_prn * (size_t)n_win);
        rc = gnssacq_sweep_file(g_handle[0], path, (int64_t)mxGetScalar(prhs[3]), (int32_t)mxGetScalar(prhs[4]), n_win, rows, NULL);
        if (rc != GNSSACQ_OK) { mxFree(rows); fail(rc, gnssacq_last_error(g_handle[0])); }
        dims[0] = (mwSize)c.n_prn; dims[1] = 8; dims[2] = (mwSize)n_win;
        plhs[0] = mxCreateNumericArray(3, dims, mxDOUBLE_CLASS, mxREAL);
        for (w = 0; w < n_win; ++w) rows_to_matrix(rows + (size_t)w * c.n_prn, c.n_prn, mxGetPr(plhs[0]) + (size_t)w * 8 * c.n_prn);
        mxFree(rows);
    } else if (strcmp(mode, "track_load") == 0) {      /* tracking: keep the segment in HBM */
        if (nrhs != 3 || !(mxIsInt8(prhs[1]) || mxIsInt16(prhs[1]))) fail(GNSSACQ_ERR_INVALID_ARG, "track_load: (segment, cfg)");
        rc = gnssacq_track_load(g_handle[0], mxGetData(prhs[1]), nbytes);
        if (rc != GNSSACQ_OK) fail(rc, gnssacq_last_error(g_handle[0]));
    } else if (strcmp(mode, "correlate") == 0) {       /* tracking correlators (trackingCT.m:85-118) */
        int n_ch, n_taps, t;
        gnssacq_channel* ch;
        double *oi, *oq, *pi, *pq;
        if (nrhs != 4 || !mxIsDouble(prhs[1]) || mxGetM(prhs[1]) != 7) fail(GNSSACQ_ERR_INVALID_ARG, "correlate: channels must be a 7 x n double matrix");
        n_ch = (int)mxGetN(prhs[1]);
        n_taps = (int)mxGetNumberOfElements(prhs[3]);
        ch = (gnssacq_channel*)mxMalloc(sizeof(gnssacq_channel) * (size_t)(n_ch + 1));
        oi = (double*)mxMalloc(sizeof(double) * (size_t)(n_ch * n_taps + 1));
        oq = (double*)mxMalloc(sizeof(double) * (size_t)(n_ch * n_taps + 1));
        channels_from(prhs[1], ch, n_ch, 1);
        rc = gnssacq_correlate(g_handle[0], n_ch, ch, n_taps, mxGetPr(prhs[3]), oi, oq);
        if (rc != GNSSACQ_OK) { mxFree(ch); mxFree(oi); mxFree(oq); fail(rc, gnssacq_last_error(g_handle[0])); }
        plhs[0] = mxCreateDoubleMatrix((mwSize)n_ch, (mwSize)n_taps, mxREAL);
        pi = mxGetPr(plhs[0]);
        if (nlhs > 1) { plhs[1] = mxCreateDoubleMatrix((mwSize)n_ch, (mwSize)n_taps, mxREAL); pq = mxGetPr(plhs[1]); } else pq = NULL;
        for (i = 0; i < n_ch; ++i)
            for (t = 0; t < n_taps; ++t) {             /* row-major [channel][tap] -> MATLAB column-major */
                pi[i + t * n_ch] = oi[i * n_taps + t];
                if (pq) pq[i + t * n_ch] = oq[i * n_taps + t];
            }
        mxFree(ch); mxFree(oi); mxFree(oq);
    } else if (strcmp(mode, "track") == 0) {           /* whole conventional loop (trackingCT.m:70-172) */
        const double* lp;
        int n_ch, n_per, k;
        gnssacq_channel* ch;
        gnssacq_track_record* rec;
        gnssacq_loop_params loops;
        mwSize dims[3];
        double *out, *bi = NULL, *bq = NULL;
        int n_taps = 0;
        if ((nrhs != 5 && nrhs != 6) || !mxIsDouble(prhs[1]) || mxGetM(prhs[1]) != 7 || mxGetNumberOfElements(prhs[3]) != 7 ||
            (nrhs == 6 && !mxIsDouble(prhs[5])))
            fail(GNSSACQ_ERR_INVALID_ARG, "track: (channels 7 x n, cfg, loops 1 x 7, n_periods[, spacing 1 x n_taps])");
        lp = mxGetPr(prhs[3]);
        n_ch = (int)mxGetN(prhs[1]);
        n_per = (int)mxGetScalar(prhs[4]);
        if (n_per < 1) fail(GNSSACQ_ERR_INVALID_ARG, "track: n_periods >= 1");
        loops.dll_bw = lp[0]; loops.dll_damp = lp[1]; loops.dll_gain = lp[2];
        loops.pll_bw = lp[3]; loops.pll_damp = lp[4]; loops.pll_gain = lp[5]; loops.spacing_chips = lp[6];
        ch = (gnssacq_channel*)mxMalloc(sizeof(gnssacq_channel) * (size_t)(n_ch + 1));
        rec = (gnssacq_track_record*)mxMalloc(sizeof(gnssacq_track_record) * ((size_t)n_ch * (size_t)n_per + 1));
        channels_from(prhs[1], ch, n_ch, 0);
        if (nrhs == 6) {                               /* I, Q: [channel][period][tap] = n_taps x n_periods x n */
            n_taps = (int)mxGetNumberOfElements(prhs[5]);
            dims[0] = (mwSize)n_taps; dims[1] = (mwSize)n_per; dims[2] = (mwSize)n_ch;
            if (nlhs > 1) { plhs[1] = mxCreateNumericArray(3, dims, mxDOUBLE_CLASS, mxREAL); bi = mxGetPr(plhs[1]); }
            else bi = (double*)mxMalloc(sizeof(double) * ((size_t)n_taps * n_per * n_ch + 1));
            if (nlhs > 2) { plhs[2] = mxCreateNumericArray(3, dims, mxDOUBLE_CLASS, mxREAL); bq = mxGetPr(plhs[2]); }
            else bq = (double*)mxMalloc(sizeof(double) * ((size_t)n_taps * n_per * n_ch + 1));
            rc = gnssacq_track_bank(g_handle[0], n_ch, ch, &loops, n_per, n_taps, mxGetPr(prhs[5]), rec, bi, bq);
            if (nlhs <= 1) mxFree(bi);
            if (nlhs <= 2) mxFree(bq);
        } else {
            rc = gnssacq_track(g_handle[0], n_ch, ch, &loops, n_per, rec);
        }
        if (rc != GNSSACQ_OK) { mxFree(ch); mxFree(rec); fail(rc, gnssacq_last_error(g_handle[0])); }
        dims[0] = 14; dims[1] = (mwSize)n_per; dims[2] = (mwSize)n_ch;
        plhs[0] = mxCreateNumericArray(3, dims, mxDOUBLE_CLASS, mxREAL);
        out = mxGetPr(plhs[0]);
        for (i = 0; i < n_ch; ++i)
            for (k = 0; k < n_per; ++k) {
                const gnssacq_track_record* r = &rec[(size_t)i * n_per + k];
                double* o = out + 14 * ((size_t)i * n_per + k);
                o[0] = r->P_i; o[1] = r->P_q; o[2] = r->E_i; o[3] = r->E_q; o[4] = r->L_i; o[5] = r->L_q;
                o[6] = r->pll_discri; o[7] = r->dll_discri; o[8] = r->rem_chip; o[9] = r->code_hz;
                o[10] = r->carrier_hz; o[11] = r->rem_phase; o[12] = (double)r->sample_end; o[13] = r->num_samples;
            }
        mxFree(ch); mxFree(rec);
    } else {
        fail(GNSSACQ_ERR_INVALID_ARG, usage);
    }
    (void)nlhs;
}
