// gnss_track.cu -- tracking on the resident recording (include/gnssacq.h: gnssacq_track_load, gnssacq_correlate,
// gnssacq_track): K7 correlators for a batch of channels, K8 the whole DLL/PLL loop on the device.
#include <cooperative_groups.h>
#include <vector>

#include "gnss_host.h"

using namespace gnss;

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
                     step = state[par].step;
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
    }
    cluster.sync();                                        // nobody exits while its slots may still be read
}

// Tracking correlators, SURVEY 8f-2.  gnssacq_track_load keeps a segment of the recording resident in HBM;
// gnssacq_correlate then runs one integration period for a batch of channels against it.
extern "C" {

int gnssacq_track_load(gnssacq_handle* h, const void* if_samples, size_t nbytes) {
    if (!h || !if_samples || nbytes == 0) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    h->trk_bytes = 0;
    if (h->trk_cap < nbytes) {
        h->trk_cap = 0;
        CU(alloc(h->d_trk_raw, nbytes), GNSSACQ_ERR_NOMEM);
        h->trk_cap = nbytes;
    }
    if (!h->trk) {
        auto t = std::make_unique<TrackState>();
        std::vector<int8_t> ca((size_t)GNSSACQ_TRACK_MAX_PRN * 1023);
        for (int p = 1; p <= GNSSACQ_TRACK_MAX_PRN; ++p) ca_chips(p, ca.data() + (size_t)(p - 1) * 1023);
        CU(alloc(t->ca, ca.size()));
        CU(alloc(t->ch, kTrackMaxChannels * sizeof(gnssacq_channel)));
        CU(alloc(t->spacing, kTrackMaxTaps * sizeof(double)));
        CU(alloc(t->partial, (size_t)kTrackMaxChannels * kTrackChunks * kTrackMaxTaps * 2 * sizeof(double)));
        CU(alloc(t->out, (size_t)kTrackMaxChannels * kTrackMaxTaps * 2 * sizeof(double)));
        CU(alloc(t->mean, (size_t)kTrackMaxChannels * 2 * sizeof(double)));
        CU(alloc(t->status, sizeof(int)));
        CU(alloc(t->h_out, (size_t)kTrackMaxChannels * kTrackMaxTaps * 2 * sizeof(double)));
        CU(cudaMemcpyAsync(t->ca.get(), ca.data(), ca.size(), cudaMemcpyHostToDevice, h->stream));
        CU(cudaStreamSynchronize(h->stream));                        // `ca` is a temporary
        h->trk = std::move(t);
    }
    CU(cudaMemcpyAsync(h->d_trk_raw.get(), if_samples, nbytes, cudaMemcpyHostToDevice, h->stream));
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
    CU(cudaMemcpyAsync(h->trk->ch.get(), ch, n_channels * sizeof(gnssacq_channel), cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(h->trk->spacing.get(), spacing_chips, n_taps * sizeof(double), cudaMemcpyHostToDevice, s));
    TrackArgs a;
    a.raw = h->d_trk_raw.get();
    a.data_type = c.data_type;
    a.precision = c.data_precision;
    a.fs_hz = c.fs_hz;
    a.ch = h->trk->ch.get();
    a.n_taps = n_taps;
    a.spacing = h->trk->spacing.get();
    a.ca = h->trk->ca.get();
    a.mean = nullptr;
    a.partial = h->trk->partial.get();
    if (c.data_precision == 2) {
        track_mean_kernel<<<n_channels, kTrackThreads, 0, s>>>(a, h->trk->mean.get());
        a.mean = h->trk->mean.get();
    }
    const dim3 grid(kTrackChunks, (unsigned)n_channels, (unsigned)((n_taps + kTrackTapsPerThread - 1) / kTrackTapsPerThread));
    correlate_kernel<<<grid, kTrackThreads, 0, s>>>(a);
    const int n_elems = n_channels * n_taps * 2;
    correlate_finish_kernel<<<(n_elems + 127) / 128, 128, 0, s>>>(h->trk->partial.get(), n_taps, n_elems, h->trk->out.get());
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(h->trk->h_out.get(), h->trk->out.get(), n_elems * sizeof(double), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    const double* r = h->trk->h_out.get();
    for (int i = 0; i < n_channels * n_taps; ++i) { out_i[i] = r[2 * i]; out_q[i] = r[2 * i + 1]; }
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
        h->trk_rec_cap = 0;
        CU(alloc(h->d_trk_rec, n_rec * sizeof(gnssacq_track_record)));
        h->trk_rec_cap = n_rec;
    }
    CU(cudaMemsetAsync(h->trk->status.get(), 0, sizeof(int), s));
    CU(cudaMemsetAsync(h->d_trk_rec.get(), 0, n_rec * sizeof(gnssacq_track_record), s));
    CU(cudaMemcpyAsync(h->trk->ch.get(), start, n_channels * sizeof(gnssacq_channel), cudaMemcpyHostToDevice, s));
    LoopArgs a;
    a.raw = h->d_trk_raw.get();
    a.total_samples = total;
    a.data_type = c.data_type;
    a.precision = c.data_precision;
    a.fs_hz = c.fs_hz;
    a.code_basis_hz = c.code_hz;
    a.start = h->trk->ch.get();
    a.ca = h->trk->ca.get();
    a.lp = *loops;
    a.n_periods = n_periods;
    a.out = h->d_trk_rec.get();
    a.status = h->trk->status.get();
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
    CU(cudaMemcpyAsync(out, h->d_trk_rec.get(), n_rec * sizeof(gnssacq_track_record), cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(&status, h->trk->status.get(), sizeof(int), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    if (status) return fail(h, GNSSACQ_ERR_SHORT_BUFFER, "Not enough raw data (trackingCT.m:107-111): a channel ran past the loaded segment");
    return GNSSACQ_OK;
}

}  // extern "C"
