// gnss_host.h -- host side shared by the C-ABI translation units (gnssacq.cu, gnss_xchg.cu, gnss_track.cu):
// owning types for CUDA resources, the library handle, the error macro, and the flags of the multi-GPU exchange.
// Not part of the public interface.
#pragma once
#include <memory>
#include <string>
#include <vector>

#include "../../include/gnssacq.h"
#include "gnss_internal.h"

namespace gnss {

// ---------------------------------------------------------------- owning types
// Each deleter also names the call that makes what it frees.
struct DeviceFree {
    static cudaError_t make(void** p, size_t bytes) { return cudaMalloc(p, bytes); }
    void operator()(void* p) const { cudaFree(p); }
};
struct PinnedFree {
    static cudaError_t make(void** p, size_t bytes) { return cudaMallocHost(p, bytes); }
    void operator()(void* p) const { cudaFreeHost(p); }
};
struct EventDestroy {
    static cudaError_t make(cudaEvent_t* e, unsigned flags) { return cudaEventCreateWithFlags(e, flags); }
    void operator()(cudaEvent_t e) const { cudaEventDestroy(e); }
};
struct StreamDestroy {
    static cudaError_t make(cudaStream_t* s, unsigned flags) { return cudaStreamCreateWithFlags(s, flags); }
    void operator()(cudaStream_t s) const { cudaStreamDestroy(s); }
};

template <class T> using DevPtr = std::unique_ptr<T, DeviceFree>;
template <class T> using PinnedPtr = std::unique_ptr<T, PinnedFree>;
using Event = std::unique_ptr<CUevent_st, EventDestroy>;
using Stream = std::unique_ptr<CUstream_st, StreamDestroy>;

// Buffers: the old one is freed before the new one is allocated, so growing a buffer never holds both.
template <class T, class D> cudaError_t alloc(std::unique_ptr<T, D>& p, size_t bytes) {
    p.reset();
    void* q = nullptr;
    const cudaError_t e = D::make(&q, bytes);
    if (e == cudaSuccess) p.reset(static_cast<T*>(q));
    return e;
}
// Events and streams.
template <class T, class D> cudaError_t create(std::unique_ptr<T, D>& p, unsigned flags) {
    T* q = nullptr;
    const cudaError_t e = D::make(&q, flags);
    p.reset(e == cudaSuccess ? q : nullptr);
    return e;
}

// The exchange block lives in the root's memory.  The root allocated it, another process opened it through IPC,
// and a shard of the root's own process (gnssacq_xchg_attach_local) only borrows the root's pointer.
enum class BlockOwner { borrowed, root, ipc };
struct BlockRelease {
    BlockOwner owner = BlockOwner::borrowed;
    void operator()(unsigned char* p) const {
        if (owner == BlockOwner::root) cudaFree(p);
        else if (owner == BlockOwner::ipc) cudaIpcCloseMemHandle(p);
    }
};
using XchgBlock = std::unique_ptr<unsigned char, BlockRelease>;

// ---------------------------------------------------------------- lazily built state, each set made all at once
// re-acquisition sweep (gnssacq_sweep): second staging pair, copy stream, per-buffer events, result slab
struct SweepState {
    Stream copy_stream;
    DevPtr<void> d_if2;
    PinnedPtr<void> h_if2;
    Event copied[2], consumed[2];
    DevPtr<gnssacq_result> d_res;          // [cap][P], grows
    int cap = 0;
};

// tracking correlators (gnssacq_track_load / gnssacq_correlate / gnssacq_track): C/A table, per-call channel table,
// partial sums and outputs
struct TrackState {
    DevPtr<int8_t> ca;                     // [GNSSACQ_TRACK_MAX_PRN][1023]
    DevPtr<gnssacq_channel> ch;            // [kTrackMaxChannels]
    DevPtr<double> spacing;                // [kTrackMaxTaps]
    DevPtr<double> partial;                // [channels][chunks][taps][2]
    DevPtr<double> out;                    // [channels][taps][2]
    DevPtr<double> mean;                   // [channels][2] int16 path
    DevPtr<int> status;                    // != 0: a channel of gnssacq_track ran out of samples
    PinnedPtr<double> h_out;
};

// fine-frequency stage scratch, kept between calls (re-made only when L changes)
struct FineState {
    int L = 0;
    DevPtr<void> raw;
    DevPtr<uint16_t> chip;
    DevPtr<cf> u;
    DevPtr<cf> v;                          // padded shapes: [chunk][K][L][NF] first Bluestein stage
    DevPtr<int8_t> ca;
    DevPtr<int> start;
    DevPtr<unsigned long long> best;
};

struct FftState { DevPtr<cf> in, out, v; };      // v: padded shapes, [NF] first Bluestein stage

// multi-GPU exchange (gnssacq_xchg_*): set up complete or not at all
struct Xchg {
    bool on = false, is_root = false;
    gnssacq_shard sh{};
    XchgBlock block;                       // the root's exchange block
    unsigned char* if_buf = nullptr;       // root's IF buffer
    Candidate* cand_all = nullptr;         // root's [n_prn_total][freq_num_total]
    unsigned* flags = nullptr;             // [0] IF ready, [1 + r] shard r done, [63] timeout
    DevPtr<int> d_prn_all;                 // root
    DevPtr<gnssacq_result> d_res_all;      // root
    PinnedPtr<gnssacq_result> h_res_all;   // root
    unsigned epoch = 0;
    Event ev_a, ev_b, ev_c, ev_d;
};

}  // namespace gnss

// ---------------------------------------------------------------- handle
struct gnssacq_handle {
    // streams first: destroyed after everything that may still be queued on them
    gnss::Stream own_stream;
    cudaStream_t stream = nullptr;         // own_stream or the caller's (gnssacq_set_stream)
    gnssacq_config cfg;
    const gnss::VariantOps* ops = nullptr;
    int device = 0;
    int N = 0, P = 0, B = 0, K = 0, M = 0;
    int NF = 0;                            // transform length: N for a built N, else the built length each ms is zero-padded into
    int w = 0;
    size_t if_bytes = 0;
    std::vector<int> bin_base, bin_shift;
    std::vector<double> base_freq;
    // device buffers
    gnss::DevPtr<void> d_if;
    gnss::DevPtr<int8_t> d_scode;
    gnss::DevPtr<gnss::cf> d_cc;
    gnss::DevPtr<gnss::cf> d_x;
    gnss::DevPtr<gnss::cf> d_chirp, d_chirp_filt;   // padded shapes: Bluestein tables ch [N] and H [NF] (gnss::ChirpArgs)
    gnss::DevPtr<int> d_bin_base, d_bin_shift, d_prn;
    gnss::DevPtr<double> d_base_freq;
    gnss::DevPtr<double> d_base_w;         // (IF + doppler) / Fs per base, cycles per sample (K1 v2)
    gnss::DevPtr<unsigned char> d_comb;    // [K*M ms][16][comb_pitch] re-ordered IF block (K1 v2), null: K1 v1
    int comb_pitch = 0;
    gnss::DevPtr<gnss::Candidate> d_cand;
    gnss::DevPtr<gnssacq_result> d_res;
    gnss::DevPtr<float> d_surface;
    gnss::DevPtr<gnss::cf> d_scratch;
    int xmode = 1;                 // exchange: 1 = DSMEM, 2 = L2 + persistent clusters, 3 = L2 + cooperative CTA groups
    // schedule of the current row set (use_schedule in gnssacq.cu); d_scratch, d_group_ctr, d_row_slots hold group_cap groups
    int l2x_clusters = 0;          // > 0: use the L2-exchange persistent search kernel with this many clusters
    int coop_groups = 0;           // > 0: use the cluster-free cooperative kernel with this many CTA groups
    bool by_blocks = false;        // cooperative kernel: block-granular tail (needs d_partial)
    int group_cap = 0;
    gnss::DevPtr<unsigned> d_group_ctr;
    int bin0 = 0, B_full = 0;      // this handle's bins are [bin0, bin0 + B) of the B_full-bin grid
    int row0 = 0, n_rows = 0;      // ... and of that P x B grid (row = bin * P + prn index) it searches rows [row0, row0 + n_rows),
    bool windows = false;          // ... or, with Doppler windows set, the n_rows rows listed in d_rows
    gnss::DevPtr<int> d_rows;      // [P*B] grid row ids inside the windows, bin-major (built by the first gnssacq_set_doppler_windows)
    int used_groups = 0, used_split = 1;   // schedule of the last enqueued search (gnssacq_stats)
    gnss::Xchg xc;
    const gnssacq_result* d_last_rows = nullptr;   // where the last enqueued search wrote its rows (d_res or the caller's buffer)
    gnss::DevPtr<gnss::Candidate> d_row_slots;
    gnss::DevPtr<float> d_partial;         // cooperative kernel: accumulators of row parts handed between groups
    int partial_groups = 0;                // ... for this many groups (0: not built yet)
    gnss::DevPtr<long long> d_sums;
    gnss::DevPtr<double> d_means;
    std::unique_ptr<gnss::FftState> fft;
    std::unique_ptr<gnss::FineState> fine;
    std::unique_ptr<gnss::SweepState> sweep;
    // tracking: resident recording segment (grows), the tables, records of the last gnssacq_track (grow)
    gnss::DevPtr<void> d_trk_raw;
    size_t trk_bytes = 0, trk_cap = 0;
    std::unique_ptr<gnss::TrackState> trk;
    gnss::DevPtr<gnssacq_track_record> d_trk_rec;   // [channels][periods]
    size_t trk_rec_cap = 0;
    gnss::DevPtr<double> d_trk_bank;       // gnssacq_track_bank: [I, Q][channels][periods][taps], trk_bank_cap per plane
    size_t trk_bank_cap = 0;
    // pinned host
    gnss::PinnedPtr<void> h_if;
    gnss::PinnedPtr<gnssacq_result> h_res;
    gnss::Event ev[6];
    gnss::Event ev_upload;                 // last DMA out of the pinned staging buffer h_if (stage_and_upload)
    bool have_h2d = false;
    int launches = 0;
    std::string err;
    // the members free themselves after this: on the handle's device, once its stream has drained
    ~gnssacq_handle() {
        cudaSetDevice(device);
        if (stream) cudaStreamSynchronize(stream);
    }
};

namespace gnss {

// Records `msg` as the handle's (and the thread's) last error and returns `code`.
int fail(gnssacq_handle* h, int code, const std::string& msg);
// A failed CUDA call: GNSSACQ_ERR_CUDA, or `oom_code` when the call ran out of memory.
int cuda_fail(gnssacq_handle* h, cudaError_t e, const char* call, int oom_code = GNSSACQ_ERR_CUDA);
#define CU(call, ...)                                                                                    \
    do {                                                                                                 \
        const cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) return ::gnss::cuda_fail(h, e__, #call, ##__VA_ARGS__);                  \
    } while (0)

// transform length for `n` samples per ms (n itself, or the built length it is zero-padded into), 0: unsupported
int transform_length(int n);
// GNSSACQ_OK, or the status for an invalid config with the reason in `why`
int validate(const gnssacq_config* c, std::string& why);

// C/A code (generateCAcode.m) and its sampled replica (acquisition.m:50-51)
void ca_chips(int prn, int8_t* out);
void code_replica(const gnssacq_config& c, int prn, int8_t* out);

// K1 .. K4 of one search on h->stream; xchg: the candidates go to the root's table of the exchange
int enqueue(gnssacq_handle* h, const void* d_if, gnssacq_result* d_out = nullptr, bool xchg = false);
// pageable caller memory -> d_dst through the handle's pinned staging buffer
int stage_and_upload(gnssacq_handle* h, void* d_dst, const void* host_src, cudaStream_t s);
// the fields of gnssacq_stats that describe the engine
void fill_engine_stats(const gnssacq_handle* h, gnssacq_stats* st);

// K4: acquisition.m:62-70 from the per-row candidates
__global__ void finalize_kernel(const Candidate* __restrict__ cand, int P, int B, int N, int w, double fmin,
                                double fstep, double thr, const int* __restrict__ prn_ids,
                                gnssacq_result* __restrict__ out, int cand_stride, int bin0);

// non-root shard of the exchange, after K2: raises its "done" flag in the root's block
__global__ void xchg_done_kernel(unsigned* flag, unsigned epoch);

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

}  // namespace gnss
