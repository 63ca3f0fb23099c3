// gnss_xchg.cu -- multi-GPU search through peer memory (include/gnssacq.h: gnssacq_shard_plan*, gnssacq_xchg_*).
//
// The root shard owns one exchange block in its HBM: its IF buffer, the candidate table of the full PRN x bin grid
// and the flag words.  Every other shard pulls the IF block out of it (comb_kernel), writes its candidates straight
// into the table and raises its "done" flag; the root waits for those flags and runs K4 over the whole table.
#include <cstring>
#include <string>

#include "gnss_host.h"

using namespace gnss;

namespace gnss {

// non-root shard, after K2: its candidates are in the root's table (stores issued by the preceding kernel)
__global__ void xchg_done_kernel(unsigned* flag, unsigned epoch) {
    __threadfence_system();
    flag_store_sys(flag, epoch);
}

}  // namespace gnss

namespace {

// root, before K4: every other shard has delivered this step's candidates
__global__ void xchg_wait_kernel(const unsigned* done_flags, int world, unsigned long long has_rows, unsigned epoch, unsigned* timeout) {
    const int r = 1 + (int)threadIdx.x;
    if (r >= world) return;
    // with fewer PRNs (or rows) than shards a shard may end up with nothing to search: it never reports
    if ((has_rows >> r) & 1ull) flag_wait_sys(done_flags + r, epoch, timeout);
}

// rows [first, first + count) of shard `rank` under the row-granular plan: the root's share is (1000 + extra) / 1000
// of the others'; what is left goes to the others in equal parts, the first few taking one row more
void plan_rows_range(long long total, int rank, int world, int extra_permille, long long& first, long long& count) {
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

size_t xchg_if_span(const gnssacq_handle* h) { return (h->if_bytes + 255) / 256 * 256; }
size_t xchg_cand_span(const gnssacq_shard* sh) {
    return ((size_t)sh->n_prn_total * sh->freq_num_total * sizeof(Candidate) + 255) / 256 * 256;
}

// Checks that `sh` describes the handle and that it is the root's shard (`root`) or another's, then starts the
// exchange state in `x`.  Nothing on the handle changes until xchg_publish.
int xchg_begin(gnssacq_handle* h, const gnssacq_shard* sh, bool root, Xchg& x) {
    if (!h || !sh) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    if (h->xc.on) return fail(h, GNSSACQ_ERR_STATE, "exchange already set up on this handle");
    if (h->windows) return fail(h, GNSSACQ_ERR_STATE, "Doppler windows are set on this handle (clear them first)");
    if (h->NF != h->N) return fail(h, GNSSACQ_ERR_STATE, "the multi-GPU exchange needs a built samples_per_ms (this handle zero-pads each ms)");
    if (sh->prn_count != h->P || sh->bin_count != h->B || sh->bin_first != h->bin0 || sh->freq_num_total != h->B_full ||
        (sh->plan_rows ? (sh->row_first != h->row0 || sh->row_count != h->n_rows) : (h->n_rows != h->P * h->B)))
        return fail(h, GNSSACQ_ERR_INVALID_ARG, "shard does not describe this handle (use gnssacq_shard_plan's config)");
    if (!h->d_comb) return fail(h, GNSSACQ_ERR_STATE, "the multi-GPU exchange needs the comb-row K1");
    if (root && sh->rank != 0) return fail(h, GNSSACQ_ERR_INVALID_ARG, "the root is shard 0");
    if (!root && sh->rank == 0) return fail(h, GNSSACQ_ERR_INVALID_ARG, "shard 0 is the root (gnssacq_xchg_root)");
    CU(cudaSetDevice(h->device));
    x.sh = *sh;
    x.is_root = root;
    for (Event* e : {&x.ev_a, &x.ev_b, &x.ev_c, &x.ev_d}) CU(create(*e, cudaEventDefault));
    return GNSSACQ_OK;
}

// Lays the exchange out over `block` and hands the complete state to the handle.
void xchg_publish(gnssacq_handle* h, Xchg& x, XchgBlock block) {
    x.if_buf = block.get();
    x.cand_all = reinterpret_cast<Candidate*>(block.get() + xchg_if_span(h));
    x.flags = reinterpret_cast<unsigned*>(block.get() + xchg_if_span(h) + xchg_cand_span(&x.sh));
    x.block = std::move(block);
    x.on = true;
    h->xc = std::move(x);
}

}  // namespace

extern "C" {

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

int gnssacq_xchg_root(gnssacq_handle* h, const gnssacq_shard* sh, void* ipc_out) {
    Xchg x;
    if (int rc = xchg_begin(h, sh, true, x)) return rc;
    const size_t bytes = xchg_if_span(h) + xchg_cand_span(sh) + 64 * sizeof(unsigned);
    void* p = nullptr;
    CU(cudaMalloc(&p, bytes));
    XchgBlock block(static_cast<unsigned char*>(p), BlockRelease{BlockOwner::root});
    CU(cudaMemsetAsync(block.get(), 0, bytes, h->stream));           // the flag words start at 0
    CU(alloc(x.d_prn_all, sh->n_prn_total * sizeof(int)));
    CU(cudaMemcpyAsync(x.d_prn_all.get(), sh->prn_total, sh->n_prn_total * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CU(alloc(x.d_res_all, sh->n_prn_total * sizeof(gnssacq_result)));
    CU(alloc(x.h_res_all, sh->n_prn_total * sizeof(gnssacq_result)));
    if (ipc_out) {
        static_assert(sizeof(cudaIpcMemHandle_t) <= GNSSACQ_IPC_BYTES, "IPC handle size");
        cudaIpcMemHandle_t ih;
        CU(cudaIpcGetMemHandle(&ih, block.get()));
        std::memset(ipc_out, 0, GNSSACQ_IPC_BYTES);
        std::memcpy(ipc_out, &ih, sizeof ih);
    }
    // the other shards use the block from their own streams (and `sh` is the caller's): the copies must be done
    CU(cudaStreamSynchronize(h->stream));
    xchg_publish(h, x, std::move(block));
    return GNSSACQ_OK;
}

int gnssacq_xchg_attach(gnssacq_handle* h, const gnssacq_shard* sh, const void* root_ipc) {
    if (!root_ipc) return fail(h, GNSSACQ_ERR_INVALID_ARG, "NULL argument");
    Xchg x;
    if (int rc = xchg_begin(h, sh, false, x)) return rc;
    cudaIpcMemHandle_t ih;
    std::memcpy(&ih, root_ipc, sizeof ih);
    void* p = nullptr;
    CU(cudaIpcOpenMemHandle(&p, ih, cudaIpcMemLazyEnablePeerAccess));      // the root's block, reachable over NVLink
    xchg_publish(h, x, XchgBlock(static_cast<unsigned char*>(p), BlockRelease{BlockOwner::ipc}));
    return GNSSACQ_OK;
}

int gnssacq_xchg_attach_local(gnssacq_handle* h, const gnssacq_shard* sh, gnssacq_handle* root) {
    if (!root || !root->xc.on || !root->xc.is_root) return fail(h, GNSSACQ_ERR_INVALID_ARG, "root has no exchange block");
    Xchg x;
    if (int rc = xchg_begin(h, sh, false, x)) return rc;
    if (h->device != root->device) {
        int can = 0;
        CU(cudaDeviceCanAccessPeer(&can, h->device, root->device));
        if (!can) return fail(h, GNSSACQ_ERR_CUDA, "no peer access to the root's GPU");
        const cudaError_t e = cudaDeviceEnablePeerAccess(root->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CU(e);
        cudaGetLastError();
    }
    xchg_publish(h, x, XchgBlock(root->xc.block.get(), BlockRelease{BlockOwner::borrowed}));
    return GNSSACQ_OK;
}

void* gnssacq_xchg_if_buffer(gnssacq_handle* h) { return (h && h->xc.on && h->xc.is_root) ? h->xc.if_buf : nullptr; }

int gnssacq_xchg_enqueue(gnssacq_handle* h, const void* host_if, size_t nbytes) {
    if (!h || !h->xc.on) return fail(h, GNSSACQ_ERR_STATE, "no exchange set up on this handle");
    if (host_if && !h->xc.is_root) return fail(h, GNSSACQ_ERR_INVALID_ARG, "only the root takes the IF block");
    if (host_if && nbytes < h->if_bytes) return fail(h, GNSSACQ_ERR_SHORT_BUFFER, "IF block shorter than noncoh_blocks*coh_ms ms");
    CU(cudaSetDevice(h->device));
    ++h->xc.epoch;
    CU(cudaEventRecord(h->ev[0].get(), h->stream));
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
    CU(cudaEventRecord(xc.ev_c.get(), s));
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
    CU(cudaEventRecord(xc.ev_d.get(), s));
    finalize_kernel<<<(xc.sh.n_prn_total + 63) / 64, 64, 0, s>>>(xc.cand_all, xc.sh.n_prn_total, xc.sh.freq_num_total, h->N, h->w,
                                                               h->cfg.freq_min_hz, h->cfg.freq_step_hz, h->cfg.snr_threshold_db,
                                                               xc.d_prn_all.get(), xc.d_res_all.get(), xc.sh.freq_num_total, 0);
    CU(cudaGetLastError());
    h->launches += 1;
    CU(cudaEventRecord(h->ev[4].get(), s));
    return GNSSACQ_OK;
}

int gnssacq_xchg_fetch(gnssacq_handle* h, gnssacq_result* out, gnssacq_stats* st) {
    if (!h || !h->xc.on) return fail(h, GNSSACQ_ERR_STATE, "no exchange set up on this handle");
    if (out && !h->xc.is_root) return fail(h, GNSSACQ_ERR_INVALID_ARG, "rows are on the root");
    CU(cudaSetDevice(h->device));
    auto& xc = h->xc;
    const int n = xc.sh.n_prn_total;
    unsigned timed_out = 0;
    if (xc.is_root && out) CU(cudaMemcpyAsync(xc.h_res_all.get(), xc.d_res_all.get(), n * sizeof(gnssacq_result), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaEventRecord(h->ev[5].get(), h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (xc.is_root) {
        CU(cudaMemcpy(&timed_out, xc.flags + 63, sizeof timed_out, cudaMemcpyDeviceToHost));
        if (timed_out) return fail(h, GNSSACQ_ERR_STATE, "a shard of the exchange did not answer within the time-out");
        if (out) std::memcpy(out, xc.h_res_all.get(), n * sizeof(gnssacq_result));
    }
    if (st) {
        std::memset(st, 0, sizeof(*st));
        if (h->have_h2d) cudaEventElapsedTime(&st->h2d_ms, h->ev[0].get(), h->ev[1].get());
        cudaEventElapsedTime(&st->wipeoff_fft_ms, h->ev[1].get(), h->ev[2].get());
        cudaEventElapsedTime(&st->search_ms, h->ev[2].get(), h->ev[3].get());
        if (xc.is_root) {
            // (before gnssacq_xchg_finish these events are unrecorded: the queries fail and leave zeros)
            if (cudaEventElapsedTime(&st->gather_wait_ms, xc.ev_c.get(), xc.ev_d.get()) != cudaSuccess) st->gather_wait_ms = 0.f;
            if (cudaEventElapsedTime(&st->finalize_ms, xc.ev_d.get(), h->ev[4].get()) != cudaSuccess) st->finalize_ms = 0.f;
            cudaEventElapsedTime(&st->d2h_ms, h->ev[4].get(), h->ev[5].get());
        } else {
            cudaEventElapsedTime(&st->if_pull_ms, xc.ev_a.get(), xc.ev_b.get());
        }
        cudaEventElapsedTime(&st->total_ms, h->ev[0].get(), h->ev[5].get());
        cudaGetLastError();                    // a failed timing query must not surface at somebody's next launch check
        st->kernel_launches = h->launches;
        fill_engine_stats(h, st);
    }
    return GNSSACQ_OK;
}

}  // extern "C"
