// The frame of one training epoch, shared by every model and by DSGD: each path supplies only the work of one attempt.
#pragma once
#include "lrk_common.cuh"
#include "sgd.cuh"
#include "topn_tc.cuh"
#include <cmath>
#include <functional>
#include <vector>

// A float array under the rollback safeguard: copied to *bk before the epoch, copied back after a rejected attempt
struct LrkSaved { float* live; LrkBuf<float>* bk; size_t n; };

struct LrkEpoch {
    std::function<int(int attempt)> enqueue;   // the attempt's work on h->stream, between the timing events ev0 and ev1
    bool refresh_norm = false;                 // refresh mean |p_u|^2 after ev1 (the stream SGD kernels read it)
    std::function<int()> after_sync;           // optional: a check once the attempt has completed
    // Safeguard (lrk_model_info().safeguard): the arrays to snapshot.  Called again for the restore, after the attempt, so
    // that `live` can name the buffer that holds the data then (the DSGD ring buffers swap during an attempt).
    std::function<std::vector<LrkSaved>()> saved;
    std::function<int()> rolled_back;          // optional: the path's bookkeeping after a restore
};

// Runs one epoch: zero the loss accumulator, record ev0, enqueue, record ev1, read the loss back, synchronise, take the
// epoch time, scale the loss, fail on a NaN or Inf loss, then mark the fp32 copies as ahead of the fp64 masters and
// the top-N cache as stale.  Models without a loss (loss_scale 0) skip the accumulator and report 0.
// Safeguard: an attempt whose loss is non-finite or more than 10x the last accepted epoch's is rolled back and re-run with
// 4x fewer samples in flight (h->conc_div), at most 6 times and up to conc_div 4096; conc_div halves again after 8 good epochs.
static int lrk_epoch(lrk_handle_s* h, const LrkEpoch& e, double* loss_out) {
    const LrkModelInfo m = lrk_model_info(h->cfg);
    cudaStream_t st = h->stream;
    int rc;
    if (m.safeguard) {
        const std::vector<LrkSaved> saved = e.saved();
        for (const LrkSaved& a : saved) if ((rc = lrk_dev_alloc(h, a.bk, a.n))) return rc;
        for (const LrkSaved& a : saved) LRK_CUDA(h, cudaMemcpyAsync(*a.bk, a.live, sizeof(float) * a.n, cudaMemcpyDeviceToDevice, st));
    }
    const bool has_loss = m.loss_scale != 0.0;
    double loss = 0.0;
    for (int attempt = 0;; ++attempt) {
        if (has_loss) LRK_CUDA(h, cudaMemsetAsync(h->d_loss, 0, sizeof(double), st));
        LRK_CUDA(h, cudaEventRecord(h->ev0, st));
        if ((rc = e.enqueue(attempt))) return rc;
        LRK_CUDA(h, cudaEventRecord(h->ev1, st));
        if (e.refresh_norm && (rc = refresh_user_norm2(h, false))) return rc;
        if (has_loss) LRK_CUDA(h, cudaMemcpyAsync(h->h_loss, h->d_loss, sizeof(double), cudaMemcpyDeviceToHost, st));
        LRK_CUDA(h, cudaStreamSynchronize(st));
        if (e.after_sync && (rc = e.after_sync())) return rc;
        LRK_CUDA(h, cudaEventElapsedTime(&h->last_epoch_ms, h->ev0, h->ev1));
        loss = has_loss ? m.loss_scale * h->h_loss[0] : 0.0;
        const bool bad = !std::isfinite(loss) || (h->prev_loss > 0.0 && loss > 10.0 * h->prev_loss);
        if (!m.safeguard || !bad || attempt >= 6 || h->conc_div >= 4096) break;
        for (const LrkSaved& a : e.saved()) LRK_CUDA(h, cudaMemcpyAsync(a.live, *a.bk, sizeof(float) * a.n, cudaMemcpyDeviceToDevice, st));
        h->conc_div *= 4; h->good_epochs = 0; h->rollbacks++;
        if (e.rolled_back && (rc = e.rolled_back())) return rc;
    }
    if (!m.f64_working) h->f64_valid = false;
    topn_tc_invalidate(h);
    if (loss_out) *loss_out = loss;
    if (!std::isfinite(loss))
        return lrk_fail(h, LRK_ERR_DIVERGED, "lrk_sgd_epoch", "Loss = NaN or Infinity: current settings does not fit the recommender!", __FILE__, __LINE__);
    h->prev_loss = loss;
    h->epochs_done++;
    if (h->conc_div > 1 && ++h->good_epochs >= 8) { h->conc_div /= 2; h->good_epochs = 0; }
    return LRK_OK;
}
