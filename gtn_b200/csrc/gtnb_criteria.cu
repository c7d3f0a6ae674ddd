/*
 * gtnb_criteria.cu -- whole-minibatch criteria: what the reference does with
 * parallelMap(fwd) + parallelMap(bwd) (benchmarks/ctc.cpp:150-165) as ONE call
 * that only enqueues device work: no per-utterance host objects, one pinned
 * staging upload, one small read-back.
 */
#include <algorithm>
#include <cstdlib>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "gtnb_internal.h"

using namespace gtnb;

/*
 * One attempt.  allow_implicit: sweep the frames without building the lattice (k_implicit.cu)
 * when the target graphs qualify; *needs_exact is set when that sweep met a non-finite weight,
 * in which case the outputs are not to be used and the caller repeats the call materialised.
 */
namespace {
/* GTNB_TIMES=1: wall-clock microseconds between the host-side phases of one gtnb_ctc_loss call (stderr) */
struct PhaseClock {
  bool on;
  std::chrono::steady_clock::time_point t;
  std::string line;
  PhaseClock() : on(std::getenv("GTNB_TIMES") != nullptr), t(std::chrono::steady_clock::now()) {}
  void mark(const char* what) {
    if (!on) return;
    const auto n = std::chrono::steady_clock::now();
    line += std::string(what) + " " + std::to_string(std::chrono::duration_cast<std::chrono::nanoseconds>(n - t).count() / 1000.0) + "  ";
    t = n;
  }
  ~PhaseClock() {
    if (on) std::fprintf(stderr, "[gtnb_ctc_loss us] %s\n", line.c_str());
  }
};
} // namespace

static int ctc_loss_run(
    gtnb_ctx* ctx, int B, int T, int C, const float* emissions, int emissions_on_device,
    const int32_t* input_lens, const int32_t* targets, const int32_t* target_lens, int blank,
    float* losses_host, float* grads, int grads_on_device, bool allow_implicit, bool* needs_exact) {
  *needs_exact = false;
  if (!ctx || B < 0 || T < 0 || C <= 0 || !emissions || !target_lens || !losses_host)
    return fail(ctx, GTNB_ERR_INVALID_ARGUMENT, "gtnb_ctc_loss: bad arguments");
  if (B == 0) return GTNB_OK;
  GTNB_CUDA(ctx, cudaSetDevice(ctx->device));
  PhaseClock pc;
  bool direct = false; // the PAIR / QUAD kernels of k_bidir.cu on mapped pinned memory (see below)
  const GraphMeta* meta_mapped = nullptr;
  const int32_t* small_mapped = nullptr;
  const long long per = (long long)T * C;
  int rc = GTNB_OK;
  float* e_dev = nullptr;
  float* g_dev = nullptr;
  float* z_dev = nullptr;
  float* deltas_dev = nullptr;
  int32_t* small_dev = nullptr; // [targets | offsets | lens | T]
  int32_t* status_dev = nullptr;
  float* row_scratch = nullptr; // k_linear.cu's per-frame scores, allocated once for all sub-batches
  float* zparts_dev = nullptr; // k_bidir.cu: forwardScore(emissions) as two partial sums per utterance
  float* boff_dev = nullptr; // k_bidir.cu: per-block score offsets of the two CTAs of every utterance
  float* bidir_scores_dev = nullptr; // k_bidir.cu: the lattices' scores, inside the read-back block
  bool implicit = false;
  bool bidir = false;
  int zp = 1;
  int K = 1; // sub-batches (implicit path with host buffers)
  std::vector<int> chunk_lo;
  cudaStream_t main_stream = ctx->stream;
  gtnb_lattice* lat = nullptr;
  cudaEvent_t h2d_event = nullptr;
  std::vector<long long> sgn, sga;

  // host: only sizes.  Graph b has 2U+1 nodes; arcs = self loops + step arcs + skip arcs
  // (benchmarks/ctc.cpp:40-58), skip arcs exist where consecutive labels differ.
  std::vector<SgDims> dims(B);
  std::vector<int32_t> Tb(B), off(B);
  long long tot_t = 0;
  for (int b = 0; b < B; b++) {
    const int U = target_lens[b];
    if (U < 0) return fail(ctx, GTNB_ERR_INVALID_ARGUMENT, "gtnb_ctc_loss: negative target length");
    if (U > 0 && !targets) return fail(ctx, GTNB_ERR_INVALID_ARGUMENT, "gtnb_ctc_loss: targets is NULL");
    off[b] = (int32_t)tot_t;
    const int32_t* tg = targets + tot_t;
    int skips = 0;
    int all_valid = blank >= 0 && blank < C;
    if (U > 0) all_valid &= (unsigned)tg[0] < (unsigned)C;
    for (int u = 1; u < U; u++) { // one pass: skip arcs exist where consecutive labels differ; labels in [0, C)
      skips += tg[u] != tg[u - 1];
      all_valid &= (unsigned)tg[u] < (unsigned)C;
    }
    const int L = 2 * U + 1;
    dims[b] = SgDims{L, L + (L - 1) + skips, L >= 2 ? 2 : 1, all_valid, /*uniform=*/1, /*max_in=*/3, /*max_out=*/3};
    tot_t += U;
    Tb[b] = input_lens ? input_lens[b] : T;
    if (Tb[b] < 0 || Tb[b] > T)
      return fail(ctx, GTNB_ERR_INVALID_ARGUMENT, "gtnb_ctc_loss: input_lens out of range");
  }
  int maxT = 0;
  for (int b = 0; b < B; b++) maxT = std::max(maxT, Tb[b]);
  pc.mark("sizes");

#define TRY(x)                 \
  do {                         \
    if ((rc = (x))) goto done; \
  } while (0)
#define TRYCUDA(call)                                      \
  do {                                                     \
    cudaError_t e__ = (call);                              \
    if (e__ != cudaSuccess) {                              \
      rc = cuda_fail(ctx, e__, #call, __FILE__, __LINE__); \
      goto done;                                           \
    }                                                      \
  } while (0)

  implicit = allow_implicit && implicit_dims_supported(dims.data(), B);
  // Host buffers: cut the batch into K sub-batches whose H2D copy, kernels and D2H copy run on
  // their own streams, so that the two PCIe directions and the (latency-bound) sweeps overlap.
  // Device buffers: K = 1, and the normaliser (k_linear.cu) runs beside the forward sweep.
  if (implicit && (!emissions_on_device || (grads && !grads_on_device))) {
    const long long bytes = (long long)sizeof(float) * per * B;
    K = (int)std::min<long long>(std::max<long long>(bytes / (4ll << 20), 1), 16);
    K = std::min(K, B);
  }
  TRY(ensure_side_streams(ctx, K, K + 2));
  chunk_lo.resize(K + 1);
  for (int k = 0; k <= K; k++) chunk_lo[k] = (int)((long long)B * k / K);
  if (emissions_on_device) {
    e_dev = const_cast<float*>(emissions);
  } else {
    // the copy runs on a second stream while this one builds the target graphs and the
    // lattice structure (k_ctc.cu, compose alive / count / scan need no emissions)
    TRY(dev_alloc(ctx, &e_dev, per * B));
  }
  if (grads) {
    if (grads_on_device)
      g_dev = grads;
    else
      TRY(dev_alloc(ctx, &g_dev, per * B));
    // with full-length utterances the normaliser's gradient overwrites every element
    if (input_lens) TRYCUDA(cudaMemsetAsync(g_dev, 0, sizeof(float) * per * B, ctx->stream));
  }
  TRY(dev_alloc(ctx, &z_dev, B));
  TRY(dev_alloc(ctx, &deltas_dev, B));
  TRY(dev_alloc(ctx, &small_dev, tot_t + 3ll * B));
  TRY(composed_alloc(ctx, B, dims.data(), B, 0, Tb.data(), C, e_dev, per, sgn, sga, &lat, implicit));
  pc.mark("alloc+meta");
  // the whole criterion in one launch per sub-batch (k_bidir.cu) when the batch qualifies
  bidir = implicit && ctx->use_bidir && ctx->use_banded == 0 && bidir_supported(lat, e_dev, per, g_dev, per);
  // PAIR / QUAD kernels (graphs from the targets, one launch): everything small goes through MAPPED pinned memory --
  // the kernel reads the descriptors and targets in place and writes its results straight into the read-back
  // block; no upload, no memset, no download on the path (23 of the step's 47 us of host work were those enqueues)
  direct = implicit && ctx->use_bidir && ctx->use_banded == 0 && ctx->bidir_mode != 0 &&
           bidir_supported(lat, e_dev, per, g_dev, per) && bidir_takes_targets(lat, 1, blank);
  if (bidir && direct) {
    const long long zpb = 2ll * B * bidir_zparts();
    TRY(readback_reserve(ctx, (zpb + 2ll * B) * sizeof(float)));
    zparts_dev = reinterpret_cast<float*>(ctx->readback);
    bidir_scores_dev = zparts_dev + zpb;
    status_dev = reinterpret_cast<int32_t*>(zparts_dev + zpb + B);
    std::memset(status_dev, 0, sizeof(int32_t) * B);
    TRY(dev_alloc(ctx, &boff_dev, 8ll * B * bidir_blocks(maxT)));
  } else if (bidir) {
    // one block for everything that is read back: [partial sums of forwardScore(e) | lattice scores | status]
    const long long zpb = 2ll * B * bidir_zparts();
    TRY(dev_alloc(ctx, &zparts_dev, zpb + 2ll * B));
    bidir_scores_dev = zparts_dev + zpb;
    status_dev = reinterpret_cast<int32_t*>(zparts_dev + zpb + B);
    TRY(dev_alloc(ctx, &boff_dev, 8ll * B * bidir_blocks(maxT)));
    TRYCUDA(cudaMemsetAsync(status_dev, 0, sizeof(int32_t) * B, ctx->stream));
  } else if (implicit) {
    TRY(dev_alloc(ctx, &row_scratch, (long long)B * std::max(maxT, 1)));
    TRY(dev_alloc(ctx, &status_dev, B));
    TRYCUDA(cudaMemsetAsync(status_dev, 0, sizeof(int32_t) * B, ctx->stream));
  }

  // one pinned staging pass for everything the kernels need from the host
  TRY(stage_begin(ctx));
  {
    // [targets | offsets | lens | T] in ONE copy (each small copy costs microseconds of stream latency)
    std::vector<int32_t> small_h;
    if (!(bidir && direct)) {
      small_h.resize((size_t)(tot_t + 3ll * B));
      if (tot_t) std::memcpy(small_h.data(), targets, sizeof(int32_t) * tot_t);
      std::memcpy(small_h.data() + tot_t, off.data(), sizeof(int32_t) * B);
      std::memcpy(small_h.data() + tot_t + B, target_lens, sizeof(int32_t) * B);
      std::memcpy(small_h.data() + tot_t + 2ll * B, Tb.data(), sizeof(int32_t) * B);
    }
    if (bidir && direct) {
      // the kernel needs the descriptors (with the target offsets) and the labels, nothing else
      void *m = nullptr, *t = nullptr;
      for (int b = 0; b < B; b++) lat->meta_h[b].tgt_off = off[b];
      TRY(stage_reserve(ctx, sizeof(GraphMeta) * B + sizeof(int32_t) * (size_t)tot_t + 1024));
      TRY(stage_place(ctx, lat->meta_h.data(), sizeof(GraphMeta) * B, &m));
      TRY(stage_place(ctx, targets, sizeof(int32_t) * (size_t)tot_t, &t));
      meta_mapped = static_cast<const GraphMeta*>(m);
      small_mapped = static_cast<const int32_t*>(t);
    } else {
      TRY(stage_upload(ctx, lat->meta, lat->meta_h.data(), sizeof(GraphMeta) * B));
      TRY(stage_upload(ctx, small_dev, small_h.data(), sizeof(int32_t) * small_h.size()));
    }
  }
  if (!bidir) {
    std::vector<float> minus1(B, -1.0f); // subtract's gradFunc, functions.cpp:53-58
    TRY(stage_upload(ctx, deltas_dev, minus1.data(), sizeof(float) * B));
  }
  if (!(bidir && direct)) TRY(stage_end(ctx)); // (direct: no copy was issued from the staging buffer; the call synchronises before it returns)
  pc.mark("staging");
  if (!emissions_on_device) {
    // enqueued AFTER the small staged upload: the copy engine serves one direction in
    // submission order, and the graphs must not queue behind 65 MB of emissions
    TRYCUDA(cudaEventRecord(ctx->ev_fork, ctx->stream)); // orders the copy after the allocation
    TRYCUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_fork, 0));
    for (int k = 0; k < K; k++) {
      const long long lo = (long long)chunk_lo[k] * per, n = (long long)(chunk_lo[k + 1] - chunk_lo[k]) * per;
      TRYCUDA(cudaMemcpyAsync(e_dev + lo, emissions + lo, sizeof(float) * n, cudaMemcpyHostToDevice,
                              ctx->copy_stream));
      TRYCUDA(cudaEventRecord(ctx->side_events[k], ctx->copy_stream));
    }
    TRYCUDA(cudaEventRecord(ctx->ev_join, ctx->copy_stream));
    h2d_event = ctx->ev_join;
  }

  // ctcGraph -> intersect(ctc, emissions) -> forwardScore -> backward(-1) -> compose gradFunc
  // (k_bidir.cu's PAIR / QUAD kernels take the CTC target graphs from the targets themselves: no tables to build)
  if (!(bidir && direct))
    TRY(launch_ctc_build(ctx, lat, small_dev, small_dev + tot_t, small_dev + tot_t + B, blank));
  if (implicit) {
    // the sweeps: k_implicit.cu, or (experimental flag) the temporally blocked ones of k_banded.cu
    const bool banded = ctx->use_banded != 0 && banded_supported(ctx, lat);
    auto sweep_forward = [&](int b0, int nb) {
      return banded ? launch_banded_forward(ctx, lat, status_dev, b0, nb)
                    : launch_implicit_forward(ctx, lat, status_dev, b0, nb);
    };
    auto sweep_backward = [&](int b0, int nb) {
      return banded ? launch_banded_backward(ctx, lat, deltas_dev, g_dev, per, b0, nb)
                    : launch_implicit_backward(ctx, lat, deltas_dev, g_dev, per, b0, nb);
    };
    // everything below only needs what is already enqueued on the main stream (graphs, staging,
    // the memset of the gradients) plus its own slice of the emissions
    cudaEvent_t ev_setup = ctx->side_events[K], ev_lin = ctx->side_events[K + 1];
    const int32_t* T_dev = small_dev + tot_t + 2ll * B;
    TRYCUDA(cudaEventRecord(ev_setup, main_stream));
    if (bidir && K == 1 && !h2d_event && !(grads && !grads_on_device)) {
      TRY(launch_bidir_ctc(ctx, lat, status_dev, zparts_dev, boff_dev, g_dev, per, 0, -1, /*zero_w=*/1, bidir_scores_dev, blank, direct ? small_mapped : small_dev,
                               (direct ? small_mapped : small_dev) + tot_t, direct ? meta_mapped : nullptr));
    } else if (bidir) {
      for (int k = 0; k < K && !rc; k++) {
        const int b0 = chunk_lo[k], nb = chunk_lo[k + 1] - chunk_lo[k];
        cudaStream_t cs = ctx->side_streams[k];
        TRYCUDA(cudaStreamWaitEvent(cs, ev_setup, 0));
        if (h2d_event) TRYCUDA(cudaStreamWaitEvent(cs, ctx->side_events[k], 0));
        ctx->stream = cs;
        rc = launch_bidir_ctc(ctx, lat, status_dev, zparts_dev, boff_dev, g_dev, per, b0, nb, /*zero_w=*/1, bidir_scores_dev, blank, direct ? small_mapped : small_dev,
                               (direct ? small_mapped : small_dev) + tot_t, direct ? meta_mapped : nullptr);
        ctx->stream = main_stream;
        if (rc) goto done;
        if (grads && !grads_on_device)
          TRYCUDA(cudaMemcpyAsync(grads + (long long)b0 * per, g_dev + (long long)b0 * per,
                                  sizeof(float) * per * nb, cudaMemcpyDeviceToHost, cs));
        TRYCUDA(cudaEventRecord(ctx->side_events[k], cs));
        TRYCUDA(cudaStreamWaitEvent(main_stream, ctx->side_events[k], 0));
      }
    } else if (K == 1 && !h2d_event && !(grads && !grads_on_device)) {
      // forwardScore(emissions) and its +1 gradient beside the forward sweep
      TRYCUDA(cudaStreamWaitEvent(ctx->copy_stream, ev_setup, 0));
      ctx->stream = ctx->copy_stream;
      rc = launch_linear_forward(ctx, B, T_dev, maxT, C, e_dev, per, 0, z_dev, g_dev, per, nullptr, 1.0f,
                                 input_lens ? 0 : 1, row_scratch);
      ctx->stream = main_stream;
      if (rc) goto done;
      TRYCUDA(cudaEventRecord(ev_lin, ctx->copy_stream));
      TRY(sweep_forward(0, -1));
      TRYCUDA(cudaStreamWaitEvent(main_stream, ev_lin, 0));
      if (grads) TRY(sweep_backward(0, -1));
    } else {
      for (int k = 0; k < K && !rc; k++) {
        const int b0 = chunk_lo[k], nb = chunk_lo[k + 1] - chunk_lo[k];
        cudaStream_t cs = ctx->side_streams[k];
        TRYCUDA(cudaStreamWaitEvent(cs, ev_setup, 0));
        if (h2d_event) TRYCUDA(cudaStreamWaitEvent(cs, ctx->side_events[k], 0));
        ctx->stream = cs;
        rc = launch_linear_forward(ctx, nb, T_dev + b0, maxT, C, e_dev + (long long)b0 * per, per, 0,
                                   z_dev + b0, g_dev ? g_dev + (long long)b0 * per : nullptr, per, nullptr,
                                   1.0f, input_lens ? 0 : 1, row_scratch + (long long)b0 * std::max(maxT, 1));
        if (!rc) rc = sweep_forward(b0, nb);
        if (!rc && grads) rc = sweep_backward(b0, nb);
        ctx->stream = main_stream;
        if (rc) goto done;
        if (grads && !grads_on_device)
          TRYCUDA(cudaMemcpyAsync(grads + (long long)b0 * per, g_dev + (long long)b0 * per,
                                  sizeof(float) * per * nb, cudaMemcpyDeviceToHost, cs));
        TRYCUDA(cudaEventRecord(ctx->side_events[k], cs));
        TRYCUDA(cudaStreamWaitEvent(main_stream, ctx->side_events[k], 0));
      }
    }
  } else {
    TRY(launch_compose(ctx, lat, h2d_event));
    // forwardScore(emissions) and its +1 gradient
    TRY(launch_linear_forward(ctx, B, small_dev + tot_t + 2ll * B, maxT, C, e_dev, per, 0, z_dev, g_dev,
                              per, nullptr, 1.0f, input_lens ? 0 : 1));
    TRY(launch_forward(ctx, lat, MODE_LOG));
    lat->forward_done = true;
    lat->forward_mode = MODE_LOG;
  }
  if (grads && !implicit) {
    // shortestDistanceGrad and compose's gradFunc fused when the lattice qualifies
    rc = launch_backward_fused(ctx, lat, deltas_dev, g_dev, per);
    if (rc == GTNB_ERR_UNSUPPORTED) {
      if (!lat->arc_grad) TRY(dev_alloc(ctx, &lat->arc_grad, lat->tot_A));
      TRY(launch_backward(ctx, lat, 0, deltas_dev));
      TRY(launch_compose_grad(ctx, lat, nullptr, g_dev, per));
    } else if (rc) {
      goto done;
    }
    if (!grads_on_device)
      TRYCUDA(cudaMemcpyAsync(grads, g_dev, sizeof(float) * per * B, cudaMemcpyDeviceToHost, ctx->stream));
  }
  pc.mark("launches");
  zp = bidir ? 2 * bidir_zparts() : 1; // partial sums of forwardScore(emissions) per utterance
  TRY(readback_reserve(ctx, (zp + 2) * sizeof(float) * B));
  {
    float* z = reinterpret_cast<float*>(ctx->readback);
    float* s = z + (long long)zp * B;
    int32_t* st = reinterpret_cast<int32_t*>(s + B);
    if (bidir && direct) {
      // the kernel wrote straight into this block
    } else if (bidir) { // one copy: the block is laid out like the host buffer
      TRYCUDA(cudaMemcpyAsync(z, zparts_dev, sizeof(float) * (zp + 2) * B, cudaMemcpyDeviceToHost, ctx->stream));
    } else {
      TRYCUDA(cudaMemcpyAsync(z, z_dev, sizeof(float) * B, cudaMemcpyDeviceToHost, ctx->stream));
      TRYCUDA(cudaMemcpyAsync(s, lat->out_scores, sizeof(float) * B, cudaMemcpyDeviceToHost, ctx->stream));
      if (implicit)
        TRYCUDA(cudaMemcpyAsync(st, status_dev, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, ctx->stream));
    }
    pc.mark("readback enqueue");
    TRYCUDA(cudaStreamSynchronize(ctx->stream));
    pc.mark("sync");
    for (int b = 0; b < B; b++) { // subtract, functions.cpp:52
      float zb = 0.0f;
      for (int k = 0; k < zp; k++) zb += z[(long long)zp * b + k];
      losses_host[b] = zb - s[b];
    }
    if (implicit)
      for (int b = 0; b < B; b++)
        if (st[b]) *needs_exact = true;
  }

done:
  ctx->stream = main_stream;
  if (rc && implicit) {
    // an error mid-way: nothing may still be running on the side streams when the buffers go
    cudaStreamSynchronize(ctx->copy_stream);
    for (int k = 0; k < K && k < (int)ctx->side_streams.size(); k++) cudaStreamSynchronize(ctx->side_streams[k]);
  }
  if (!bidir) dev_free(ctx, status_dev); // (bidir: part of the zparts block)
  dev_free(ctx, row_scratch);
  if (!direct) dev_free(ctx, zparts_dev);
  dev_free(ctx, boff_dev);
  if (lat) gtnb_lattice_destroy(ctx, lat);
  if (!emissions_on_device) dev_free(ctx, e_dev);
  if (grads && !grads_on_device) dev_free(ctx, g_dev);
  dev_free(ctx, z_dev);
  dev_free(ctx, deltas_dev);
  dev_free(ctx, small_dev);
  return rc;
#undef TRY
#undef TRYCUDA
}

extern "C" int gtnb_ctc_loss(
    gtnb_ctx* ctx, int B, int T, int C, const float* emissions, int emissions_on_device,
    const int32_t* input_lens, const int32_t* targets, const int32_t* target_lens, int blank,
    float* losses_host, float* grads, int grads_on_device) {
  bool needs_exact = false;
  if (ctx) arena_begin(ctx);
  int rc = ctc_loss_run(ctx, B, T, C, emissions, emissions_on_device, input_lens, targets, target_lens, blank,
                        losses_host, grads, grads_on_device, ctx && ctx->use_implicit, &needs_exact);
  if (ctx) arena_end(ctx);
  if (rc == GTNB_OK && needs_exact)
    // a non-finite emission: the materialised lattice reproduces the reference's inf / NaN
    // propagation arc by arc (shortest.cpp:62-80), the implicit sweep cannot tell a missing
    // node from one whose score is -inf
    rc = ctc_loss_run(ctx, B, T, C, emissions, emissions_on_device, input_lens, targets, target_lens, blank,
                      losses_host, grads, grads_on_device, false, &needs_exact);
  return rc;
}

/*
 * viterbiPath(compose(linearGraph(T, C; e_b), transitions)) for a whole minibatch, with the
 * dense transitions graph of test/criterion_test.cpp:244-254 / :316-326, through the
 * factored kernel (k_dense.cu): the T*C*C lattice is never materialised.
 */
static int viterbi_dense_run(
    gtnb_ctx* ctx, int B, int T, int C, const float* emissions, int emissions_on_device,
    const int32_t* input_lens, const float* trans_w_host, int32_t* paths_host, float* scores_host) {
  if (!ctx || B < 0 || T < 0 || C <= 0 || !emissions || !trans_w_host)
    return fail(ctx, GTNB_ERR_INVALID_ARGUMENT, "gtnb_viterbi_dense: bad arguments");
  if (B == 0) return GTNB_OK;
  GTNB_CUDA(ctx, cudaSetDevice(ctx->device));
  const long long per = (long long)T * C;
  int rc = GTNB_OK;
  float *e_dev = nullptr, *tr_dev = nullptr, *sc_dev = nullptr;
  int32_t *T_dev = nullptr, *paths_dev = nullptr;
  uint8_t* bp = nullptr;
#define TRY(x)                 \
  do {                         \
    if ((rc = (x))) goto done; \
  } while (0)
#define TRYCUDA(call)                                      \
  do {                                                     \
    cudaError_t e__ = (call);                              \
    if (e__ != cudaSuccess) {                              \
      rc = cuda_fail(ctx, e__, #call, __FILE__, __LINE__); \
      goto done;                                           \
    }                                                      \
  } while (0)
  if (input_lens)
    for (int b = 0; b < B; b++)
      if (input_lens[b] < 0 || input_lens[b] > T)
        return fail(ctx, GTNB_ERR_INVALID_ARGUMENT, "gtnb_viterbi_dense: input_lens out of range");
  if (emissions_on_device) {
    e_dev = const_cast<float*>(emissions);
  } else {
    TRY(dev_alloc(ctx, &e_dev, per * B));
    TRYCUDA(cudaMemcpyAsync(e_dev, emissions, sizeof(float) * per * B, cudaMemcpyHostToDevice, ctx->stream));
  }
  TRY(dev_alloc(ctx, &tr_dev, (long long)C + (long long)C * C));
  TRY(dev_alloc(ctx, &sc_dev, B));
  TRY(dev_alloc(ctx, &paths_dev, (long long)B * std::max(T, 1)));
  TRY(dev_alloc(ctx, &bp, (long long)B * std::max(T, 1) * C));
  if (input_lens) TRY(dev_alloc(ctx, &T_dev, B));
  TRY(stage_begin(ctx));
  TRY(stage_upload(ctx, tr_dev, trans_w_host, sizeof(float) * ((size_t)C + (size_t)C * C)));
  if (input_lens) TRY(stage_upload(ctx, T_dev, input_lens, sizeof(int32_t) * B));
  TRY(stage_end(ctx));
  TRY(launch_viterbi_dense(ctx, B, T, C, T_dev, e_dev, per, tr_dev, bp, paths_dev, sc_dev));
  if (paths_host && T > 0)
    TRYCUDA(cudaMemcpyAsync(paths_host, paths_dev, sizeof(int32_t) * (size_t)B * T, cudaMemcpyDeviceToHost, ctx->stream));
  if (scores_host)
    TRYCUDA(cudaMemcpyAsync(scores_host, sc_dev, sizeof(float) * B, cudaMemcpyDeviceToHost, ctx->stream));
  TRYCUDA(cudaStreamSynchronize(ctx->stream));
done:
  if (!emissions_on_device) dev_free(ctx, e_dev);
  dev_free(ctx, tr_dev);
  dev_free(ctx, sc_dev);
  dev_free(ctx, paths_dev);
  dev_free(ctx, bp);
  dev_free(ctx, T_dev);
  return rc;
#undef TRY
#undef TRYCUDA
}

/* (the device scratch of a call comes from the context's call-scoped arena, as in gtnb_ctc_loss: no stream-ordered
 * allocations on the path after the first call of a shape) */
extern "C" int gtnb_viterbi_dense(
    gtnb_ctx* ctx, int B, int T, int C, const float* emissions, int emissions_on_device,
    const int32_t* input_lens, const float* trans_w_host, int32_t* paths_host, float* scores_host) {
  if (ctx) arena_begin(ctx);
  const int rc = viterbi_dense_run(ctx, B, T, C, emissions, emissions_on_device, input_lens, trans_w_host, paths_host,
                                   scores_host);
  if (ctx) arena_end(ctx);
  return rc;
}

/*
 * CTC forced alignment for a whole minibatch: viterbiPath + viterbiScore of intersect(ctcGraph(target_b), e_b)
 * on the implicit lattice (k_align.cu).  Utterances outside the kernel's envelope are rerun one by one on the
 * lattice route (compose + k_order.cu + the MODE_PATH kernels), which reproduces the reference's handling of
 * non-finite weights and unmatched labels arc by arc.
 */
namespace {

/* the CTC graph of benchmarks/ctc.cpp:40-58 as a host view, out lists in arcSort order when `sorted` */
struct CtcView {
  std::vector<uint8_t> flags;
  std::vector<int32_t> src, dst, lab, out_ptr, out_arcs;
  gtnb_graph_view v;
  CtcView(const int32_t* y, int U, int blank, bool sorted) {
    const int L = 2 * U + 1;
    flags.assign(L, 0);
    flags[0] |= 1;
    flags[L - 1] |= 2;
    if (L >= 2) flags[L - 2] |= 2;
    auto add = [&](int s, int d, int l) {
      src.push_back(s);
      dst.push_back(d);
      lab.push_back(l);
    };
    for (int l = 0; l < L; l++) {
      const int label = (l & 1) ? y[(l - 1) / 2] : blank;
      add(l, l, label);
      if (l > 0) add(l - 1, l, label);
      if ((l & 1) && l > 1 && label != y[(l - 3) / 2]) add(l - 2, l, label);
    }
    out_ptr.assign(L + 1, 0);
    for (int s : src) out_ptr[s + 1]++;
    for (int n = 0; n < L; n++) out_ptr[n + 1] += out_ptr[n];
    out_arcs.resize(src.size());
    std::vector<int32_t> pos(out_ptr.begin(), out_ptr.end() - 1);
    for (size_t a = 0; a < src.size(); a++) out_arcs[pos[src[a]]++] = (int32_t)a;
    if (sorted) // Graph::arcSort (graph.cpp:162-177): stable on these lists of <= 3 arcs
      for (int n = 0; n < L; n++)
        std::stable_sort(out_arcs.begin() + out_ptr[n], out_arcs.begin() + out_ptr[n + 1],
                         [&](int a, int b) { return lab[a] < lab[b]; });
    std::memset(&v, 0, sizeof(v));
    v.num_nodes = L;
    v.num_arcs = (int32_t)src.size();
    v.node_flags = flags.data();
    v.arc_src = src.data();
    v.arc_dst = dst.data();
    v.arc_ilabel = v.arc_olabel = lab.data();
    v.out_ptr = out_ptr.data();
    v.out_arcs = out_arcs.data();
  }
};

/* utterance b on the lattice route: labels / states rows [T] (states nullable) and the score, on the host */
int ctc_align_lattice(gtnb_ctx* ctx, const CtcView& g, int Tb, int T, int C, const float* e_dev, int32_t* labels,
                      int32_t* states, float* score) {
  const bool ties = ctx->exact_ties;
  ctx->exact_ties = true;
  gtnb_lattice* lat = nullptr;
  int rc = gtnb_compose_linear(ctx, 1, &g.v, 1, 0, &Tb, C, e_dev, (int64_t)Tb * C, &lat);
  ctx->exact_ties = ties;
  if (rc) return rc;
  std::vector<int32_t> arcs(std::max(Tb, 1), -1), il(std::max(Tb, 1), -1);
  int32_t len = -1;
  rc = gtnb_viterbi_path(ctx, lat, Tb, arcs.data(), il.data(), nullptr, nullptr, &len, nullptr);
  if (!rc) rc = gtnb_forward(ctx, lat, 1, score, nullptr);
  std::vector<int32_t> gi;
  if (!rc && states && len > 0) {
    int32_t nn = 0, na = 0;
    rc = gtnb_lattice_sizes(ctx, lat, &nn, &na);
    gi.resize(std::max(na, 1));
    if (!rc) rc = gtnb_lattice_download(ctx, lat, 0, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, gi.data(), nullptr);
  }
  gtnb_lattice_destroy(ctx, lat);
  if (rc) return rc;
  for (int t = 0; t < T; t++) {
    const bool on = t < len;
    labels[t] = on ? il[t] : -1;
    if (states) states[t] = on ? g.dst[gi[arcs[t]]] : -1;
  }
  return GTNB_OK;
}

} // namespace

static int ctc_align_run(
    gtnb_ctx* ctx, int B, int T, int C, const float* emissions, int emissions_on_device, const int32_t* input_lens,
    const int32_t* targets, const int32_t* target_lens, int blank, int arc_sorted, int32_t* labels, int32_t* states,
    int outputs_on_device, float* scores_host, std::vector<int32_t>& status) {
  if (!ctx || B < 0 || T < 0 || C <= 0 || (B > 0 && (!target_lens || !scores_host)) ||
      ((long long)B * T > 0 && (!emissions || !labels)))
    return fail(ctx, GTNB_ERR_INVALID_ARGUMENT, "gtnb_ctc_align: bad arguments");
  std::vector<int32_t> small(3ll * B);
  long long tot_t = 0;
  int maxL = 1;
  for (int b = 0; b < B; b++) {
    const int U = target_lens[b];
    if (U < 0) return fail(ctx, GTNB_ERR_INVALID_ARGUMENT, "gtnb_ctc_align: negative target length");
    if (U > 0 && !targets) return fail(ctx, GTNB_ERR_INVALID_ARGUMENT, "gtnb_ctc_align: targets is NULL");
    const int Tb = input_lens ? input_lens[b] : T;
    if (Tb < 0 || Tb > T) return fail(ctx, GTNB_ERR_INVALID_ARGUMENT, "gtnb_ctc_align: input_lens out of range");
    const int32_t* y = targets + tot_t;
    int out_deg = U > 0 ? 2 : 1;
    for (int u = 1; u < U; u++)
      if (y[u] != y[u - 1]) out_deg = 3; // a skip arc
    if (arc_sorted && out_deg > C)
      return fail(ctx, GTNB_ERR_UNSUPPORTED,
                  "gtnb_ctc_align: sorted CTC graph with out-degree > C (the reference's doubly-sorted matcher then "
                  "enumerates arcs in emission-label order, which neither route reproduces)");
    small[b] = Tb;
    small[B + b] = (int32_t)tot_t;
    small[2 * B + b] = U;
    maxL = std::max(maxL, 2 * U + 1);
    tot_t += U;
  }
  if (B == 0) return GTNB_OK;
  GTNB_CUDA(ctx, cudaSetDevice(ctx->device));
  const long long per = (long long)T * C;
  const long long n_out = (long long)B * T;
  int rc = GTNB_OK;
  float* e_dev = nullptr;
  int32_t *small_dev = nullptr, *lab_dev = nullptr, *st_dev = nullptr;
  uint8_t* bp = nullptr;
  float* res_dev = nullptr; // [scores | status]
#define TRY(x)                 \
  do {                         \
    if ((rc = (x))) goto done; \
  } while (0)
#define TRYCUDA(call)                                      \
  do {                                                     \
    cudaError_t e__ = (call);                              \
    if (e__ != cudaSuccess) {                              \
      rc = cuda_fail(ctx, e__, #call, __FILE__, __LINE__); \
      goto done;                                           \
    }                                                      \
  } while (0)
  if (emissions_on_device) {
    e_dev = const_cast<float*>(emissions);
  } else {
    TRY(dev_alloc(ctx, &e_dev, per * B));
    if (per) TRYCUDA(cudaMemcpyAsync(e_dev, emissions, sizeof(float) * per * B, cudaMemcpyHostToDevice, ctx->stream));
  }
  if (outputs_on_device) {
    lab_dev = labels;
    st_dev = states;
  } else {
    TRY(dev_alloc(ctx, &lab_dev, n_out));
    if (states) TRY(dev_alloc(ctx, &st_dev, n_out));
  }
  TRY(dev_alloc(ctx, &small_dev, 3ll * B + tot_t));
  TRY(dev_alloc(ctx, &bp, (long long)B * T * (long long)ctc_align_bp_pitch(maxL)));
  TRY(dev_alloc(ctx, &res_dev, 2ll * B));
  TRY(stage_begin(ctx));
  TRY(stage_upload(ctx, small_dev, small.data(), sizeof(int32_t) * small.size()));
  if (tot_t) TRY(stage_upload(ctx, small_dev + 3ll * B, targets, sizeof(int32_t) * tot_t));
  TRY(stage_end(ctx));
  TRY(launch_ctc_align(ctx, B, T, C, blank, arc_sorted, maxL, small_dev, e_dev, per, bp, lab_dev, st_dev, res_dev,
                       reinterpret_cast<int32_t*>(res_dev + B)));
  if (!outputs_on_device && n_out) {
    TRYCUDA(cudaMemcpyAsync(labels, lab_dev, sizeof(int32_t) * n_out, cudaMemcpyDeviceToHost, ctx->stream));
    if (states)
      TRYCUDA(cudaMemcpyAsync(states, st_dev, sizeof(int32_t) * n_out, cudaMemcpyDeviceToHost, ctx->stream));
  }
  TRY(readback_reserve(ctx, 2 * sizeof(float) * B));
  TRYCUDA(cudaMemcpyAsync(ctx->readback, res_dev, 2 * sizeof(float) * B, cudaMemcpyDeviceToHost, ctx->stream));
  TRYCUDA(cudaStreamSynchronize(ctx->stream));
  std::memcpy(scores_host, ctx->readback, sizeof(float) * B);
  status.assign(reinterpret_cast<int32_t*>(ctx->readback) + B, reinterpret_cast<int32_t*>(ctx->readback) + 2 * B);
done:
  if (!emissions_on_device) dev_free(ctx, e_dev);
  if (!outputs_on_device) {
    dev_free(ctx, lab_dev);
    dev_free(ctx, st_dev);
  }
  dev_free(ctx, small_dev);
  dev_free(ctx, bp);
  dev_free(ctx, res_dev);
  return rc;
#undef TRY
#undef TRYCUDA
}

extern "C" int gtnb_ctc_align(
    gtnb_ctx* ctx, int B, int T, int C, const float* emissions, int emissions_on_device, const int32_t* input_lens,
    const int32_t* targets, const int32_t* target_lens, int blank, int arc_sorted, int32_t* labels, int32_t* states,
    int outputs_on_device, float* scores_host) {
  std::vector<int32_t> status;
  if (ctx) arena_begin(ctx);
  int rc = ctc_align_run(ctx, B, T, C, emissions, emissions_on_device, input_lens, targets, target_lens, blank,
                         arc_sorted, labels, states, outputs_on_device, scores_host, status);
  if (ctx) arena_end(ctx);
  // the utterances outside the kernel's envelope, on the lattice route (outside the call's arena: their lattices
  // are large and rare, the arena keeps the size of the last call)
  long long off = 0;
  bool rerun = false;
  for (int b = 0; b < B && rc == GTNB_OK; off += target_lens[b], b++) {
    if (!status[b]) continue;
    rerun = true;
    const int Tb = input_lens ? input_lens[b] : T;
    const CtcView g(targets + off, target_lens[b], blank, arc_sorted != 0);
    std::vector<int32_t> lab_row(std::max(T, 1)), st_row(std::max(T, 1));
    float* e_b = nullptr;
    if (emissions_on_device) {
      e_b = const_cast<float*>(emissions) + (long long)b * T * C;
    } else if ((rc = dev_alloc(ctx, &e_b, (long long)Tb * C)) == GTNB_OK && Tb) {
      const cudaError_t ce = cudaMemcpyAsync(e_b, emissions + (long long)b * T * C, sizeof(float) * Tb * C,
                                             cudaMemcpyHostToDevice, ctx->stream);
      if (ce != cudaSuccess) rc = cuda_fail(ctx, ce, "cudaMemcpyAsync", __FILE__, __LINE__);
    }
    if (rc == GTNB_OK)
      rc = ctc_align_lattice(ctx, g, Tb, T, C, e_b, lab_row.data(), states ? st_row.data() : nullptr, &scores_host[b]);
    if (!emissions_on_device) dev_free(ctx, e_b);
    if (rc || !T) continue;
    const size_t row = sizeof(int32_t) * T;
    if (outputs_on_device) {
      rc = gtnb_memcpy_h2d(ctx, labels + (long long)b * T, lab_row.data(), row);
      if (!rc && states) rc = gtnb_memcpy_h2d(ctx, states + (long long)b * T, st_row.data(), row);
    } else {
      std::memcpy(labels + (long long)b * T, lab_row.data(), row);
      if (states) std::memcpy(states + (long long)b * T, st_row.data(), row);
    }
  }
  if (rc == GTNB_OK && outputs_on_device && rerun) rc = gtnb_ctx_synchronize(ctx);
  return rc;
}

/*
 * ASG criterion for a whole minibatch (test/criterion_test.cpp:244-305, examples/asg.cpp:59-81):
 *   loss_b = forwardScore(compose(e_b, transitions))
 *          - forwardScore(compose(compose(fal_b, transitions), e_b))
 * with the dense transitions graph shared by the batch; gradients w.r.t. the emissions and
 * (accumulated over the batch, graph.cpp:96-100) the transitions.  The denominator lattice
 * is materialised on the device (C + (T-1) C^2 arcs per utterance); compose(fal_b,
 * transitions) is a 2U-arc chain built on the host from the target (pure construction).
 */
static int asg_loss_run(
    gtnb_ctx* ctx, int B, int T, int C, const float* emissions, int emissions_on_device,
    const float* trans_w_host, const int32_t* targets, const int32_t* target_lens,
    float* losses_host, float* grads, int grads_on_device, float* trans_grad_host) {
  if (!ctx || B < 0 || T < 0 || C <= 0 || !emissions || !trans_w_host || !target_lens || !losses_host)
    return fail(ctx, GTNB_ERR_INVALID_ARGUMENT, "gtnb_asg_loss: bad arguments");
  if (B == 0) return GTNB_OK;
  GTNB_CUDA(ctx, cudaSetDevice(ctx->device));
  const long long per = (long long)T * C;
  const int nTrans = C + C * C;
  const bool want = grads || trans_grad_host;
  int rc = GTNB_OK;
  float *e_dev = nullptr, *g_dev = nullptr, *tg_dev = nullptr, *ft_grad = nullptr, *minus1 = nullptr;
  int32_t* ft_map_dev = nullptr;
  int32_t* status_dev = nullptr;
  bool implicit = false, needs_exact = false;
  gtnb_lattice *den = nullptr, *num = nullptr;
  cudaStream_t asg_main = ctx->stream;

  // transitions graph view (criterion_test.cpp:244-254)
  std::vector<uint8_t> tflags(C + 1, 2);
  tflags[0] = 1;
  std::vector<int32_t> tsrc(nTrans), tdst(nTrans), tlab(nTrans);
  for (int i = 0; i < C; i++) {
    tsrc[i] = 0;
    tdst[i] = i + 1;
    tlab[i] = i;
  }
  for (int i = 0; i < C; i++)
    for (int j = 0; j < C; j++) {
      const int a = C + i * C + j;
      tsrc[a] = j + 1;
      tdst[a] = i + 1;
      tlab[a] = i;
    }
  gtnb_graph_view tview;
  std::memset(&tview, 0, sizeof(tview));
  tview.num_nodes = C + 1;
  tview.num_arcs = nTrans;
  tview.node_flags = tflags.data();
  tview.arc_src = tsrc.data();
  tview.arc_dst = tdst.data();
  tview.arc_ilabel = tview.arc_olabel = tlab.data();
  tview.weights = trans_w_host;

  // compose(fal_b, transitions): node l = "l labels consumed"; arcs: 0->1, then per node a
  // self loop and the step to the next label, in the reference's creation order
  struct Ft {
    std::vector<uint8_t> flags;
    std::vector<int32_t> src, dst, lab, map;
    std::vector<float> w;
  };
  std::vector<Ft> ft(B);
  std::vector<gtnb_graph_view> fviews(B);
  std::vector<int32_t> ft_map;
  std::vector<int32_t> Tb(B, T);
  long long toff = 0;
  for (int b = 0; b < B; b++) {
    const int U = target_lens[b];
    if (U < 0) return fail(ctx, GTNB_ERR_INVALID_ARGUMENT, "gtnb_asg_loss: negative target length");
    const int32_t* y = targets + toff;
    toff += U;
    for (int u = 0; u < U; u++)
      if (y[u] < 0 || y[u] >= C) return fail(ctx, GTNB_ERR_INVALID_ARGUMENT, "gtnb_asg_loss: label out of range");
    Ft& f = ft[b];
    f.flags.assign(U + 1, 0);
    f.flags[0] |= 1;
    if (U > 0) f.flags[U] |= 2;
    auto add = [&](int s, int d, int lab, int tarc) {
      f.src.push_back(s);
      f.dst.push_back(d);
      f.lab.push_back(lab);
      f.w.push_back(trans_w_host[tarc]);
      f.map.push_back(tarc);
    };
    if (U > 0) add(0, 1, y[0], y[0]);
    for (int l = 1; l <= U; l++) {
      add(l, l, y[l - 1], C + y[l - 1] * C + y[l - 1]);
      if (l < U) add(l, l + 1, y[l], C + y[l] * C + y[l - 1]);
    }
    gtnb_graph_view& v = fviews[b];
    std::memset(&v, 0, sizeof(v));
    v.num_nodes = U + 1;
    v.num_arcs = (int)f.src.size();
    v.node_flags = f.flags.data();
    v.arc_src = f.src.data();
    v.arc_dst = f.dst.data();
    v.arc_ilabel = v.arc_olabel = f.lab.data();
    v.weights = f.w.data();
    ft_map.insert(ft_map.end(), f.map.begin(), f.map.end());
  }
  const long long nFt = (long long)ft_map.size();

#define TRY(x)                 \
  do {                         \
    if ((rc = (x))) goto done; \
  } while (0)
#define TRYCUDA(call)                                      \
  do {                                                     \
    cudaError_t e__ = (call);                              \
    if (e__ != cudaSuccess) {                              \
      rc = cuda_fail(ctx, e__, #call, __FILE__, __LINE__); \
      goto done;                                           \
    }                                                      \
  } while (0)
  if (emissions_on_device) {
    e_dev = const_cast<float*>(emissions);
  } else {
    TRY(dev_alloc(ctx, &e_dev, per * B));
    TRYCUDA(cudaMemcpyAsync(e_dev, emissions, sizeof(float) * per * B, cudaMemcpyHostToDevice, ctx->stream));
  }
  if (want) {
    if (grads && grads_on_device)
      g_dev = grads;
    else
      TRY(dev_alloc(ctx, &g_dev, per * B));
    TRYCUDA(cudaMemsetAsync(g_dev, 0, sizeof(float) * per * B, ctx->stream));
    TRY(dev_alloc(ctx, &tg_dev, nTrans));
    TRYCUDA(cudaMemsetAsync(tg_dev, 0, sizeof(float) * nTrans, ctx->stream));
    TRY(dev_alloc(ctx, &ft_grad, std::max<long long>(nFt, 1)));
    TRYCUDA(cudaMemsetAsync(ft_grad, 0, sizeof(float) * std::max<long long>(nFt, 1), ctx->stream));
    TRY(dev_alloc(ctx, &ft_map_dev, std::max<long long>(nFt, 1)));
    TRY(dev_alloc(ctx, &minus1, B));
  }
  // implicit sweeps (k_implicit.cu): neither lattice is built; the dense transitions graph takes
  // the G-lanes-per-node kernels, the forced-alignment chains the one-node-per-thread kernels
  implicit = ctx->use_implicit;
  if (implicit) {
    rc = compose_linear_impl(ctx, B, &tview, 1, 1, Tb.data(), C, e_dev, per, true, &den);
    if (!rc) rc = compose_linear_impl(ctx, B, fviews.data(), B, 0, Tb.data(), C, e_dev, per, true, &num);
    if (rc == GTNB_ERR_UNSUPPORTED) {
      if (den) gtnb_lattice_destroy(ctx, den);
      den = nullptr;
      implicit = false;
      rc = GTNB_OK;
    } else if (rc) {
      goto done;
    }
  }
  if (implicit) {
    TRY(ensure_side_streams(ctx, 0, 0));
    TRY(dev_alloc(ctx, &status_dev, 2ll * B));
    TRYCUDA(cudaMemsetAsync(status_dev, 0, sizeof(int32_t) * 2 * B, ctx->stream));
    // the numerator's sweeps (forced-alignment chains: small) run on the second stream beside the
    // denominator's (dense transitions: wide); they share nothing but the emission gradient, which both
    // accumulate with red.global.add
    TRYCUDA(cudaEventRecord(ctx->ev_fork, ctx->stream));
    TRYCUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_fork, 0));
    TRY(launch_implicit_forward(ctx, den, status_dev));
    ctx->stream = ctx->copy_stream;
    rc = launch_implicit_forward(ctx, num, status_dev + B);
    ctx->stream = asg_main;
    if (rc) goto done;
  } else {
    TRY(gtnb_compose_linear(ctx, B, &tview, 1, 1, Tb.data(), C, e_dev, per, &den));
    TRY(gtnb_compose_linear(ctx, B, fviews.data(), B, 0, Tb.data(), C, e_dev, per, &num));
    TRY(gtnb_forward(ctx, den, 0, nullptr, nullptr));
    TRY(gtnb_forward(ctx, num, 0, nullptr, nullptr));
  }
  if (want) {
    std::vector<float> m1(B, -1.0f);
    if (implicit) {
      TRY(stage_begin(ctx));
      TRY(stage_upload(ctx, minus1, m1.data(), sizeof(float) * B));
      TRY(stage_end(ctx));
      // +1 / -1: subtract's gradFunc (functions.cpp:53-58); graph-side gradients straight into
      // the transitions' (shared by the batch) and the forced-alignment chains' slabs
      TRYCUDA(cudaEventRecord(ctx->ev_fork, ctx->stream)); // the staged -1 seeds
      TRYCUDA(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_fork, 0));
      TRY(launch_implicit_backward(ctx, den, nullptr, g_dev, per, 0, -1, tg_dev));
      ctx->stream = ctx->copy_stream;
      rc = launch_implicit_backward(ctx, num, minus1, g_dev, per, 0, -1, ft_grad);
      ctx->stream = asg_main;
      if (rc) goto done;
    } else {
      TRY(gtnb_backward(ctx, den, 0, nullptr)); // +1 (subtract's gradFunc, functions.cpp:53-58)
      TRY(gtnb_backward(ctx, num, 0, m1.data())); // -1
      TRY(gtnb_compose_grad(ctx, den, tg_dev, g_dev, per));
      TRY(gtnb_compose_grad(ctx, num, ft_grad, g_dev, per));
    }
    if (implicit) { // join the numerator's stream
      TRYCUDA(cudaEventRecord(ctx->ev_join, ctx->copy_stream));
      TRYCUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
    }
    if (nFt) {
      TRY(stage_begin(ctx));
      TRY(stage_upload(ctx, ft_map_dev, ft_map.data(), sizeof(int32_t) * nFt));
      TRY(stage_end(ctx));
      TRY(launch_scatter_add(ctx, tg_dev, ft_map_dev, ft_grad, nFt));
    }
    if (grads && !grads_on_device)
      TRYCUDA(cudaMemcpyAsync(grads, g_dev, sizeof(float) * per * B, cudaMemcpyDeviceToHost, ctx->stream));
    if (trans_grad_host)
      TRYCUDA(cudaMemcpyAsync(trans_grad_host, tg_dev, sizeof(float) * nTrans, cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (implicit && !want) { // loss only: the numerator's forward sweep is still on the second stream
    TRYCUDA(cudaEventRecord(ctx->ev_join, ctx->copy_stream));
    TRYCUDA(cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
  }
  TRY(readback_reserve(ctx, 4 * sizeof(float) * B));
  {
    float* d = reinterpret_cast<float*>(ctx->readback);
    float* n = d + B;
    int32_t* st = reinterpret_cast<int32_t*>(n + B);
    TRYCUDA(cudaMemcpyAsync(d, den->out_scores, sizeof(float) * B, cudaMemcpyDeviceToHost, ctx->stream));
    TRYCUDA(cudaMemcpyAsync(n, num->out_scores, sizeof(float) * B, cudaMemcpyDeviceToHost, ctx->stream));
    if (implicit)
      TRYCUDA(cudaMemcpyAsync(st, status_dev, sizeof(int32_t) * 2 * B, cudaMemcpyDeviceToHost, ctx->stream));
    TRYCUDA(cudaStreamSynchronize(ctx->stream));
    for (int b = 0; b < B; b++) losses_host[b] = d[b] - n[b];
    if (implicit)
      for (int b = 0; b < 2 * B; b++) needs_exact |= st[b] != 0;
  }
done:
  dev_free(ctx, status_dev);
  if (den) gtnb_lattice_destroy(ctx, den);
  if (num) gtnb_lattice_destroy(ctx, num);
  if (!emissions_on_device) dev_free(ctx, e_dev);
  if (!(grads && grads_on_device)) dev_free(ctx, g_dev);
  dev_free(ctx, tg_dev);
  dev_free(ctx, ft_grad);
  dev_free(ctx, ft_map_dev);
  dev_free(ctx, minus1);
  if (rc == GTNB_OK && needs_exact) {
    // a non-finite weight: repeat through the materialised lattices, which reproduce the
    // reference's inf / NaN propagation arc by arc
    ctx->use_implicit = false;
    rc = gtnb_asg_loss(ctx, B, T, C, emissions, emissions_on_device, trans_w_host, targets, target_lens,
                       losses_host, grads, grads_on_device, trans_grad_host);
    ctx->use_implicit = true;
  }
  return rc;
#undef TRY
#undef TRYCUDA
}

extern "C" int gtnb_asg_loss(
    gtnb_ctx* ctx, int B, int T, int C, const float* emissions, int emissions_on_device,
    const float* trans_w_host, const int32_t* targets, const int32_t* target_lens,
    float* losses_host, float* grads, int grads_on_device, float* trans_grad_host) {
  if (ctx) arena_begin(ctx);
  const int rc = asg_loss_run(ctx, B, T, C, emissions, emissions_on_device, trans_w_host, targets, target_lens,
                              losses_host, grads, grads_on_device, trans_grad_host);
  if (ctx) arena_end(ctx);
  return rc;
}
