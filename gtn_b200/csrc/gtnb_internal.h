/*
 * Internal declarations shared by the C-ABI translation units.
 * Nothing here is visible through include/gtn_b200.h.
 */
#pragma once

#ifdef GTNB_HOST_EMU
#error "GTNB_HOST_EMU is for tests/emu only (kernel sources compiled by g++ for the CPU test suite): the product library is never built with it, and this header is not part of that build"
#endif

#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "gtn_b200.h"

#include "gtnb_meta.h" // GraphMeta + layout constants: plain data, shared with the host-side kernel emulation (tests/emu)

/* dynamic shared memory of the CTA (the host-side emulation defines its own) */
#define GTNB_DYNAMIC_SMEM(type, name) extern __shared__ __align__(16) type name[]
#define GTNB_DYNAMIC_SMEM_128(type, name) extern __shared__ __align__(128) type name[]
#define GTNB_STATIC_SMEM(type, name, count) __shared__ type name[count]
#define GTNB_STATIC_SMEM_2D(type, name, d0, d1) __shared__ type name[d0][d1]

// k_bidir.cu is gtnb_ctc_loss's default path (gtnb_ctx_set_flag("bidir", 0): the two sweeps of k_implicit.cu):
// 0.39 ms in one launch against 0.17 + 0.24 ms (+ k_linear.cu beside them), and 4-5x closer to float64
constexpr bool kBidirDefault = true;

struct gtnb_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  std::string err;
  int64_t launches = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  void* flush_buf = nullptr;
  size_t flush_bytes = 0;
  int sm_count = 148;
  size_t total_mem = 0; // device memory, read once at context creation
  // pinned staging: every small host->device upload of one API call is packed here and
  // copied asynchronously (pageable copies would stall the stream each time)
  unsigned char* stage = nullptr;
  size_t stage_bytes = 0, stage_used = 0;
  cudaEvent_t stage_ev = nullptr;
  bool stage_pending = false;
  // second stream + events: overlap the host->device copy of the emissions with the
  // composition passes that only need the target graphs
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  // chunk streams / events: a host-buffer criterion call is cut into sub-batches whose
  // H2D copy, kernels and D2H copy overlap each other (gtnb_criteria.cu)
  std::vector<cudaStream_t> side_streams;
  std::vector<cudaEvent_t> side_events;
  // pinned read-back buffer for small device->host results
  unsigned char* readback = nullptr;
  size_t readback_bytes = 0;
  // optional per-kernel CUDA-event timing (gtnb_profile_*)
  struct ProfEntry {
    const char* name;
    cudaEvent_t a, b;
  };
  bool use_staged = true; // gtnb_ctx_set_flag("staged", 0) forces the generic kernels
  bool use_implicit = true; // gtnb_ctx_set_flag("implicit", 0): criteria materialise the lattice
  int bidir_mode = -1; // k_bidir.cu on CTC graphs ("bidir_mode" flag): 1 PAIR kernels, 2 QUAD, 0 one node per thread; -1 (default) = what was measured fastest: PAIR with a gradient (0.282 vs 0.309 ms), QUAD for loss-only calls (0.087 vs 0.095 ms)
  bool use_bidir = kBidirDefault; // gtnb_ctx_set_flag("bidir", 0): the CTC criterion takes the two sweeps of k_implicit.cu instead of the bidirectional kernel (k_bidir.cu)
  bool exact_ties = true; // gtnb_ctx_set_flag("exact_ties", 0) turns it off: composed lattices are put in the reference's relaxation order so that viterbiPath breaks exact ties like shortest.cpp:212-218 (k_order.cu)
  int use_banded = 0; // gtnb_ctx_set_flag("banded", K): EXPERIMENTAL temporally blocked CTC sweeps (k_banded.cu), K frames per barrier
  // Call-scoped device arena (the criteria): while arena_on, dev_alloc bumps a pointer inside one cached
  // allocation instead of ~25 stream-ordered allocations per call (each a microsecond or two of host time
  // ahead of the first launch); everything allocated in the scope is released together when it ends.
  unsigned char* arena = nullptr;
  size_t arena_cap = 0, arena_off = 0, arena_need = 0;
  bool arena_on = false;
  bool profiling = false;
  std::vector<ProfEntry> prof;
  std::vector<cudaEvent_t> ev_pool;
  std::string prof_text;
};

// rows of the saved scores of an implicit lattice whose graphs have at most this many nodes (k_bidir.cu's FX kernels)
constexpr int kImplicitFixedPitch = 224;

struct gtnb_lattice {
  int B = 0;
  bool composed = false;
  bool linear_first = false;
  bool shared_graph = false;
  bool level_local = false; // every arc goes level l-1 -> l
  bool forward_done = false;
  bool sizes_known = false;
  int score_pitch = 0; // implicit lattices: floats per saved-score row when every row has the same (0: the graph's node count rounded up to 4)
  bool order_pending = false; // exact_ties: rows still in compose order; sorted by the first viterbi_path
  bool order_locked = false; // arc ids already handed out (download / backward): the rows stay as they are
  int forward_mode = -1;
  int C = 0;
  int max_lvl_nodes = 0, max_lvl_arcs = 0; // upper bounds over the batch
  int max_in_deg = 0, max_out_deg = 0; // of the graph operands (composed lattices)
  int max_T = 0;
  long long tot_N = 0, tot_A = 0, tot_L = 0, tot_acc = 0, tot_bl = 0, tot_bn = 0;
  long long tot_sgN = 0, tot_sgA = 0;

  std::vector<gtnb::GraphMeta> meta_h;
  gtnb::GraphMeta* meta = nullptr;

  // lattice proper
  int32_t* lvl_node_ptr = nullptr;
  int32_t* lvl_arc_ptr = nullptr;
  uint32_t* row_ptr = nullptr;
  int2* arcs = nullptr; // per arc {x = source node, y = bits of the fp32 weight}
  int32_t* acc_nodes = nullptr;
  // provenance of composed arcs (gradInfo)
  int2* gi = nullptr; // per arc {x = arc of the graph operand, y = arc of the linear operand}
  // packed graphs: mapping back to Graph numbering + backward schedule
  int32_t* node_orig = nullptr;
  int32_t* arc_orig = nullptr;
  int32_t* relax_rank = nullptr;
  int32_t* blvl_ptr = nullptr;
  int32_t* bnodes = nullptr;
  // saved state
  float* scores = nullptr;
  float* out_scores = nullptr; // [B]
  int32_t* best_accept = nullptr; // [B] tropical: best accept node
  float* node_grad = nullptr;
  float* arc_grad = nullptr;
  int32_t* back_ptr = nullptr;
  // compose operands kept on the device
  const float* emissions = nullptr;
  int64_t emissions_stride = 0;
  uint8_t* sg_flags = nullptr; // per small-graph node
  int32_t* sg_in_ptr = nullptr; // [sgN + 1] per graph
  int32_t* sg_in_src = nullptr; // per in-entry (sgA)
  int32_t* sg_in_label = nullptr; // matched label, -1 = can never match
  int32_t* sg_in_arc = nullptr; // Graph arc id
  float* sg_in_w = nullptr;
  int32_t* sg_ilabel = nullptr; // by arc id
  int32_t* sg_olabel = nullptr;
  // exact_ties only (else NULL): per in-entry the arc's position in its source's out list; per node its index in g.start()
  int32_t* sg_out_pos = nullptr;
  int32_t* sg_start_rank = nullptr;
  uint32_t* alive = nullptr; // [B][max_T+1][W] bitmasks
  int alive_words = 0;

  // host copies needed to answer queries on packed graphs
  std::vector<std::vector<int32_t>> h_node_orig, h_arc_orig, h_ilabel, h_olabel;
  std::vector<int32_t> h_arcs_orig_count; // Graph's own arc count (>= device A)
};

namespace gtnb {

struct SgDims {
  int N, A, n_acc;
  int all_valid = 0;
  int uniform = 0;
  int max_in = 0, max_out = 0; // largest in- / out-degree of a node
};
int composed_alloc(
    gtnb_ctx* ctx, int B, const SgDims* dims, int n_graphs, int linear_first, const int32_t* T,
    int C, const float* emissions_dev, int64_t emissions_stride, std::vector<long long>& sgn,
    std::vector<long long>& sga, gtnb_lattice** out, bool implicit_only = false);
int stage_begin(gtnb_ctx* ctx);
int stage_upload(gtnb_ctx* ctx, void* dst_dev, const void* src_host, size_t bytes);
int stage_end(gtnb_ctx* ctx);
/* copies into the pinned staging buffer WITHOUT an upload and returns the address: pinned memory is mapped into the
 * device's address space (unified addressing), a kernel may read it in place */
int stage_reserve(gtnb_ctx* ctx, size_t bytes); // room for everything the pass will place (256-byte granules)
int stage_place(gtnb_ctx* ctx, const void* src_host, size_t bytes, void** where);
int readback_reserve(gtnb_ctx* ctx, size_t bytes);
int launch_ctc_build(
    gtnb_ctx* ctx, gtnb_lattice* lat, const int32_t* targets_dev, const int32_t* tgt_off_dev,
    const int32_t* tgt_len_dev, int blank);

int launch_scatter_add(gtnb_ctx* ctx, float* dst, const int32_t* idx, const float* src, long long n);
int launch_sub(gtnb_ctx* ctx, const float* a, const float* b, float* out, int n);

int fail(gtnb_ctx* ctx, int code, const std::string& msg);
int cuda_fail(gtnb_ctx* ctx, cudaError_t e, const char* what, const char* file, int line);

#define GTNB_CUDA(ctx, call)                                              \
  do {                                                                    \
    cudaError_t e__ = (call);                                             \
    if (e__ != cudaSuccess)                                               \
      return ::gtnb::cuda_fail((ctx), e__, #call, __FILE__, __LINE__);    \
  } while (0)

#define GTNB_CHECK_LAUNCH(ctx)                                            \
  do {                                                                    \
    (ctx)->launches++;                                                    \
    cudaError_t e__ = cudaGetLastError();                                 \
    if (e__ != cudaSuccess)                                               \
      return ::gtnb::cuda_fail((ctx), e__, "kernel launch", __FILE__, __LINE__); \
  } while (0)

inline cudaEvent_t prof_event(gtnb_ctx* ctx) {
  cudaEvent_t e;
  if (!ctx->ev_pool.empty()) {
    e = ctx->ev_pool.back();
    ctx->ev_pool.pop_back();
  } else {
    cudaEventCreate(&e);
  }
  return e;
}
inline void prof_begin(gtnb_ctx* ctx, const char* name) {
  if (!ctx->profiling) return;
  gtnb_ctx::ProfEntry pe{name, prof_event(ctx), prof_event(ctx)};
  cudaEventRecord(pe.a, ctx->stream);
  ctx->prof.push_back(pe);
}
inline void prof_end(gtnb_ctx* ctx) {
  if (!ctx->profiling || ctx->prof.empty()) return;
  cudaEventRecord(ctx->prof.back().b, ctx->stream);
}

/* Launch a kernel on the context's stream, count it, time it when profiling. */
#define GTNB_LAUNCH(ctx, name, ...)  \
  do {                               \
    ::gtnb::prof_begin((ctx), name); \
    __VA_ARGS__;                     \
    ::gtnb::prof_end((ctx));         \
    GTNB_CHECK_LAUNCH(ctx);          \
  } while (0)

/* Opt a kernel in to the full dynamic shared-memory window, once per (device, kernel).  The
 * attribute is process-wide: setting it per launch to that launch's size races between the
 * per-thread contexts of the gtn:: layer (one thread lowers it under another's launch). */
constexpr int kMaxDynamicSmem = 227 * 1024;
int ensure_max_smem(gtnb_ctx* ctx, const void* kernel);

template <typename T>
int dev_alloc(gtnb_ctx* ctx, T** p, long long n) {
  *p = nullptr;
  if (n <= 0) n = 1;
  // +16 elements of slack: staged copies round their windows up to 16 bytes
  const size_t bytes = sizeof(T) * (size_t)(n + 16);
  if (ctx->arena_on) {
    const size_t sz = (bytes + 255) & ~(size_t)255;
    ctx->arena_need += sz;
    if (ctx->arena_off + sz <= ctx->arena_cap) {
      *p = reinterpret_cast<T*>(ctx->arena + ctx->arena_off);
      ctx->arena_off += sz;
      return GTNB_OK;
    }
  }
  GTNB_CUDA(ctx, cudaMallocAsync((void**)p, bytes, ctx->stream));
  return GTNB_OK;
}

template <typename T>
void dev_free(gtnb_ctx* ctx, T*& p) {
  const unsigned char* q = reinterpret_cast<const unsigned char*>(p);
  if (p && !(ctx->arena && q >= ctx->arena && q < ctx->arena + ctx->arena_cap)) cudaFreeAsync((void*)p, ctx->stream);
  p = nullptr;
}

/* the arena scope of one criterion call: begin before the first dev_alloc, end after the last dev_free (and
 * after the stream was synchronised, which every criterion does to return its losses) */
inline void arena_begin(gtnb_ctx* ctx) {
  ctx->arena_on = true;
  ctx->arena_off = 0;
  ctx->arena_need = 0;
}
inline void arena_end(gtnb_ctx* ctx) {
  ctx->arena_on = false;
  if (ctx->arena_need > ctx->arena_cap) { // grow for the next call of this shape
    if (ctx->arena) cudaFreeAsync(ctx->arena, ctx->stream);
    ctx->arena = nullptr;
    ctx->arena_cap = 0;
    const size_t want = ctx->arena_need + (ctx->arena_need >> 3);
    void* fresh = nullptr;
    if (cudaMallocAsync(&fresh, want, ctx->stream) == cudaSuccess) {
      ctx->arena = static_cast<unsigned char*>(fresh);
      ctx->arena_cap = want;
    } else {
      cudaGetLastError(); // no arena: the plain allocations keep working
    }
  }
}

// Upload through pinned staging is overkill for the small metadata here;
// pageable cudaMemcpyAsync is synchronous wrt the host and safe.
template <typename T>
int upload(gtnb_ctx* ctx, T* dst, const T* src, long long n) {
  if (n <= 0) return GTNB_OK;
  GTNB_CUDA(ctx, cudaMemcpyAsync(dst, src, sizeof(T) * (size_t)n, cudaMemcpyHostToDevice, ctx->stream));
  return GTNB_OK;
}

inline long long align_up(long long v, long long a) {
  return (v + a - 1) / a * a;
}

// kernels (k_shortest.cu)
int launch_forward(gtnb_ctx* ctx, gtnb_lattice* lat, int mode);
int launch_backward(gtnb_ctx* ctx, gtnb_lattice* lat, int tropical, const float* deltas_dev);
int launch_traceback(gtnb_ctx* ctx, gtnb_lattice* lat, int max_len, int32_t* path_dev, int32_t* len_dev);
int launch_gather_prov(gtnb_ctx* ctx, gtnb_lattice* lat, int max_len, const int32_t* path_dev, const int32_t* len_dev, int32_t* prov_graph, int32_t* prov_linear, float* path_w);
// kernels (k_staged.cu): TMA-staged persistent kernels for level-local lattices
bool staged_supported(const gtnb_lattice* lat);
int launch_forward_staged(gtnb_ctx* ctx, gtnb_lattice* lat, int mode);
int launch_backward_staged(gtnb_ctx* ctx, gtnb_lattice* lat, int tropical, const float* deltas_dev);
int launch_backward_fused(
    gtnb_ctx* ctx, gtnb_lattice* lat, const float* deltas_dev, float* grad_emis, int64_t grad_stride);
// kernels (k_dense.cu): factored dense-trellis Viterbi
bool implicit_supported(const gtnb_lattice* lat);
bool implicit_dims_supported(const SgDims* dims, int n_graphs);
int launch_implicit_forward(gtnb_ctx* ctx, gtnb_lattice* lat, int32_t* status_dev, int b0 = 0, int nb = -1);
/* k_bidir.cu: the CTC criterion in one launch (two-CTA clusters meeting in the middle), normaliser included */
bool bidir_supported(const gtnb_lattice* lat, const float* emissions, int64_t stride, const float* grad, int64_t grad_stride);
int bidir_blocks(int max_T);
int bidir_zparts(); // partial sums of forwardScore(emissions) per CTA
int launch_bidir_ctc(
    gtnb_ctx* ctx, gtnb_lattice* lat, int32_t* status_dev, float* zparts_dev, float* boff_dev, float* grad_emis,
    int64_t grad_stride, int b0 = 0, int nb = -1, int zero_w = 0, float* out_scores_dev = nullptr,
    int ctc_blank = -1, const int32_t* targets_dev = nullptr, const int32_t* tgt_off_dev = nullptr,
    const GraphMeta* meta_src = nullptr); // meta_src: the descriptors somewhere else than lat->meta (mapped host memory)
// ctc_blank >= 0 + the targets: CTC target graphs, taken from the targets themselves (PAIR / QUAD kernels)
bool bidir_takes_targets(const gtnb_lattice* lat, int zero_w, int ctc_blank);
/* k_order.cu (experimental): a composed lattice's rows and accept list in the order the reference's shortestPath relaxes / creates them */
int launch_relax_order(gtnb_ctx* ctx, gtnb_lattice* lat);
/* k_banded.cu (experimental): same contract as the implicit sweeps, for band-shaped graph operands */
bool banded_supported(const gtnb_ctx* ctx, const gtnb_lattice* lat);
int launch_banded_forward(gtnb_ctx* ctx, gtnb_lattice* lat, int32_t* status_dev, int b0 = 0, int nb = -1);
int launch_banded_backward(
    gtnb_ctx* ctx, gtnb_lattice* lat, const float* deltas_dev, float* grad_emis, int64_t grad_stride,
    int b0 = 0, int nb = -1);
int launch_implicit_backward(
    gtnb_ctx* ctx, gtnb_lattice* lat, const float* deltas_dev, float* grad_emis, int64_t grad_stride,
    int b0 = 0, int nb = -1, float* grad_graph = nullptr);
int compose_linear_impl(
    gtnb_ctx* ctx, int B, const gtnb_graph_view* graphs, int n_graphs, int linear_first, const int32_t* T,
    int C, const float* emissions_dev, int64_t emissions_stride, bool implicit_only, gtnb_lattice** out);
int ensure_side_streams(gtnb_ctx* ctx, int n_streams, int n_events);
int launch_viterbi_dense(
    gtnb_ctx* ctx, int B, int T_max, int C, const int32_t* T_dev, const float* emis, int64_t stride,
    const float* trans_dev, uint8_t* bp, int32_t* paths, float* scores);
// kernels (k_align.cu): CTC forced alignment on the implicit lattice; small_dev = [T_b | target offsets | U | targets],
// outputs [B][T_max]; status[b] != 0: utterance b is outside the kernel's envelope and was not written
int launch_ctc_align(
    gtnb_ctx* ctx, int B, int T_max, int C, int blank, int arc_sorted, int maxL, const int32_t* small_dev,
    const float* emis, int64_t stride, uint8_t* bp, int32_t* labels, int32_t* states, float* scores,
    int32_t* status);
size_t ctc_align_bp_pitch(int maxL); // bytes of one back-pointer row
// kernels (k_compose.cu)
int launch_compose(gtnb_ctx* ctx, gtnb_lattice* lat, cudaEvent_t emissions_ready = nullptr);
int launch_compose_grad(gtnb_ctx* ctx, gtnb_lattice* lat, float* grad_graph, float* grad_emis, int64_t grad_stride);
// kernels (k_linear.cu)
int launch_linear_forward(
    gtnb_ctx* ctx, int B, const int32_t* T_dev, int maxT, int C, const float* emis, int64_t stride,
    int tropical, float* scores, float* grad, int64_t grad_stride, const float* deltas, float delta_all,
    int overwrite = 0, float* scratch = nullptr);


} // namespace gtnb
