/*
 * gtn_b200.h -- C ABI of the B200-native gtn hot path.
 *
 * One shared library (gtn_b200/lib/libgtn_b200.so, sm_100a CUDA inside)
 * exporting plain-C entry points: opaque handles, plain pointers and sizes,
 * int status returns, no exceptions, no torch / STL types.  This is the seam a
 * gtn maintainer binds instead of the CPU implementations of
 *
 *   gtn::compose / gtn::intersect     /root/reference/gtn/functions.cpp:225-251
 *                                       -> detail::compose, functions/compose.cpp:377-522
 *   gtn::forwardScore / viterbiScore  functions.cpp:320-326 -> detail::shortestDistance,
 *                                       functions/shortest.cpp:86-188 (+ grad :33-82)
 *   gtn::viterbiPath                  functions.cpp:328-330 -> detail::shortestPath,
 *                                       functions/shortest.cpp:190-272
 *   compose gradFunc                  functions/compose.cpp:496-518
 *   gtn::linearGraph + setWeights     creations.cpp:20-33, graph.cpp:179-181
 *   parallelMap(fwd) / parallelMap(bwd)  benchmarks/ctc.cpp:150-165 (the batch seam)
 *
 * The reference has no FFI layer of its own (SURVEY.md section 8(b)); the C++
 * mirror of its public headers (gtn_b200/csrc/gtn/) and the pybind11 module
 * sit on top of exactly these functions -- see INTEGRATION.md.
 *
 * Conventions
 *  - every function returns GTNB_OK or a negative-free positive error code;
 *    gtnb_last_error(ctx) gives the message.  The C++ shim maps
 *    GTNB_ERR_INVALID_ARGUMENT -> std::invalid_argument,
 *    GTNB_ERR_LOGIC -> std::logic_error, others -> std::runtime_error, which
 *    is what the reference throws (shortest.cpp:150,230; graph.cpp:71-94).
 *  - all device work is enqueued on the context's stream; functions that
 *    return host results synchronise that stream, the others do not.
 *  - "dev" pointers are device memory on the context's device, "host"
 *    pointers are host memory (pinned or pageable).
 *  - there is NO CPU fallback: every compute entry point launches sm_100a
 *    kernels and fails with GTNB_ERR_RUNTIME when no CUDA device is usable.
 */
#ifndef GTN_B200_H
#define GTN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GTNB_VERSION 100

#define GTNB_OK 0
#define GTNB_ERR_INVALID_ARGUMENT 2 /* std::invalid_argument */
#define GTNB_ERR_LOGIC 3 /* std::logic_error */
#define GTNB_ERR_RUNTIME 4 /* std::runtime_error, incl. CUDA failures */
#define GTNB_ERR_UNSUPPORTED 5 /* shape outside what the device path covers */

#define GTNB_EPSILON (-1) /* gtn::epsilon, graph.h:21 */

typedef struct gtnb_ctx gtnb_ctx;
/* A packed batch of B device-resident graphs (levelised CSR-by-destination). */
typedef struct gtnb_lattice gtnb_lattice;

/*
 * Host view of one gtn::Graph (graph.h:56-465), borrowed for the call only.
 * Arrays are indexed by arc id / node id exactly as Graph numbers them.
 * in_ptr/in_arcs and out_ptr/out_arcs are the per-node arc lists in the
 * Graph's current order (i.e. after any arcSort, graph.cpp:162-177); pass NULL
 * for "insertion order".  accept/start give g.accept()/g.start() order; NULL
 * means ascending node id.
 */
typedef struct gtnb_graph_view {
  int32_t num_nodes;
  int32_t num_arcs;
  const uint8_t* node_flags; /* bit0 = start, bit1 = accept */
  const int32_t* arc_src;
  const int32_t* arc_dst;
  const int32_t* arc_ilabel;
  const int32_t* arc_olabel;
  const float* weights; /* NULL = all 0 */
  const int32_t* in_ptr; /* [num_nodes+1] or NULL */
  const int32_t* in_arcs; /* [num_arcs] */
  const int32_t* out_ptr;
  const int32_t* out_arcs;
  const int32_t* start; /* [num_start] or NULL */
  int32_t num_start;
  const int32_t* accept; /* [num_accept] or NULL */
  int32_t num_accept;
} gtnb_graph_view;

/* ---- context ------------------------------------------------------- */

/* cuda_stream: a cudaStream_t to enqueue on, or NULL for a private stream. */
int gtnb_ctx_create(int device, void* cuda_stream, gtnb_ctx** out);
void gtnb_ctx_destroy(gtnb_ctx* ctx);
/* ctx may be NULL: returns the calling thread's last creation error. */
const char* gtnb_last_error(const gtnb_ctx* ctx);
int gtnb_ctx_synchronize(gtnb_ctx* ctx);
void* gtnb_ctx_stream(gtnb_ctx* ctx);
/* the CUDA device ordinal the context was created on */
int gtnb_ctx_device(const gtnb_ctx* ctx);
int gtnb_version(void);
/* number of kernels this context has launched so far (bench bookkeeping) */
int64_t gtnb_ctx_launch_count(const gtnb_ctx* ctx);

/*
 * Tuning / testing switches.  "staged" (default 1): use the TMA-staged persistent
 * kernels for composed lattices; 0 forces the generic any-DAG kernels (libm-precise),
 * which is how the tests cross-check the two families.  "implicit" (default 1): the
 * criteria (gtnb_ctc_loss) sweep the frames of intersect(target graph, emissions) without
 * materialising the lattice; 0 makes them build it and run the lattice kernels.
 * "banded" (default 0, EXPERIMENTAL): value K in {1, 2, 4, 8}: gtnb_ctc_loss's implicit sweeps run
 * K frames per barrier with warp-shuffle neighbour exchange (k_banded.cu) when the target graphs
 * are band shaped.  "exact_ties" (default 0, EXPERIMENTAL; set before gtnb_compose_linear): gtnb_viterbi_path
 * on a composed lattice breaks exact score ties like the reference's shortestPath (k_order.cu).
 */
int gtnb_ctx_set_flag(gtnb_ctx* ctx, const char* name, int value);

/* device / pinned memory helpers so callers need no CUDA runtime of their own.
 * gtnb_device_alloc / _free are stream-ordered on the context's stream (cudaMallocAsync):
 * the memory is valid for work enqueued on that stream; synchronise before using it elsewhere. */
int gtnb_device_alloc(gtnb_ctx* ctx, size_t bytes, void** out);
int gtnb_device_free(gtnb_ctx* ctx, void* p);
int gtnb_host_alloc(gtnb_ctx* ctx, size_t bytes, void** out); /* pinned */
int gtnb_host_free(gtnb_ctx* ctx, void* p);
int gtnb_memcpy_h2d(gtnb_ctx* ctx, void* dst_dev, const void* src_host, size_t bytes);
int gtnb_memcpy_d2h(gtnb_ctx* ctx, void* dst_host, const void* src_dev, size_t bytes);
int gtnb_memset(gtnb_ctx* ctx, void* dst_dev, int value, size_t bytes);
/* CUDA-event timing on the context's stream */
int gtnb_timer_start(gtnb_ctx* ctx);
int gtnb_timer_stop(gtnb_ctx* ctx, float* ms); /* synchronises */
/*
 * Per-kernel CUDA-event timing on the context's stream.  gtnb_profile_read
 * synchronises, returns "name launches total_ms\n" lines (one per kernel name,
 * valid until the next call) and clears the log.
 */
int gtnb_profile_enable(gtnb_ctx* ctx, int on);
const char* gtnb_profile_read(gtnb_ctx* ctx);
/* write `bytes` of scratch to evict L2 between timed iterations */
int gtnb_flush_l2(gtnb_ctx* ctx);

/* ---- building device graphs ---------------------------------------- */

/*
 * Generic path: levelise B arbitrary host graphs (Kahn order exactly as
 * shortest.cpp:92-145 walks them) and upload them as one packed batch.
 * Structural errors the reference reports lazily ("Graph has a cycle,
 * self-loop or is disconnected!", shortest.cpp:149-152) are recorded per graph
 * and raised by gtnb_forward / gtnb_viterbi_path.
 */
int gtnb_pack(gtnb_ctx* ctx, int B, const gtnb_graph_view* graphs, gtnb_lattice** out);

/*
 * Frame-synchronous device composition (detail::compose, compose.cpp:377-522,
 * for the case one operand is a gtn::linearGraph): lattice_b =
 *   linear_first ? compose(linear(T_b, C; emissions_b), graphs_b)
 *                : compose(graphs_b, linear(T_b, C; emissions_b)).
 * graphs: n_graphs == B, or == 1 to share one graph across the batch (ASG
 * transitions).  The matched side of each graph must be epsilon-free
 * (GTNB_ERR_UNSUPPORTED otherwise; the host compose handles those).
 * emissions_dev: utterance b's row-major [T_b][C] matrix starts at
 * emissions_dev + b * emissions_stride.  The lattice keeps this pointer: it
 * must stay valid until the lattice is destroyed (weights are read again by
 * nothing, but compose_grad writes through grad pointers you pass then).
 * Arc weight = w_graph + e[t][label]  (compose.cpp:435), provenance kept per
 * arc for gtnb_compose_grad (gradInfo, compose.cpp:445).
 */
int gtnb_compose_linear(
    gtnb_ctx* ctx,
    int B,
    const gtnb_graph_view* graphs,
    int n_graphs,
    int linear_first,
    const int32_t* T, /* host [B] */
    int C,
    const float* emissions_dev,
    int64_t emissions_stride,
    gtnb_lattice** out);

/*
 * General composition on the device (k_gcompose.cu): replaces detail::compose (compose.cpp:377-522) for
 * operand pairs that are NOT frame-synchronous -- epsilon arcs on the matched side (compose.cpp:146-208,
 * 461-488), cyclic graphs, neither operand a chain (intersect(ctc, transitions) of timeNgramCtc,
 * benchmarks/ctc.cpp:118-123).  n_pairs pairs in one call, one CTA each; n_first / n_second are n_pairs, or 1
 * for an operand shared by every pair (parallel_map.h:77-89).  match_kind[b] is the matcher functions.cpp:225-251
 * would pick: 0 unsorted, 1 only the first operand sorted on the matched label, 2 only the second, 3 both.
 * The composed graphs keep the reference's node ids, arc ids and per-node arc order exactly.
 * GTNB_ERR_UNSUPPORTED when the product state space does not fit (>= 2^27 states per pair, or scratch larger
 * than half of the device memory).
 */
typedef struct gtnb_composed gtnb_composed;
int gtnb_compose_graphs(
    gtnb_ctx* ctx,
    int n_pairs,
    const gtnb_graph_view* first,
    int n_first,
    const gtnb_graph_view* second,
    int n_second,
    const int32_t* match_kind,
    gtnb_composed** out);
int gtnb_composed_sizes(const gtnb_composed* c, int pair, int32_t* num_nodes, int32_t* num_arcs);
/* any pointer may be NULL; gi_first / gi_second: compose.cpp:445's gradInfo (-1 on the epsilon side, :201-205) */
int gtnb_composed_download(
    gtnb_ctx* ctx,
    gtnb_composed* c,
    int pair,
    uint8_t* node_flags,
    int32_t* arc_src,
    int32_t* arc_dst,
    int32_t* arc_ilabel,
    int32_t* arc_olabel,
    float* weights,
    int32_t* gi_first,
    int32_t* gi_second);
void gtnb_composed_destroy(gtnb_ctx* ctx, gtnb_composed* c);

void gtnb_lattice_destroy(gtnb_ctx* ctx, gtnb_lattice* lat);
int gtnb_lattice_batch(const gtnb_lattice* lat);
/* per-graph node / arc counts (synchronises) */
int gtnb_lattice_sizes(gtnb_ctx* ctx, gtnb_lattice* lat, int32_t* num_nodes, int32_t* num_arcs);
/*
 * Materialise graph b on the host in Graph numbering (any pointer may be
 * NULL).  gi_graph / gi_linear are the compose provenance (-1 if none).
 */
int gtnb_lattice_download(
    gtnb_ctx* ctx,
    gtnb_lattice* lat,
    int b,
    uint8_t* node_flags,
    int32_t* arc_src,
    int32_t* arc_dst,
    int32_t* arc_ilabel,
    int32_t* arc_olabel,
    float* weights,
    int32_t* gi_graph,
    int32_t* gi_linear);

/* ---- the dynamic programs ------------------------------------------ */

/*
 * detail::shortestDistance over every graph of the batch (log semiring, or
 * tropical when `tropical`).  scores_host [B] (NULL = keep on device only).
 * Node scores stay in the lattice for the backward pass.
 * status_host [B] (nullable): per-graph GTNB_OK / GTNB_ERR_INVALID_ARGUMENT;
 * the call itself returns the first non-OK status.
 */
int gtnb_forward(gtnb_ctx* ctx, gtnb_lattice* lat, int tropical, float* scores_host, int32_t* status_host);

/*
 * shortestDistanceGrad (shortest.cpp:33-82): arc gradients of the last
 * gtnb_forward, scaled per graph by deltas_host[b] (NULL = 1).  Results stay
 * on the device; read them with gtnb_lattice_arc_grads or push them to the
 * compose operands with gtnb_compose_grad.
 */
int gtnb_backward(gtnb_ctx* ctx, gtnb_lattice* lat, int tropical, const float* deltas_host);

/* copy graph b's arc gradients (Graph arc numbering) to the host */
int gtnb_lattice_arc_grads(gtnb_ctx* ctx, gtnb_lattice* lat, int b, float* out_host);
/*
 * Overwrite graph b's arc gradients from the host (composed lattices; Graph arc
 * numbering == device numbering there).  Lets compose's gradFunc run on the device
 * when the deltas were produced or accumulated on the host (autograd.h:37).
 */
int gtnb_lattice_set_arc_grads(gtnb_ctx* ctx, gtnb_lattice* lat, int b, const float* grads_host);
/* device pointer to all arc gradients (device arc order) -- advanced use */
const float* gtnb_lattice_arc_grads_dev(const gtnb_lattice* lat);

/*
 * compose gradFunc (compose.cpp:496-518) for a lattice made by
 * gtnb_compose_linear: scatter-add the arc gradients to
 *   grad_graph_dev   [sum of graph arc counts] (one slab per graph, in batch
 *                    order; a single slab when the graph is shared), nullable
 *   grad_emissions_dev  utterance b at + b * grad_stride, [T_b][C], nullable
 * Both are accumulated into (addGrad semantics, graph.cpp:91-129); zero them
 * first for a fresh gradient.
 */
int gtnb_compose_grad(
    gtnb_ctx* ctx,
    gtnb_lattice* lat,
    float* grad_graph_dev,
    float* grad_emissions_dev,
    int64_t grad_stride);

/*
 * detail::shortestPath.  For each graph writes the best path's arcs (Graph
 * arc numbering, start -> end) into path_arcs_host + b * max_len and its
 * length into path_len_host[b] (-1: no accepting path).  ilabels/olabels of
 * those arcs go to path_ilabels_host / path_olabels_host (nullable).
 */
int gtnb_viterbi_path(
    gtnb_ctx* ctx,
    gtnb_lattice* lat,
    int max_len,
    int32_t* path_arcs_host,
    int32_t* path_ilabels_host,
    int32_t* path_olabels_host,
    float* path_weights_host, /* nullable: weights of the path's arcs */
    int32_t* path_len_host,
    int32_t* status_host);

/*
 * forwardScore of the emissions chain itself, forwardScore(linearGraph(T,C))
 * (the CTC normaliser, benchmarks/ctc.cpp:157): scores_dev[b] (device, [B]);
 * when grad_emissions_dev != NULL also accumulates delta_b * d score_b / d e
 * into it (delta = deltas_dev[b], or `delta_all` when deltas_dev == NULL).
 */
int gtnb_linear_forward(
    gtnb_ctx* ctx,
    int B,
    const int32_t* T, /* host [B] */
    int C,
    const float* emissions_dev,
    int64_t emissions_stride,
    int tropical,
    float* scores_dev,
    float* grad_emissions_dev,
    int64_t grad_stride,
    const float* deltas_dev,
    float delta_all);

/* ---- batched criteria: parallelMap(fwd)+parallelMap(bwd) in one call ---- */

/*
 * benchmarks/ctc.cpp:150-165 for a whole minibatch:
 *   loss_b = forwardScore(e_b) - forwardScore(intersect(ctcGraph(target_b), e_b))
 * and, when grads != NULL, d loss_b / d e_b.
 * emissions / grads: [B][T][C] row-major, on the device when *_on_device,
 * else host (copied in / out inside the call on the context's stream).
 * targets: concatenated labels, target_lens[B]; losses_host [B].
 * input_lens (nullable) gives per-utterance frame counts <= T.
 */
int gtnb_ctc_loss(
    gtnb_ctx* ctx,
    int B,
    int T,
    int C,
    const float* emissions,
    int emissions_on_device,
    const int32_t* input_lens,
    const int32_t* targets,
    const int32_t* target_lens,
    int blank,
    float* losses_host,
    float* grads,
    int grads_on_device);

/*
 * ASG criterion for a whole minibatch (test/criterion_test.cpp:244-305, examples/asg.cpp:59-81,
 * BASELINE.json configs[2]):
 *   loss_b = forwardScore(compose(e_b, transitions))
 *          - forwardScore(compose(compose(fal_b, transitions), e_b))
 * transitions: the dense graph described at gtnb_viterbi_dense, weights trans_w_host
 * [C + C*C], shared by the batch.  grads (nullable): d loss_b / d e_b, [B][T][C];
 * trans_grad_host (nullable): sum over the batch of d loss_b / d transitions, [C + C*C]
 * (the reference accumulates it under grad_lock, graph.cpp:96-100).
 */
int gtnb_asg_loss(
    gtnb_ctx* ctx,
    int B,
    int T,
    int C,
    const float* emissions,
    int emissions_on_device,
    const float* trans_w_host,
    const int32_t* targets,
    const int32_t* target_lens,
    float* losses_host,
    float* grads,
    int grads_on_device,
    float* trans_grad_host);

/*
 * viterbiPath + viterbiScore of compose(linearGraph(T, C; e_b), transitions) for a whole
 * minibatch (test/criterion_test.cpp:308-345, BASELINE.json configs[3]) WITHOUT
 * materialising the T*C*C lattice (32.75 M arcs per utterance at T=2000, C=128).
 * transitions is the dense graph of criterion_test.cpp:316-326: node 0 start, nodes 1..C
 * accept, arcs 0 -> i+1 (label i, weight trans_w[i]) and j+1 -> i+1 (label i, weight
 * trans_w[C + i*C + j]).  paths_host [B][T]: the best path's labels (-1 where there is no
 * accepting path / beyond input_lens[b]); scores_host [B]: viterbiScore.  Paths are
 * bit-identical to the reference's, ties included.  Needs C <= 256, C % 4 == 0.
 */
int gtnb_viterbi_dense(
    gtnb_ctx* ctx,
    int B,
    int T,
    int C,
    const float* emissions,
    int emissions_on_device,
    const int32_t* input_lens,
    const float* trans_w_host,
    int32_t* paths_host,
    float* scores_host);

/*
 * CTC forced alignment for a whole minibatch: for utterance b, with T_b = input_lens ? input_lens[b] : T,
 *   labels[b][t] (t < T_b) = ilabel of the t-th arc of viterbiPath(intersect(ctc_b, linearGraph(T_b, C; e_b)))
 *   scores_host[b]         = viterbiScore of the same lattice (shortest.cpp:190-272)
 * ctc_b is the CTC graph of benchmarks/ctc.cpp:40-58 for target b with `blank`, after arcSort() when
 * arc_sorted != 0 (as benchmarks/ctc.cpp:56 and the criterion do), in insertion order otherwise; the two differ
 * only in how exact score ties are broken.  Paths and scores are bit-identical to the reference's, ties
 * included.  states (nullable) [B][T]: the CTC graph node (0 .. 2U_b) the path is in after frame t.
 * Where there is no accepting path, or at t >= T_b, labels / states are -1; with no accepting path the score
 * is -inf (T_b = 0: 0 when U_b = 0).  emissions [B][T][C] (device pointer when emissions_on_device);
 * labels / states are device pointers when outputs_on_device, else host.  Targets, target_lens, input_lens
 * are host arrays as for gtnb_ctc_loss.
 * The lattice is never built (k_align.cu); utterances with a non-finite emission on a lattice arc, labels or
 * blank outside [0, C), or more than 2047 target labels are computed on the lattice route instead.
 * GTNB_ERR_UNSUPPORTED when arc_sorted and a CTC graph node has more out-arcs than C (C < 3): the reference's
 * doubly-sorted matcher then orders a state's arcs by emission label, which neither route reproduces.
 */
int gtnb_ctc_align(
    gtnb_ctx* ctx,
    int B,
    int T,
    int C,
    const float* emissions,
    int emissions_on_device,
    const int32_t* input_lens,
    const int32_t* targets,
    const int32_t* target_lens,
    int blank,
    int arc_sorted,
    int32_t* labels,
    int32_t* states,
    int outputs_on_device,
    float* scores_host);

#ifdef __cplusplus
}
#endif
#endif /* GTN_B200_H */
