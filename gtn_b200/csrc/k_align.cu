/*
 * k_align.cu -- batched CTC forced alignment WITHOUT the lattice: viterbiPath + viterbiScore of
 * intersect(ctcGraph(target_b), linearGraph(T_b, C; e_b)) (shortest.cpp:190-272, benchmarks/ctc.cpp:40-58),
 * the CTC graph taken from the targets in the kernel.  The lattice route (compose + k_order.cu + the
 * MODE_PATH kernels) writes ~2 M arcs per utterance at T=2000, U=200 and sorts them; this sweep keeps one
 * score, two order keys and one back-pointer byte per (frame, node).
 *
 * Exactness (paths and scores == the reference's, ties included):
 *   - candidate = fl(score[u] + fl(0 + e[t][label(v)])): the composed arc weight is ctc weight (0) +
 *     emission (compose.cpp:435), relaxed as fl(score + w) (shortest.cpp:214).  Candidates are compared
 *     after the add.
 *   - the first-relaxed predecessor among the maxima wins (strict '>', shortest.cpp:215).  In-arc
 *     e: (u, t) -> (v, t+1) is relaxed at rank pos_P[u] * 4 + o(e), o(e) the position of e in u's out
 *     list (insertion order [self, step, skip], or the stable ilabel sort of arcSort, graph.cpp:162-177).
 *     pos_P / pos_D, the states' positions in the reference's pop / creation orders, follow the key_P /
 *     key_D recurrences of k_order.cu (max / min over the alive in-arcs, then the rank among the frame's
 *     alive states), computed per frame inside the sweep: presence bitmaps of the keys + prefix popcounts.
 *   - the best accept node is the first strictly greatest in creation (pos_D) order at frame T_b.
 *   A state (v, t) is alive -- exists in the composed graph -- iff v is reachable from node 0 in t arcs and
 *   reaches an accept node in T_b - t arcs.  Every node has a self-loop, so that is
 *   fmin(v) <= t <= T_b - dist(v) with fmin / dist the shortest arc counts from node 0 / to an accept node.
 *
 * Envelope: finite candidate scores (a non-finite emission on a used arc, or an overflow, breaks the
 * equivalence with the lattice's -inf handling), labels and blank in [0, C), 2U+1 <= the layout's
 * capacity.  Otherwise status[b] != 0 and nothing else of utterance b is written: the host reruns it on
 * the lattice route.
 *
 * One CTA per utterance, NPT nodes per thread (node v = tid + k * blockDim).  Per frame: candidates and new
 * keys (reading the sources' ranks straight from the previous frame's bitmaps), barrier, prefix popcounts
 * (warps 0 and 1), barrier.  Back-pointers (0 self, 1 step, 2 skip) go to HBM, one byte per (frame, node);
 * the traceback stages kTraceRows rows of the window the path can occupy into shared memory with the
 * whole CTA, then one thread walks them.
 */
#ifdef GTNB_HOST_EMU // this file compiled by g++ against tests/emu/simt_emu.h (CPU test suite)
#include <algorithm>

#include "simt_emu.h"
#else
#include <cuda_runtime.h>
#include <math_constants.h>

#include <algorithm>

#include "gtnb_internal.h"
#endif

namespace gtnb {

constexpr int kAlignMaxThreads = 512;
constexpr int kAlignMaxNPT = 8;
constexpr int kAlignMaxNodes = kAlignMaxThreads * kAlignMaxNPT; // 2U + 1, i.e. U <= 2047
constexpr int kAlignTraceRows = 64;
constexpr int kAlignStageW = kAlignTraceRows / 2 + 2; // words of one staged row: 2 * rows + 1 bytes at any alignment

/* node pitch of the shared-memory rows for a batch whose largest CTC graph has maxL nodes */
inline int align_pitch(int maxL) {
  return (std::min(std::max(maxL, 1), kAlignMaxNodes) + 31) / 32 * 32;
}
/* block size and nodes per thread for pitch P: one node per thread up to kAlignMaxThreads nodes */
inline void align_layout(int P, int* threads, int* npt) {
  *threads = std::max(64, std::min(P, kAlignMaxThreads));
  int n = 1;
  while (n * *threads < P) n *= 2;
  *npt = n;
}
inline size_t align_smem_bytes(int P) {
  const int WB = P / 8; // key bitmap words: keys < 4 P
  return sizeof(float) * 2 * P + sizeof(int) * 4 * P // scores, key_D, key_P (two frames each)
         + sizeof(uint32_t) * 4 * WB + sizeof(int) * 2 * WB // bitmaps (two frames x D / P), prefix popcounts
         + sizeof(int) * (P / 2 + 1) // targets
         + sizeof(int) * 2 * P // first / last alive frame
         + sizeof(uint32_t) * kAlignTraceRows * kAlignStageW + sizeof(int) * 4;
}

namespace {

constexpr int kNoKey = 0x7fffffff;

__device__ __forceinline__ int key_rank(const uint32_t* bm, const int* pf, int key) {
  return pf[key >> 5] + __popc(bm[key >> 5] & ((1u << (key & 31)) - 1u));
}

/*
 * small: [T_b (B) | target offset (B) | U (B) | targets].  Outputs [B][T_max]; states nullable.
 * status[b]: 0 ok, 1 non-finite score, 2 labels / size outside the envelope.
 */
template <int NPT>
__global__ void __launch_bounds__(kAlignMaxThreads) ctc_align_kernel(
    int B,
    int T_max,
    int C,
    int blank,
    int arc_sorted,
    int P,
    const int32_t* __restrict__ small,
    const float* __restrict__ emis,
    long long stride,
    uint8_t* __restrict__ bp, // [B][T_max][P]
    int32_t* __restrict__ labels,
    int32_t* __restrict__ states,
    float* __restrict__ scores,
    int32_t* __restrict__ status) {
  GTNB_DYNAMIC_SMEM(unsigned char, smem_raw);
  const int WB = P / 8;
  float* sc = reinterpret_cast<float*>(smem_raw); // [2][P]
  int* kD = reinterpret_cast<int*>(sc + 2 * P); // [2][P]
  int* kP = kD + 2 * P; // [2][P]
  uint32_t* bm = reinterpret_cast<uint32_t*>(kP + 2 * P); // [2 frames][D, P][WB]
  int* pf = reinterpret_cast<int*>(bm + 4 * WB); // [D, P][WB]
  int* tg = pf + 2 * WB; // [P / 2 + 1]
  int* first = tg + P / 2 + 1; // [P]
  int* last = first + P; // [P]
  uint32_t* stage = reinterpret_cast<uint32_t*>(last + P); // [kAlignTraceRows][kAlignStageW]
  int* s_misc = reinterpret_cast<int*>(stage + kAlignTraceRows * kAlignStageW); // best node

  const int b = blockIdx.x;
  const int tid = threadIdx.x, nth = blockDim.x;
  const int lane = tid & 31, warp = tid >> 5;
  const int Tb = small[b], U = small[2 * B + b];
  const int32_t* tgt = small + 3 * B + small[B + b];
  const int L = 2 * U + 1;
  const float* e = emis + (long long)b * stride;

  // envelope: labels and blank in [0, C), the graph within the layout
  int bad = L > P || L > NPT * nth || (unsigned)blank >= (unsigned)C;
  if (L <= P)
    for (int u = tid; u < U; u += nth) {
      const int y = tgt[u];
      bad |= (unsigned)y >= (unsigned)C;
      tg[u] = y;
    }
  if (__syncthreads_or(bad)) {
    if (tid == 0) status[b] = 2;
    return;
  }
  auto lab = [&](int v) { return (v & 1) ? tg[v >> 1] : blank; };
  auto skip_from = [&](int u) { return (u & 1) && u + 2 < L && tg[(u + 1) >> 1] != tg[(u - 1) >> 1]; };

  // first / last frame each node is alive in (one thread: 2 L steps)
  if (tid == 0) {
    for (int v = 0; v < L; v++) { // fmin: arcs from node 0
      int f = v == 0 ? 0 : first[v - 1] + 1;
      if (v >= 3 && skip_from(v - 2)) f = min(f, first[v - 2] + 1);
      first[v] = f;
    }
    for (int v = L - 1; v >= 0; v--) { // dist: arcs to an accept node (L-1, L-2)
      int d = v >= L - 2 ? 0 : last[v + 1] + 1;
      if (v < L - 2 && skip_from(v)) d = min(d, last[v + 2] + 1);
      last[v] = d;
    }
    for (int v = 0; v < L; v++) last[v] = Tb - last[v];
  }
  for (int w = tid; w < 4 * WB; w += nth) bm[w] = 0u;
  for (int w = tid; w < 2 * WB; w += nth) pf[w] = 0;
  __syncthreads();

  // per owned node: label, alive window, out-list positions of its in-arcs, the next emission
  int lv[NPT], fv[NPT], lst[NPT], o0[NPT], o1[NPT], o2[NPT];
  bool sk[NPT];
  float ew[NPT];
#pragma unroll
  for (int k = 0; k < NPT; k++) {
    const int v = tid + k * nth;
    lv[k] = 0;
    fv[k] = 1;
    lst[k] = 0; // never alive
    o0[k] = 0;
    o1[k] = 1;
    o2[k] = 2;
    sk[k] = false;
    ew[k] = 0.0f;
    if (v < L) {
      const int y = lab(v);
      lv[k] = y;
      fv[k] = first[v];
      lst[k] = last[v];
      sk[k] = v >= 3 && skip_from(v - 2);
      if (arc_sorted) { // position in the stable label sort of the source's [self, step, skip] list
        o0[k] = (v + 1 < L && lab(v + 1) < y) + (skip_from(v) && lab(v + 2) < y);
        if (v >= 1) o1[k] = (lab(v - 1) <= y) + (skip_from(v - 1) && lab(v + 1) < y);
        if (sk[k]) o2[k] = (lab(v - 2) <= y) + (lab(v - 1) <= y);
      }
      if (Tb > 0) ew[k] = __ldg(&e[y]);
    }
    // frame 0: the start state alone (alive iff the target fits into T_b frames)
    if (v < P) {
      const bool start = v == 0 && fv[0] <= 0 && 0 <= lst[0];
      kD[v] = kP[v] = start ? 0 : kNoKey;
      sc[v] = 0.0f;
      if (start) bm[0] = bm[WB] = 1u;
    }
  }
  __syncthreads();

  uint8_t* mybp = bp + (long long)b * T_max * P;
  for (int t = 0; t < Tb; t++) {
    const int cur = t & 1, nxt = cur ^ 1;
    const float* scc = sc + cur * P;
    const int* kDc = kD + cur * P;
    const int* kPc = kP + cur * P;
    const uint32_t* bDc = bm + cur * 2 * WB;
    const uint32_t* bPc = bDc + WB;
    uint32_t* bDn = bm + nxt * 2 * WB;
    uint32_t* bPn = bDn + WB;
#pragma unroll
    for (int k = 0; k < NPT; k++) {
      const int v = tid + k * nth;
      if (v >= P) break;
      int kd = kNoKey, kp = -1;
      if (fv[k] <= t + 1 && t + 1 <= lst[k]) {
        const float w = __fadd_rn(0.0f, ew[k]);
        float best = -CUDART_INF_F;
        int br = 0x7fffffff, bd = 0;
#pragma unroll
        for (int d = 0; d < 3; d++) {
          const int u = v - d;
          if (d == 1 && v < 1) continue;
          if (d == 2 && !sk[k]) continue;
          const int ku = kPc[u];
          if (ku == kNoKey) continue; // (u, t) not alive
          const int o = d == 0 ? o0[k] : (d == 1 ? o1[k] : o2[k]);
          const int r = key_rank(bPc, pf + WB, ku) * 4 + o;
          kd = min(kd, key_rank(bDc, pf, kDc[u]) * 4 + o);
          kp = max(kp, r);
          const float c = __fadd_rn(scc[u], w);
          if (c > best || (c == best && r < br)) { // the first relaxation reaching the maximum
            best = c;
            br = r;
            bd = d;
          }
        }
        bad |= !(best > -CUDART_INF_F && best < CUDART_INF_F);
        sc[nxt * P + v] = best;
        mybp[(long long)t * P + v] = (uint8_t)bd;
        atomicOr(&bDn[kd >> 5], 1u << (kd & 31));
        atomicOr(&bPn[kp >> 5], 1u << (kp & 31));
      }
      kD[nxt * P + v] = kd;
      kP[nxt * P + v] = kd == kNoKey ? kNoKey : kp;
      if (t + 1 < Tb && v < L) ew[k] = __ldg(&e[(long long)(t + 1) * C + lv[k]]);
    }
    __syncthreads();
    // prefix popcounts of the new frame's bitmaps (warp 0: D, warp 1: P); the old frame's are cleared
    for (int w = tid; w < 2 * WB; w += nth) bm[cur * 2 * WB + w] = 0u;
    if (warp < 2) {
      const uint32_t* bmx = bm + nxt * 2 * WB + warp * WB;
      int* pfx = pf + warp * WB;
      int run = 0;
      for (int w0 = 0; w0 < WB; w0 += 32) {
        const int c = w0 + lane < WB ? __popc(bmx[w0 + lane]) : 0;
        int x = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int y = __shfl_up_sync(0xffffffffu, x, o);
          if (lane >= o) x += y;
        }
        if (w0 + lane < WB) pfx[w0 + lane] = run + x - c;
        run += __shfl_sync(0xffffffffu, x, 31);
      }
    }
    __syncthreads();
  }

  if (__syncthreads_or(bad)) {
    if (tid == 0) status[b] = 1;
    return;
  }
  // best accept node: the first strictly greatest in creation order (frame T_b)
  const int fin = Tb & 1;
  if (tid == 0) {
    int cand[2], posd[2], n = 0;
    for (int a = max(L - 2, 0); a < L; a++)
      if (kP[fin * P + a] != kNoKey) {
        cand[n] = a;
        posd[n++] = key_rank(bm + fin * 2 * WB, pf, kD[fin * P + a]);
      }
    if (n == 2 && posd[1] < posd[0]) {
      const int a = cand[0];
      cand[0] = cand[1];
      cand[1] = a;
    }
    float best = -CUDART_INF_F;
    int bn = -1;
    for (int i = 0; i < n; i++)
      if (sc[fin * P + cand[i]] > best) {
        best = sc[fin * P + cand[i]];
        bn = cand[i];
      }
    scores[b] = best;
    status[b] = 0;
    s_misc[0] = bn;
  }
  __syncthreads();
  const int bn = s_misc[0];
  int32_t* ol = labels + (long long)b * T_max;
  int32_t* os = states ? states + (long long)b * T_max : nullptr;
  for (int t = (bn < 0 ? 0 : Tb) + tid; t < T_max; t += nth) { // beyond T_b, or no accepting path
    ol[t] = -1;
    if (os) os[t] = -1;
  }
  if (bn < 0) return;

  // traceback: stage the rows' windows [v - 2R, v] with the whole CTA, walk them with one thread
  const uint32_t* bpw = reinterpret_cast<const uint32_t*>(mybp);
  const int PW = P / 4;
  for (int f = Tb; f > 0; f -= kAlignTraceRows) {
    const int R = min(kAlignTraceRows, f);
    const int vhi = s_misc[0];
    const int wlo = max(vhi - 2 * R, 0) >> 2, nw = (vhi >> 2) - wlo + 1;
    for (int i = tid; i < R * nw; i += nth) {
      const int r = i / nw, w = i - r * nw;
      stage[r * kAlignStageW + w] = __ldcg(bpw + (long long)(f - 1 - r) * PW + wlo + w);
    }
    __syncthreads();
    if (tid == 0) {
      int v = vhi;
      for (int r = 0; r < R; r++) {
        const int row = f - 1 - r;
        ol[row] = lab(v);
        if (os) os[row] = v;
        v -= (int)((stage[r * kAlignStageW + (v >> 2) - wlo] >> (8 * (v & 3))) & 0xffu);
      }
      s_misc[0] = v;
    }
    __syncthreads();
  }
}

} // namespace

#ifndef GTNB_HOST_EMU

size_t ctc_align_bp_pitch(int maxL) {
  return (size_t)align_pitch(maxL);
}

int launch_ctc_align(
    gtnb_ctx* ctx, int B, int T_max, int C, int blank, int arc_sorted, int maxL, const int32_t* small_dev,
    const float* emis, int64_t stride, uint8_t* bp, int32_t* labels, int32_t* states, float* scores,
    int32_t* status) {
  if (B == 0) return GTNB_OK;
  const int P = align_pitch(maxL);
  int threads, npt;
  align_layout(P, &threads, &npt);
  const size_t smem = align_smem_bytes(P);
#define LAUNCH_ALIGN(N_)                                                                                      \
  do {                                                                                                        \
    int rc__ = ensure_max_smem(ctx, (const void*)ctc_align_kernel<N_>);                                       \
    if (rc__) return rc__;                                                                                    \
    GTNB_LAUNCH(ctx, "ctc_align",                                                                             \
                ctc_align_kernel<N_><<<B, threads, smem, ctx->stream>>>(B, T_max, C, blank, arc_sorted, P,    \
                                                                       small_dev, emis, (long long)stride, bp, \
                                                                       labels, states, scores, status));     \
  } while (0)
  switch (npt) {
    case 1: LAUNCH_ALIGN(1); break;
    case 2: LAUNCH_ALIGN(2); break;
    case 4: LAUNCH_ALIGN(4); break;
    default: LAUNCH_ALIGN(8); break;
  }
#undef LAUNCH_ALIGN
  return GTNB_OK;
}

#endif // GTNB_HOST_EMU

} // namespace gtnb
