/*
 * tests/emu/align_emu.cpp -- TEST INFRASTRUCTURE: the SOURCE of gtn_b200/csrc/k_align.cu (CTC forced alignment
 * on the implicit lattice) on the CPU through tests/emu/simt_emu.h.
 */
#define GTNB_HOST_EMU 1
#include "../../gtn_b200/csrc/k_align.cu"

#include <vector>

extern "C" {

/* emissions [B][T][C], input_lens (nullable), targets concatenated, target_lens [B]; labels / states [B][T],
 * scores / status [B].  threads > 0 overrides the block size (nodes per thread follow from it). */
int emu_ctc_align(int B, int T, int C, const float* emissions, const int32_t* input_lens, const int32_t* targets,
                  const int32_t* target_lens, int blank, int arc_sorted, int threads, int32_t* labels,
                  int32_t* states, float* scores, int32_t* status) {
  using namespace gtnb;
  std::vector<int32_t> small(3 * (size_t)B);
  int tot = 0, maxL = 1;
  for (int b = 0; b < B; b++) {
    small[b] = input_lens ? input_lens[b] : T;
    small[B + b] = tot;
    small[2 * B + b] = target_lens[b];
    maxL = std::max(maxL, 2 * target_lens[b] + 1);
    tot += target_lens[b];
  }
  small.insert(small.end(), targets, targets + tot);
  const int P = align_pitch(maxL);
  int nth, npt;
  align_layout(P, &nth, &npt);
  if (threads > 0) {
    nth = threads;
    npt = 1;
    while (npt * nth < P) npt *= 2;
    if (npt > kAlignMaxNPT) return 1;
  }
  std::vector<uint8_t> bp((size_t)B * std::max(T, 1) * P, 0xee);
  const size_t smem = align_smem_bytes(P);
#define RUN(N_)                                                                                              \
  emu::launch(B, nth, smem, [&] {                                                                            \
    ctc_align_kernel<N_>(B, T, C, blank, arc_sorted, P, small.data(), emissions, (long long)T * C, bp.data(), \
                         labels, states, scores, status);                                                    \
  })
  switch (npt) {
    case 1: RUN(1); break;
    case 2: RUN(2); break;
    case 4: RUN(4); break;
    default: RUN(8); break;
  }
#undef RUN
  if (emu::g_launch_failed.exchange(false)) return emu::kEmuNoThreads; // the host refused the threads
  return 0;
}

} // extern "C"
