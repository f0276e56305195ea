// TEST HARNESS (not product): checks the fused qshmm pass 1 of the kernels (qshmm_chunk_pass1, run by k_qs_pass1)
// against the split statement the CPU harness runs and compares with the oracle (qshmm_quality_range, then
// qshmm_error_segment per segment), segment slot by segment slot and SegResult by SegResult, compiled as plain C++.
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <vector>

#include "../../include/pbsim_cuda.h"
#include "../../pbsim_b200/csrc/model_image.hpp"
#include "../../pbsim_b200/csrc/sim_core.cuh"

extern "C" {

// Every accuracy of the model that has a chain: n_reads reads of n_seg segments each, both passes, walked in chain
// chunks of `chunk` segments (0: one chunk per read).  del_floor > 0 raises every deletion threshold (T32 scale) to at
// least that value and lets insertions take the same share, so that positions with >= PB_QS_DEL_SAT deletions (the
// generic redo) and reads that start with insertions (the hp[-1] rule) are common.
// stats[0..3] = segments compared, segments redone generically, reads whose first entry is an insertion, mismatches.
// Returns the number of mismatching segments, < 0 on error.
long qs_pass1_compare(const pbsim_model *m, uint32_t seed, uint32_t n_reads, uint32_t n_seg, uint32_t chunk,
                      uint32_t del_floor, long *stats) {
  pb::ModelImage img;
  if (!img.build(*m)) { fprintf(stderr, "qs_pass1_check: %s\n", img.error.c_str()); return -1; }
  double bias[12];
  for (int h = 0; h < 12; ++h) bias[h] = 1.0;
  img.apply_bias(*m, bias);
  std::vector<pb::QsFast> fast(PBSIM_NQV);
  std::memcpy(fast.data(), img.qs_fast.data(), PBSIM_NQV * sizeof(pb::QsFast));
  if (del_floor) {
    for (pb::QsFast &f : fast) {
      if (f.del < del_floor) f.del = del_floor;
      const uint32_t ins = f.sub + (del_floor >> 2);
      if (ins > f.ins && ins > f.sub) f.ins = ins;
    }
  }
  pb::PhiloxKeys K;
  K.init(seed, 1u);
  for (int i = 0; i < 4; ++i) stats[i] = 0;
  const size_t n_slot = (size_t)n_seg * PB_SEG_STRIDE + 16;
  std::vector<uint16_t> ref(n_slot), got(n_slot);
  std::vector<pb::SegResult> ref_res(n_seg), got_res(n_seg);
  for (uint32_t a = 0; a < PBSIM_NACC; ++a) {
    const pb::AccEntry &ae = img.acc[a];
    if (!ae.valid || !ae.has_model) continue;
    pb::QsView T;
    const uint8_t *b = img.blob.data() + ae.blob_off;
    T.t2 = reinterpret_cast<const uint32_t *>(b + pb::QsBlobLayout::t2_off);
    T.emis = b + pb::QsBlobLayout::emis_off;
    T.freq = b;
    T.has_model = 1; T.init_mod = ae.init_mod; T.freq_mod = ae.freq_mod;
    T.thr = nullptr; T.thr_hp = nullptr; T.qc_prob = nullptr;
    T.thr32 = reinterpret_cast<const pb::QsThr *>(img.qs_thr32.data()); T.thr_hp32 = nullptr;
    T.fast = fast.data();
    pb::QsSegAux X;
    X.tmod = b + pb::QsBlobLayout::tmod_off;
    X.emodv = b + pb::QsBlobLayout::emodv_off;
    X.reach = ae.reach;
    const uint32_t per = chunk ? chunk : n_seg;
    for (uint32_t r = 0; r < n_reads; ++r) {
      const uint32_t read_id = a * 1000u + r + 1u;
      for (uint32_t pass = 0; pass < 2u; ++pass) {
        std::fill(ref.begin(), ref.end(), 0xEEEEu);
        std::fill(got.begin(), got.end(), 0xEEEEu);
        for (uint32_t k_from = 0; k_from < n_seg; k_from += per) {
          const uint32_t k_to = k_from + per < n_seg ? k_from + per : n_seg;
          uint32_t row = 0, mod = T.init_mod, emod = 1;
          if (k_from > 0)
            pb::qshmm_segment_start(T, X, K, read_id, pass, k_from * PB_TILE, ae.seg_ok ? ae.seg_ok : 512u, row, mod,
                                    emod);
          pb::qshmm_quality_range(T, K, read_id, pass, row, mod, emod, k_from, k_to, ref.data());
          for (uint32_t k = k_from; k < k_to; ++k)
            pb::qshmm_error_segment(T, K, read_id, pass, k * PB_TILE, k == 0, ref.data() + (size_t)k * PB_SEG_STRIDE,
                                    ref_res[k]);
          pb::qshmm_chunk_pass1(T, K, read_id, pass, row, mod, k_from, k_to, got.data(), got_res.data());
        }
        if (((ref[0] >> 7) & 3u) == PB_KIND_INS) ++stats[2];
        for (uint32_t k = 0; k < n_seg; ++k) {
          ++stats[0];
          if (ref_res[k].n_entries != PB_TILE) ++stats[1];
          const bool same = std::memcmp(&ref_res[k], &got_res[k], sizeof(pb::SegResult)) == 0 &&
                            std::memcmp(ref.data() + (size_t)k * PB_SEG_STRIDE, got.data() + (size_t)k * PB_SEG_STRIDE,
                                        PB_SEG_STRIDE * sizeof(uint16_t)) == 0;
          if (!same) {
            if (stats[3] < 5)
              fprintf(stderr, "qs_pass1_check: accuracy %u read %u pass %u segment %u differs\n", a, read_id, pass, k);
            ++stats[3];
          }
        }
      }
    }
  }
  return stats[3];
}

}  // extern "C"
