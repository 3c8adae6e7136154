// tc_plan.h — the host-side launch plan of the tensor-core batched scan (kernels_tc.cu).  Plain C++: the library
// decides with it whether a scan runs on the tensor cores (run_scan), which exchange format the multi-GPU flow uses
// (dist_layout) and how the scan is launched; the CPU tests check every plan it accepts.
#pragma once
#include <algorithm>
#include <cstdint>

namespace pirb {

constexpr int TC_MAX_ACC = 2;                    // accumulator buffers / epilogue groups (4 measured 7 % slower)
constexpr uint32_t TC_A_STAGE_BYTES = 128 * 128; // one A tile: 128 lanes x one 128-byte K chunk
constexpr uint32_t TC_SMEM_BUDGET = 227 * 1024;  // dynamic shared memory of one CTA
constexpr uint32_t TC_MAX_DIML = 32768;          // s32 accumulators: dimL * 255^2 < 2^31

struct TcPlan {
  uint32_t qt;      // queries per MMA tile (8, 16 or 24)
  uint32_t n_qt;    // query tiles per coefficient slot
  uint32_t n_cols;  // N of the MMA = qt * 2 * nb
  uint32_t Kp;      // dimL rounded up to a multiple of 16
  uint32_t kch;     // 128-byte K chunks; the B operand keeps all of them resident
  uint32_t b_bufs;  // shared-memory B buffers (2: the next query tile's B loads while this one computes)
  uint32_t stages;  // depth of the A-tile ring
  uint32_t smem;    // dynamic shared memory bytes
};

// Plan of a scan of n_queries queries over a last dimension of dimL entries with nb byte limbs per residue (5 or 6).
// requested_qt (PIRB_TC_QT, 16 when unset) is rounded down to a multiple of 8 and capped by the MMA's N <= 256; the
// plan takes the largest qt up to it whose B operand (all of K for one query tile) fits shared memory next to a ring
// of at least two A stages.  Returns false when not even qt = 8 fits (nb 5: dimL > 2048, nb 6: dimL > 1280): the
// caller then scans on the CUDA cores.  Whether some plan exists does not depend on requested_qt.
inline bool tc_plan(uint32_t nb, uint32_t dimL, uint32_t n_queries, int requested_qt, TcPlan* out) {
  if ((nb != 5 && nb != 6) || dimL == 0 || dimL > TC_MAX_DIML || n_queries == 0) return false;
  const uint32_t qpad = (n_queries + 7) / 8 * 8;
  const uint32_t qt_max = nb == 5 ? 24 : 16;  // qt * 2 * nb <= 256
  const uint32_t Kp = (dimL + 15) / 16 * 16;
  const uint32_t kch = (Kp + 127) / 128;
  const uint32_t e_bytes = TC_MAX_ACC * 16 * 128 * 8 * (nb <= 5 ? 1 : 2);  // epilogue exchange, [group][16 qp][128][EW]
  const uint32_t fixed = e_bytes + 1024;                                     // + barriers, TMEM slot, alignment slack
  uint32_t qt = std::min(std::min(qpad, qt_max), (uint32_t)std::max(8, requested_qt / 8 * 8));
  for (; qt >= 8; qt -= 8) {
    const uint32_t n_cols = qt * 2 * nb;
    const uint32_t b_buf = kch * n_cols * 128;
    const uint32_t b_bufs = (2 * b_buf + fixed + 4 * TC_A_STAGE_BYTES <= TC_SMEM_BUDGET) ? 2 : 1;
    if (b_bufs * b_buf + fixed + 2 * TC_A_STAGE_BYTES > TC_SMEM_BUDGET) continue;
    out->qt = qt;
    out->n_qt = (qpad + qt - 1) / qt;
    out->n_cols = n_cols;
    out->Kp = Kp;
    out->kch = kch;
    out->b_bufs = b_bufs;
    out->stages = std::min<uint32_t>(8, (TC_SMEM_BUDGET - fixed - b_bufs * b_buf) / TC_A_STAGE_BYTES);
    out->smem = out->stages * TC_A_STAGE_BYTES + b_bufs * b_buf + fixed;
    return true;
  }
  return false;
}

}  // namespace pirb
