// Data format shared by the two tensor-core engines (dp_tc2.cu, dp_tcx.cu): the tile shape and the fp16 weight-block and
// operand-block layouts (canonical K-major SWIZZLE_NONE UMMA operands), plus the configurations both engines serve.
// Engine-specific constants (row maps, ring depths, shared-memory and TMEM column maps) stay in the engines.
#pragma once
#include "dp_internal.h"

namespace dp {

// hid_dim = 96 with 4 heads on the 17-joint skeleton, coordinates at most 5 wide (uvxyz)
inline bool tc_supported(const Dims& d) {
  return d.hid == 96 && d.n_head == 4 && d.n_pts == 17 && d.c_in >= 1 && d.c_in <= 5 && d.c_out >= 1 && d.c_out <= 5;
}

namespace tc {

constexpr int NP = 17;
constexpr int TM = 128;              // tile rows = UMMA M
constexpr int TP = 7;                // poses per tile
constexpr int H = 96;
constexpr int WK = 112;              // weight block K extent: 96 weights + 16 (bias slab; k=96 hi, k=97 lo)
constexpr int W_LBO = 12 * 128;      // bytes between K-adjacent 8x8 core matrices of a weight block
constexpr int W_SBO = 128;           // bytes between N-adjacent core matrices
constexpr int WBLK_BYTES = (WK / 8) * W_LBO;        // 21504
constexpr int A_LBO = 16 * 128 + 16; // 2064: chunk column stride (+16 B skews consecutive chunk columns across banks)
constexpr int ABLK_BYTES = 12 * A_LBO;              // 24768
constexpr int ONES_BYTES = 2 * A_LBO;               // 4128
constexpr int BLOCKS_PER_LAYER = 14;                // weight blocks per layer: q, k, v, o, fc1 x2, fc2 x2, cheb1 x3, cheb2 x3
constexpr int TMEM_COLS = 512;

constexpr int al16(int x) { return (x + 15) / 16 * 16; }

}  // namespace tc
}  // namespace dp
