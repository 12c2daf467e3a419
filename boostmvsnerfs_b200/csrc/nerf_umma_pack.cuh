// Packed weights of the ENeRF per-sample MLP for the tcgen05 render kernel (render_multi_umma.cu):
// mlp_pack.pack_nerf_weights_umma writes this layout (CPU restatement of packing + dataflow: tests/test_umma_pack.py).
#pragma once

namespace bmv {

// ----------------------------------------------------------------------------------------- packed weights
// [hi block][lo block][fp32 vectors]; inside a block the matrices below, each as [K/8][N][8] fp16.
constexpr int UW_GS = 0;                       // global_fc [var16 | mean16] : N=32, K=32
constexpr int UW_GV = UW_GS + 32 * 32 * 2;     // global_fc per-view x       : N=32, K=16
constexpr int UW_FC = UW_GV + 32 * 16 * 2;     // agg.fc                     : N=16, K=32
constexpr int UW_L0 = UW_FC + 16 * 32 * 2;     // lr0 [pooled16 | vox8 | 0]  : N=64, K=32
constexpr int UW_CS = UW_L0 + 64 * 32 * 2;     // color.0 [hid64 | pooled16 | vox8 | 0] : N=64, K=96
constexpr int UW_CV = UW_CS + 64 * 96 * 2;     // color.0 per-view f_v       : N=64, K=16
constexpr int UW_BLOCK = UW_CV + 64 * 16 * 2;  // bytes per hi (or lo) block = 22528
// fp32 vectors (float offsets from the start of the vector area) — same order as the mma.sync packing
constexpr int UV_BG = 0, UV_WA = 32, UV_BFC = 64, UV_BL = 80, UV_WS = 144, UV_BC = 208, UV_W2 = 272, UV_WV = 336,
              UV_BV = 384, UV_SC = 396, UV_TAG = 400, UV_COUNT = 404;   // UV_TAG: 'UMMA' + 3 zero words (packing id)
constexpr int UMMA_PACK_BYTES = 2 * UW_BLOCK + UV_COUNT * 4;
constexpr int UMMA_PACK_WORDS = UMMA_PACK_BYTES / 4;

}  // namespace bmv
