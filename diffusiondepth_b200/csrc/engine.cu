// libddengine.so — C ABI (include/dd_engine.h) over the sm_100a kernels in conv_umma.cuh / kernels.cuh.
// Host side: weight pre-pack, workspace carving, TMA descriptor construction, per-step launch schedule
// (captured once into a CUDA graph), status polling.  No CPU compute path exists in this library.
#include <cuda.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include "../../include/dd_engine.h"
#include "kernels.cuh"
#include "convgen.cuh"
#include "conv_halo.cuh"
#include "conv_swap.cuh"
#include "swin.cuh"
#include "mpvit.cuh"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CUDA_TRY(expr)                                                                          \
  do {                                                                                          \
    cudaError_t _e = (expr);                                                                    \
    if (_e != cudaSuccess)                                                                      \
      return fail(DD_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));             \
  } while (0)

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;

int load_driver() {
  if (g_encode) return DD_OK;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult q;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
  if (e != cudaSuccess || fn == nullptr || q != cudaDriverEntryPointSuccess)
    return fail(DD_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
  g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  return DD_OK;
}

int absmax_grid(size_t n) {  // blocks of 256 threads, ~4 elements per thread, at most two per SM
  const size_t b = (n + 1023) / 1024;
  return static_cast<int>(b < 1 ? 1 : (b > 296 ? 296 : b));
}

CUtensorMapSwizzle swizzle_for(int bk) {
  return bk == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (bk == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
}

// activations: NHWC fp16 plane [B][H][W][C]; box = {bk, 16, 8, 1}
int make_act_map(CUtensorMap* m, const __half* base, int B, int H, int W, int C, int bk) {
  cuuint64_t gdim[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t gstr[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {(cuuint32_t)bk, dd::TILE_W, dd::TILE_H, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<__half*>(base), gdim, gstr, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(bk), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(DD_ERR_CUDA, "cuTensorMapEncodeTiled(activation) failed: " + std::to_string((int)r));
  return DD_OK;
}
// activations sampled with a spatial stride (stride-2 convs): elementStrides = {1, s, s, 1}; the box spans 16*s x 8*s
// input positions and still delivers 16 x 8 pixels
int make_act_map_strided(CUtensorMap* m, const __half* base, int B, int H, int W, int C, int bk, int stride) {
  cuuint64_t gdim[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t gstr[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {(cuuint32_t)bk, (cuuint32_t)(dd::TILE_W * stride), (cuuint32_t)(dd::TILE_H * stride), 1};
  cuuint32_t estr[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<__half*>(base), gdim, gstr, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(bk), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(DD_ERR_CUDA, "cuTensorMapEncodeTiled(strided activation) failed: " + std::to_string((int)r));
  return DD_OK;
}
// activation strip for the halo kernel: box = {bk, 8, 18, 1}
int make_strip_map(CUtensorMap* m, const __half* base, int B, int H, int W, int C, int bk) {
  cuuint64_t gdim[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t gstr[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {(cuuint32_t)bk, dd::HALO_TW, dd::HALO_TH + 2, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<__half*>(base), gdim, gstr, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(bk), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(DD_ERR_CUDA, "cuTensorMapEncodeTiled(strip) failed: " + std::to_string((int)r));
  return DD_OK;
}
// e4m3 activation strip (fp8-correction planes): [B][H][W][C] bytes, box = {64, 8, 18, 1}: 64-byte rows, 64-byte swizzle
int make_strip_map8(CUtensorMap* m, const uint8_t* base, int B, int H, int W, int C) {
  cuuint64_t gdim[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t gstr[3] = {(cuuint64_t)C, (cuuint64_t)W * C, (cuuint64_t)H * W * C};
  cuuint32_t box[4] = {64, dd::HALO_TW, dd::HALO_TH + 2, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, const_cast<uint8_t*>(base), gdim, gstr, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(DD_ERR_CUDA, "cuTensorMapEncodeTiled(e4m3 strip) failed: " + std::to_string((int)r));
  return DD_OK;
}
// e4m3 weights: [9][COUT][CIN] bytes; box = {64, rows, 1}, 64-byte swizzle
int make_w_map8(CUtensorMap* m, const uint8_t* base, int cout, int cin, int box_rows) {
  cuuint64_t gdim[3] = {(cuuint64_t)cin, (cuuint64_t)cout, 9};
  cuuint64_t gstr[2] = {(cuuint64_t)cin, (cuuint64_t)cout * cin};
  cuuint32_t box[3] = {64, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<uint8_t*>(base), gdim, gstr, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(DD_ERR_CUDA, "cuTensorMapEncodeTiled(e4m3 weight) failed: " + std::to_string((int)r));
  return DD_OK;
}
// 16x16 pixel patch for the swapped-operand kernel: box = {bk, 16, 16, 1}
int make_patch_map(CUtensorMap* m, const __half* base, int B, int H, int W, int C, int bk) {
  cuuint64_t gdim[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t gstr[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {(cuuint32_t)bk, dd::SWAP_TW, dd::SWAP_TH, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<__half*>(base), gdim, gstr, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(bk), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(DD_ERR_CUDA, "cuTensorMapEncodeTiled(patch) failed: " + std::to_string((int)r));
  return DD_OK;
}
// column-shifted strip for the row-halo variant of the swapped-operand kernel: box = {bk, 16, 18, 1}
int make_swap_strip_map(CUtensorMap* m, const __half* base, int B, int H, int W, int C, int bk) {
  cuuint64_t gdim[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t gstr[3] = {(cuuint64_t)C * 2, (cuuint64_t)W * C * 2, (cuuint64_t)H * W * C * 2};
  cuuint32_t box[4] = {(cuuint32_t)bk, dd::SWAP_TW, dd::SWAP_TH + 2, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<__half*>(base), gdim, gstr, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(bk), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(DD_ERR_CUDA, "cuTensorMapEncodeTiled(swap strip) failed: " + std::to_string((int)r));
  return DD_OK;
}
// weights: [9][COUT][CIN] fp16; box = {bk, COUT, 1}
int make_w_map(CUtensorMap* m, const __half* base, int cout, int cin, int bk, int box_rows = 0) {
  cuuint64_t gdim[3] = {(cuuint64_t)cin, (cuuint64_t)cout, 9};
  cuuint64_t gstr[2] = {(cuuint64_t)cin * 2, (cuuint64_t)cout * cin * 2};
  cuuint32_t box[3] = {(cuuint32_t)bk, (cuuint32_t)(box_rows ? box_rows : cout), 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<__half*>(base), gdim, gstr, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(bk), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(DD_ERR_CUDA, "cuTensorMapEncodeTiled(weight) failed: " + std::to_string((int)r));
  return DD_OK;
}

// general conv weights: [taps][COUT][CIN] fp16; box = {GEN_BK, NT, 1}
int make_wgen_map(CUtensorMap* m, const __half* base, int cout, int cin, int taps, int nt) {
  cuuint64_t gdim[3] = {(cuuint64_t)cin, (cuuint64_t)cout, (cuuint64_t)taps};
  cuuint64_t gstr[2] = {(cuuint64_t)cin * 2, (cuuint64_t)cout * cin * 2};
  cuuint32_t box[3] = {dd::GEN_BK, (cuuint32_t)nt, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<__half*>(base), gdim, gstr, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_for(dd::GEN_BK), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(DD_ERR_CUDA, "cuTensorMapEncodeTiled(gen weight) failed: " + std::to_string((int)r));
  return DD_OK;
}

// ---- conv shapes served by the engine
struct ShapeInfo {
  int cin, cout, bk;
};
constexpr ShapeInfo kShapes[5] = {{16, 64, 16}, {64, 256, 32}, {256, 256, 32}, {256, 64, 64}, {64, 16, 64}};
int shape_id(int cin, int cout) {
  for (int i = 0; i < 5; ++i)
    if (kShapes[i].cin == cin && kShapes[i].cout == cout) return i;
  return -1;
}

template <int CIN, int COUT, int BK, int EPI>
cudaError_t configure_umma() {
  using C = dd::ConvCfg<CIN, COUT, BK>;
  return cudaFuncSetAttribute(dd::conv3x3_umma_kernel<CIN, COUT, BK, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              C::SMEM_BYTES);
}
template <int CIN, int COUT, int BK>
cudaError_t configure_umma_all_epi() {
  cudaError_t e;
  if ((e = configure_umma<CIN, COUT, BK, dd::EPI_F32_STATS>()) != cudaSuccess) return e;
  if ((e = configure_umma<CIN, COUT, BK, dd::EPI_SPLIT>()) != cudaSuccess) return e;
  return configure_umma<CIN, COUT, BK, dd::EPI_F32>();
}
cudaError_t configure_all_kernels() {
  cudaError_t e;
  if ((e = cudaFuncSetAttribute(dd::window_attention_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                dd::WAU_SMEM)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(dd::decoder_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dd::DEC_SMEM)) != cudaSuccess)
    return e;
  if ((e = configure_umma_all_epi<16, 64, 16>()) != cudaSuccess) return e;
  if ((e = configure_umma_all_epi<64, 256, 32>()) != cudaSuccess) return e;
  if ((e = configure_umma_all_epi<256, 256, 32>()) != cudaSuccess) return e;
  if ((e = configure_umma_all_epi<256, 64, 64>()) != cudaSuccess) return e;
  if ((e = configure_umma_all_epi<64, 16, 64>()) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(dd::convgen_umma_kernel<256, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                dd::GenCfg<256, true>::SMEM_BYTES)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(dd::convgen_umma_kernel<192, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                dd::GenCfg<192, true>::SMEM_BYTES)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(dd::convgen_umma_kernel<128, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                dd::GenCfg<128, true>::SMEM_BYTES)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(dd::convgen_umma_kernel<64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                dd::GenCfg<64, true>::SMEM_BYTES)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(dd::convgen_umma_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                dd::GenCfg<256>::SMEM_BYTES)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(dd::convgen_umma_kernel<192>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                dd::GenCfg<192>::SMEM_BYTES)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(dd::convgen_umma_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                dd::GenCfg<128>::SMEM_BYTES)) != cudaSuccess) return e;
  return cudaFuncSetAttribute(dd::convgen_umma_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              dd::GenCfg<64>::SMEM_BYTES);
}

template <int CIN, int COUT, int BK, int EPI>
cudaError_t launch_umma(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& b_hi,
                        const CUtensorMap& b_lo, const dd::ConvArgs& args, int sm_count, cudaStream_t st) {
  using C = dd::ConvCfg<CIN, COUT, BK>;
  auto kern = dd::conv3x3_umma_kernel<CIN, COUT, BK, EPI>;  // smem attribute set in configure_all_kernels()
  int grid = args.num_tiles < sm_count ? args.num_tiles : sm_count;
  kern<<<grid, C::THREADS, C::SMEM_BYTES, st>>>(a_hi, a_lo, b_hi, b_lo, args);
  return cudaGetLastError();
}
constexpr int kHaloBK[5] = {16, 32, 32, 32, 32};  // K chunk of the halo kernel per shape id
constexpr int kSwapBK[5] = {16, 0, 0, 32, 32};    // K chunk of the swapped-operand kernel (narrow-N shapes only)
// Which kernel serves which shape inside the engine when the flags allow it (measured, profiles/README.md,
// tiny_probe.py): the swapped-operand kernel wins where MMA issue dominates (256->64: 356 vs 700 us; 64->16: 92 vs 129 us
// with the quarter-local epilogue); 16->64: halo kernel with the weights resident in shared memory and two epilogue warp
// sets, 82 us (classic 88, swap 182; its MMAs cost ~210 cycles each on 32-byte operand rows — padding K to 64-byte rows
// through TMA zero fill was slower still, 110-125 us); row-halo reuse pays for the wide layers.
constexpr bool kUseSwap[5] = {false, false, false, true, true};
constexpr bool kUseHalo[5] = {true, true, true, false, false};
// CTA pairs (cta_group::2, M = 256), measured (profiles/README.md, round 2 `ab_probe.py`, same box, 1 kW power cap):
// 64->256 with two epilogue warp sets 262 us vs 362 us single-CTA; 256->256 948 us / 1.29 M cycles vs 1119 us / 1.56 M
// cycles single-CTA (793 cycles per (chunk, tap) stage for 768 cycles of MMA work: the pair halves each SM's weight
// traffic through shared memory, and since the TMA producers issue from an elected lane of a whole warp the two CTAs'
// copies no longer trail the MMAs).  Round 1 had measured the 256->256 pair as equal: that was with lone-lane producers.
constexpr bool kUsePair[5] = {false, true, true, false, false};
template <int CIN, int COUT, int BK, int EPI, bool HALO = false>
cudaError_t launch_swap(const CUtensorMap& p_hi, const CUtensorMap& p_lo, const CUtensorMap& w, const dd::ConvArgs& args,
                        int sm_count, cudaStream_t st) {
  using C = dd::SwapCfg<CIN, COUT, BK, HALO>;
  int grid = args.num_tiles < sm_count ? args.num_tiles : sm_count;
  dd::conv3x3_swap_kernel<CIN, COUT, BK, EPI, HALO><<<grid, 256, C::SMEM_BYTES, st>>>(p_hi, p_lo, w, args);
  return cudaGetLastError();
}
template <int CIN, int COUT, int BK, bool HALO = false>
cudaError_t configure_swap() {
  using C = dd::SwapCfg<CIN, COUT, BK, HALO>;
  cudaError_t e = cudaFuncSetAttribute(dd::conv3x3_swap_kernel<CIN, COUT, BK, dd::EPI_F32_STATS, HALO>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(dd::conv3x3_swap_kernel<CIN, COUT, BK, dd::EPI_F32, HALO>,
                              cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES);
}
cudaError_t configure_swap_kernels() {
  cudaError_t e;
  if ((e = configure_swap<16, 64, 16>()) != cudaSuccess) return e;
  if ((e = configure_swap<256, 64, 32>()) != cudaSuccess) return e;
  if ((e = configure_swap<64, 16, 32>()) != cudaSuccess) return e;
  if ((e = configure_swap<256, 64, 32, true>()) != cudaSuccess) return e;
  return configure_swap<64, 16, 32, true>();
}
template <int CIN, int COUT, int BK, int EPI>
cudaError_t launch_halo(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& b_hi,
                        const CUtensorMap& b_lo, const dd::ConvArgs& args, int sm_count, cudaStream_t st) {
  using C = dd::HaloCfg<CIN, COUT, BK>;
  int grid = args.num_tiles < sm_count ? args.num_tiles : sm_count;
  dd::conv3x3_halo_kernel<CIN, COUT, BK, EPI><<<grid, C::THREADS, C::SMEM_BYTES, st>>>(a_hi, a_lo, b_hi, b_lo, a_lo, b_lo, args);
  return cudaGetLastError();
}
// CTA-pair variant (cluster of 2, tcgen05 cta_group::2) of the halo kernel for the 256-wide layers.  F8: fp8 correction
// products (a_lo / b_lo = the a8 / w8 maps, a_x / b_x = the l8 / lw8 maps).
template <int CIN, int COUT, int BK, int EPI, bool F8 = false>
cudaError_t launch_pair(const CUtensorMap& a_hi, const CUtensorMap& a_lo, const CUtensorMap& b_hi,
                        const CUtensorMap& b_lo, const dd::ConvArgs& args, int sm_count, cudaStream_t st,
                        const CUtensorMap* a_x = nullptr, const CUtensorMap* b_x = nullptr) {
  using C = dd::HaloCfg<CIN, COUT, BK, true, F8>;
  int grid = ((args.num_tiles + 1) & ~1) < (sm_count & ~1) ? ((args.num_tiles + 1) & ~1) : (sm_count & ~1);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(C::THREADS);
  cfg.dynamicSmemBytes = C::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, dd::conv3x3_halo_kernel<CIN, COUT, BK, EPI, true, F8>, a_hi, a_lo, b_hi, b_lo,
                            a_x ? *a_x : a_lo, b_x ? *b_x : b_lo, args);
}
template <int CIN, int COUT, int BK>
cudaError_t configure_pair_all_epi() {
  using C = dd::HaloCfg<CIN, COUT, BK, true>;
  cudaError_t e;
  if ((e = cudaFuncSetAttribute(dd::conv3x3_halo_kernel<CIN, COUT, BK, dd::EPI_F32_STATS, true>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(dd::conv3x3_halo_kernel<CIN, COUT, BK, dd::EPI_SPLIT, true>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES)) != cudaSuccess) return e;
  return cudaFuncSetAttribute(dd::conv3x3_halo_kernel<CIN, COUT, BK, dd::EPI_F32, true>,
                              cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES);
}
template <int CIN, int COUT, int BK>
cudaError_t configure_halo_all_epi() {
  using C = dd::HaloCfg<CIN, COUT, BK>;
  cudaError_t e;
  if ((e = cudaFuncSetAttribute(dd::conv3x3_halo_kernel<CIN, COUT, BK, dd::EPI_F32_STATS>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(dd::conv3x3_halo_kernel<CIN, COUT, BK, dd::EPI_SPLIT>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES)) != cudaSuccess) return e;
  return cudaFuncSetAttribute(dd::conv3x3_halo_kernel<CIN, COUT, BK, dd::EPI_F32>,
                              cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES);
}
cudaError_t configure_halo_kernels() {
  cudaError_t e;
  if ((e = cudaFuncSetAttribute(dd::conv3x3_halo_kernel<256, 256, 64, dd::EPI_SPLIT, true, true>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize,
                                dd::HaloCfg<256, 256, 64, true, true>::SMEM_BYTES)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(dd::conv3x3_halo_kernel<64, 256, 64, dd::EPI_F32_STATS, true, true>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize,
                                dd::HaloCfg<64, 256, 64, true, true>::SMEM_BYTES)) != cudaSuccess) return e;
  if ((e = cudaFuncSetAttribute(dd::conv3x3_halo_kernel<256, 256, 64, dd::EPI_F32, true, true>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize,
                                dd::HaloCfg<256, 256, 64, true, true>::SMEM_BYTES)) != cudaSuccess) return e;
  if ((e = configure_pair_all_epi<64, 256, 32>()) != cudaSuccess) return e;
  if ((e = configure_pair_all_epi<256, 256, 32>()) != cudaSuccess) return e;
  if ((e = configure_halo_all_epi<16, 64, 16>()) != cudaSuccess) return e;
  if ((e = configure_halo_all_epi<64, 256, 32>()) != cudaSuccess) return e;
  if ((e = configure_halo_all_epi<256, 256, 32>()) != cudaSuccess) return e;
  if ((e = configure_halo_all_epi<256, 64, 32>()) != cudaSuccess) return e;
  return configure_halo_all_epi<64, 16, 32>();
}

template <int CIN, int COUT, int EPI>
cudaError_t launch_simt(const dd::SimtArgs& a, cudaStream_t st) {
  constexpr int CO_T = COUT < 64 ? COUT : 64;
  dim3 grid(a.c.num_tiles, COUT / CO_T);
  dd::conv3x3_simt_kernel<CIN, COUT, EPI><<<grid, 256, 0, st>>>(a);
  return cudaGetLastError();
}

struct ConvLayer {
  int sid = -1;
  __half* w_hi = nullptr;
  __half* w_lo = nullptr;
  float* w_simt = nullptr;
  float* bias = nullptr;
  float wscale = 1.f;
  CUtensorMap mb_hi, mb_lo;
  CUtensorMap mh_hi, mh_lo;  // same planes, box for the halo kernel's K chunk
  CUtensorMap mp_hi, mp_lo;  // same, box of COUT/2 rows for the CTA-pair kernel (256-wide layers)
  __half* w_swap = nullptr;  // [9][128][CIN]: rows co = hi, 64+co = lo (swapped-operand kernel, narrow layers)
  CUtensorMap mw_swap;
  uint8_t *w8 = nullptr, *lw8 = nullptr;  // e4m3 correction planes [9][COUT][CIN] (DD_FLAG_FP8_CORR, the Cout = 256 layers)
  CUtensorMap m8_hi, m8_w, m8_lw;         // 64-channel boxes of COUT / 2 rows (fp16 hi plane, e4m3 planes): CTA-pair fp8 kernel
};

struct Raw {
  const float* ptr;
  std::vector<int64_t> shape;
};

// One producer convolution (neck / FPN): eval-BN folded into the weights (scale) and `shift`.
struct GenLayer {
  int cin = 0, cout = 0, taps = 1, nt = 256, relu = 1, shuffle = 0;
  int stride = 1, add_first = 0;
  __half* w_hi = nullptr;
  __half* w_lo = nullptr;
  float* shift = nullptr;
  float wscale = 1.f;
  CUtensorMap mb_hi, mb_lo;
  CUtensorMap mp_hi, mp_lo;  // box of nt / 2 rows: each CTA of a pair stages half of the N tile
  bool alt = false;          // cout divisible by 256 and 192: run_gen picks the width whose last wave wastes least
  CUtensorMap mb_hi_alt, mb_lo_alt, mp_hi_alt, mp_lo_alt;  // boxes of 192 / 96 rows
};
struct Planes {
  __half* hi = nullptr;
  __half* lo = nullptr;
};
struct Gemm {  // Linear layer on the tensor-core GEMM path: W [N][K] as fp16 hi/lo planes
  int K = 0, N = 0, nt = 256;
  __half* w_hi = nullptr;
  __half* w_lo = nullptr;
  float* bias = nullptr;  // [N] (zeros if the layer has none)
  float wscale = 1.f;
  CUtensorMap mb_hi, mb_lo;          // box {32, nt}
  bool alt = false;                  // N tiles by both 256 and 192: second pair of maps for the other width
  CUtensorMap mb_hi_alt, mb_lo_alt;  // box {32, 192}
  CUtensorMap mp_hi, mp_lo, mp_hi_alt, mp_lo_alt;  // the same with boxes of nt / 2 rows (CTA pairs)
};
struct SwinBlockW {
  float *ln1_g = nullptr, *ln1_b = nullptr, *ln2_g = nullptr, *ln2_b = nullptr, *table = nullptr;
  Gemm qkv, proj, ffn1, ffn2;
};
struct SwinStageW {
  std::vector<SwinBlockW> blocks;
  float *out_g = nullptr, *out_b = nullptr, *dn_g = nullptr, *dn_b = nullptr;
  Gemm reduction;
};
struct Backbone {
  bool enabled = false, ready = false;
  int E = 0, window = 7, H = 0, W = 0;
  int depths[4] = {0, 0, 0, 0}, heads[4] = {0, 0, 0, 0}, Hs[4] = {0, 0, 0, 0}, Ws[4] = {0, 0, 0, 0};
  float *pe_w = nullptr, *pe_b = nullptr, *pe_g = nullptr, *pe_beta = nullptr;
  SwinStageW stage[4];
  // workspace views
  float* X[2] = {nullptr, nullptr};
  float* QKV = nullptr;
  Planes AP, HP;
};
struct Producers {
  bool enabled = false, ready = false, neck = false;
  int nlev = 0;
  int C[4] = {0, 0, 0, 0}, H[4] = {0, 0, 0, 0}, W[4] = {0, 0, 0, 0};
  GenLayer lat[4], proj[4], fus[4], fl[4], fu[3];
  Planes F[4], L[4], P[4], O[4], XP[4];
  float* X[4] = {nullptr, nullptr, nullptr, nullptr};   // fp32 NHWC FPN outputs (X[0] aliases the loop's cond)
  float* UP[3] = {nullptr, nullptr, nullptr};           // fp32 NHWC upsampled maps at level i
  bool resample = false;                                // pyramid is not exactly 2x: adaptive_avg_pool2d is a real resample
  float* UPR[3] = {nullptr, nullptr, nullptr};          // raw ConvT output [B, 2H[i+1], 2W[i+1], 256] before pooling to level i
};
struct ResBlockW {
  GenLayer c1, c2, ds;
  bool has_ds = false;
};
struct ResNetW {
  bool enabled = false, ready = false;
  int H = 0, W = 0;
  int depths[4] = {0, 0, 0, 0}, C[4] = {64, 128, 256, 512}, Hs[4] = {0, 0, 0, 0}, Ws[4] = {0, 0, 0, 0};
  std::vector<ResBlockW> blocks[4];
  Planes IN, T, Yp[2];
  float* Y32[2] = {nullptr, nullptr};
  float* D32 = nullptr;
};

// MPViT (reference backbone/mpvit.py): depthwise layers as tap-major fp32 tables, every 1x1 conv / Linear on the GEMM path
struct DwLayer {
  int C = 0, K = 3;
  float* w = nullptr;     // [K*K][C], eval-BN scale folded in
  float* bias = nullptr;  // [C]
};
struct MpBlockW {
  float *ln1_g = nullptr, *ln1_b = nullptr, *ln2_g = nullptr, *ln2_b = nullptr;
  Gemm qkv, proj, fc1, fc2;
};
struct MpEncoderW {
  DwLayer cpe;              // ConvPosEnc, shared by the encoder's layers
  float* crpe_w = nullptr;  // [49][C]: the 3 / 5 / 7 windows of the head groups, centred in one 7 x 7 layout
  float* crpe_b = nullptr;
  std::vector<MpBlockW> layers;
};
struct MpStageW {
  DwLayer pe_dw[4], inv_dw;
  GenLayer pe_pw[4], inv1, inv2, agg;
  MpEncoderW enc[4];
};
struct MPViTW {
  bool enabled = false, ready = false;
  int H = 0, W = 0, heads = 8, mlp_ratio = 4;
  int dims[4] = {0, 0, 0, 0}, out_dims[4] = {0, 0, 0, 0}, layers[4] = {0, 0, 0, 0}, paths[4] = {0, 0, 0, 0};
  int Hs[4] = {0, 0, 0, 0}, Ws[4] = {0, 0, 0, 0};
  int radius[16] = {0};     // crpe window / 2 per head ({3: 2, 5: 3, 7: 3} heads)
  GenLayer stem0, stem1;
  MpStageW stage[4];
  // workspace views
  Planes IN, S1, D, EP0, AP, HP, CAT;
  float* XS = nullptr;      // stem output, then each stage's output (fp32 NHWC)
  float* E[4] = {nullptr, nullptr, nullptr, nullptr};  // the paths' token maps + one swap buffer
  float* R1 = nullptr;
  float* QKV = nullptr;
  float *part_m = nullptr, *part_s = nullptr, *colinv = nullptr, *part_ktv = nullptr, *ktv = nullptr;
};
constexpr int kMpChunksMax = 256;  // token chunks of the factorised attention's reductions

}  // namespace

struct dd_engine {
  dd_config cfg;
  int sm_count = 0;
  int up_qpb = 4;      // quads per block in gn_apply_up_split_kernel; DD_PROBES build: DD_UP_QPB=1 -> one 64-thread block per quad (A/B: equal)
  bool f8_ne3 = true;  // DD_PROBES build: DD_F8_NE3=0 keeps noise_embedding.3 on the 3-pass split (A/B timing)
  unsigned long long* clk_probe = nullptr;  // DD_CLK_PROBE=1: per-launch SM cycles / nanoseconds (dd_bench_conv)
  // tuning / timing probes: read from the environment ONCE in dd_create, and only in a -DDD_PROBES build
  // (profiles/README.md); a product build ignores the variables altogether
  int probe_fp8 = 0, swap_mask = -1, halo_mask = -1, pair_mask = -1;
  int genpair_mask = 1;  // DD_GENPAIR=0 (probes build): producer convs / GEMMs on single CTAs
  int swaphalo_mask = 1; // DD_SWAPHALO=0 (probes build): narrow layers on the plain swapped-operand kernel
  int attn_simt = 0;     // DD_ATTN_SIMT=1 (probes build): window attention on the fp32 CUDA-core kernel
  bool want_clk_probe = false;
  bool weights_ready = false;
  std::map<std::string, Raw> raw;
  // packed parameters (device memory owned by the engine)
  ConvLayer L[6];  // 0 ne.0, 1 ne.3, 2 convA, 3 convB, 4 pred.0, 5 pred.3
  float* gn_gamma[4] = {nullptr, nullptr, nullptr, nullptr};  // ne.1, ne.4, pred.1, pred.4
  float* gn_beta[4] = {nullptr, nullptr, nullptr, nullptr};
  float* temb = nullptr;    // [1280][256]
  float* dec_wt = nullptr;  // [4][4][16][16] folded
  float* dec_bt = nullptr;  // [16]
  float* dec_wc = nullptr;  // [9][16]
  float dec_bc = 0.f;
  float *enc_w1 = nullptr, *enc_b1 = nullptr, *enc_w2 = nullptr, *enc_b2 = nullptr;  // folded encoder (optional)
  std::vector<void*> owned;
  // schedule
  std::vector<int64_t> ts;
  std::vector<float> cx, ce;
  std::vector<float> sg;  // per-step sigma of stochastic DDIM (DD_FLAG_STOCHASTIC; zeros after dd_set_schedule)
  // workspace views
  void* ws = nullptr;
  float *x32 = nullptr, *Y = nullptr, *cond = nullptr, *stats[4] = {}, *mr[4] = {}, *temb_sel = nullptr;
  __half *xs_hi = nullptr, *xs_lo = nullptr, *S_hi[2] = {}, *S_lo[2] = {};
  int* status = nullptr;
  int stats_tiles_img[4] = {0, 0, 0, 0};  // tiles per image of the kernel that last filled stats[i]
  // graph
  Producers prod;
  Backbone bb;
  ResNetW rn;
  MPViTW mp;
  bool feats_ready = false;  // dd_run_backbone has filled the neck's input planes
  bool cond_ready = false;  // dd_build_condition has filled `cond` for the next dd_denoise_decode(cond = NULL)
  // CUDA graphs (DD_FLAG_CUDA_GRAPH), captured on first use and replayed: the T-step loop, the same loop with a decode
  // after every step (dd_denoise_decode_steps), the native backbone, the neck + FPN, and the stochastic loop
  // (dd_denoise_decode_stochastic) in its four shapes: G_STOCH + (decoded maps per step ? 1 : 0) + (latents per step ? 2 : 0)
  enum { G_LOOP = 0, G_LOOP_STEPS = 1, G_BACKBONE = 2, G_COND = 3, G_STOCH = 4, G_COUNT = 8 };
  cudaGraphExec_t graphs[G_COUNT] = {};
  int64_t graph_launches[G_COUNT] = {};  // kernel nodes per graph (added to `launches` per replay)
  cudaStream_t cap_stream = nullptr;  // capture happens here (the caller's stream may be the legacy default stream)
  float* rgb_stage = nullptr;         // workspace copy of the image batch the backbone graph reads
  float* inter = nullptr;             // [T][B][2h][2w] per-step decoded depth (DD_FLAG_STEP_DECODE)
  float* step_noise = nullptr;        // [T][B][P][16] staged per-step noise z (DD_FLAG_STOCHASTIC)
  float* lat_steps = nullptr;         // [T][B][16][P] NCHW latent after every step (DD_FLAG_STOCHASTIC)
  int64_t launches = 0;
  int* status_host = nullptr;  // pinned
};

namespace {

constexpr float kActScale = 16.f;  // power-of-two pre-scale of conv inputs before the fp16 split
constexpr float kXScale = 1.f;     // the raw latent keeps scale 1 (random-init trajectories reach |x| ~ 5e2)

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct Carver {
  uint8_t* base;
  size_t off = 0;
  template <typename T>
  T* take(size_t n) {
    off = align_up(off, 1024);
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += n * sizeof(T);
    return p;
  }
};

struct Geom {
  int B, h, w, P, tiles_x, tiles_y, tiles_img, tiles;  // tiles of the conv kernel selected by cfg.flags
  int tiles_max;                                       // max over both tilings (buffer sizing)
};
Geom geom_of(const dd_config& c) {
  Geom g;
  g.B = c.batch;
  g.h = c.latent_h;
  g.w = c.latent_w;
  g.P = g.h * g.w;
  const int t816 = ((g.w + dd::TILE_W - 1) / dd::TILE_W) * ((g.h + dd::TILE_H - 1) / dd::TILE_H);
  const int t168 = ((g.w + dd::HALO_TW - 1) / dd::HALO_TW) * ((g.h + dd::HALO_TH - 1) / dd::HALO_TH);
  g.tiles_x = (g.w + dd::TILE_W - 1) / dd::TILE_W;
  g.tiles_y = (g.h + dd::TILE_H - 1) / dd::TILE_H;
  g.tiles_img = g.tiles_x * g.tiles_y;
  g.tiles = g.tiles_img * g.B;
  g.tiles_max = (t816 > t168 ? t816 : t168) * g.B;
  return g;
}

void drop_graphs(dd_engine* e) {
  for (int i = 0; i < dd_engine::G_COUNT; ++i)
    if (e->graphs[i]) {
      cudaGraphExecDestroy(e->graphs[i]);
      e->graphs[i] = nullptr;
    }
}

// Capture `body(stream)` into graph slot `which` on first use, then replay it on `st`.  Every pointer the body's kernels
// take must live in the workspace or in engine-owned memory (caller buffers are staged in / copied out around the graph).
template <typename F>
int graph_run(dd_engine* e, int which, cudaStream_t st, F&& body) {
  if (!e->graphs[which]) {
    cudaGraph_t graph = nullptr;
    const int64_t before = e->launches;
    CUDA_TRY(cudaStreamBeginCapture(e->cap_stream, cudaStreamCaptureModeThreadLocal));
    const int rc = body(e->cap_stream);
    const cudaError_t ce = cudaStreamEndCapture(e->cap_stream, &graph);
    e->graph_launches[which] = e->launches - before;
    e->launches = before;
    if (rc != DD_OK) {
      if (graph) cudaGraphDestroy(graph);
      return rc;
    }
    if (ce != cudaSuccess) return fail(DD_ERR_CUDA, std::string("graph capture: ") + cudaGetErrorString(ce));
    const cudaError_t ci = cudaGraphInstantiate(&e->graphs[which], graph, 0);
    cudaGraphDestroy(graph);
    if (ci != cudaSuccess) return fail(DD_ERR_CUDA, std::string("graph instantiate: ") + cudaGetErrorString(ci));
  }
  CUDA_TRY(cudaGraphLaunch(e->graphs[which], st));
  e->launches += e->graph_launches[which];
  return DD_OK;
}

// Lay the workspace out.  With base == nullptr only the size is computed (the engine's views are untouched).
size_t carve(dd_engine* e, void* base) {
  const Geom g = geom_of(e->cfg);
  const size_t BP = static_cast<size_t>(g.B) * g.P;
  Carver c{reinterpret_cast<uint8_t*>(base)};
  dd_engine tmp_views;  // scratch target when only sizing
  dd_engine* v = base ? e : &tmp_views;
  v->status = c.take<int>(16);
  v->x32 = c.take<float>(BP * 16);
  v->xs_hi = c.take<__half>(BP * 16);
  v->xs_lo = c.take<__half>(BP * 16);
  v->Y = c.take<float>(BP * 256);
  for (int i = 0; i < 2; ++i) {
    v->S_hi[i] = c.take<__half>(BP * 256);
    v->S_lo[i] = c.take<__half>(BP * 256);
  }
  v->cond = c.take<float>(static_cast<size_t>(g.B) * e->cfg.cond_h * e->cfg.cond_w * 256);
  for (int i = 0; i < 4; ++i) {
    v->stats[i] = c.take<float>(static_cast<size_t>(g.tiles_max) * 8);
    v->mr[i] = c.take<float>(static_cast<size_t>(g.B) * 8);
  }
  v->temb_sel = c.take<float>(static_cast<size_t>(g.B) * 256);
  if (e->cfg.flags & DD_FLAG_STEP_DECODE)
    v->inter = c.take<float>(static_cast<size_t>(e->cfg.num_inference_steps) * BP * 4);
  if (e->cfg.flags & DD_FLAG_STOCHASTIC) {
    v->step_noise = c.take<float>(static_cast<size_t>(e->cfg.num_inference_steps) * BP * 16);
    v->lat_steps = c.take<float>(static_cast<size_t>(e->cfg.num_inference_steps) * BP * 16);
  }
  if (e->rn.enabled || e->bb.enabled || e->mp.enabled)
    v->rgb_stage = c.take<float>(static_cast<size_t>(g.B) * 3 *
                                 (e->rn.enabled ? e->rn.H * e->rn.W : (e->mp.enabled ? e->mp.H * e->mp.W : e->bb.H * e->bb.W)));
  if (e->prod.enabled) {
    const Producers& pc = e->prod;
    Producers* pv = &v->prod;
    for (int i = 0; i < pc.nlev; ++i) {
      const size_t px = static_cast<size_t>(g.B) * pc.H[i] * pc.W[i];
      auto planes = [&](Planes& pl, size_t ch) {
        pl.hi = c.take<__half>(px * ch);
        pl.lo = c.take<__half>(px * ch);
      };
      planes(pv->F[i], pc.C[i]);
      if (pc.neck) {
        planes(pv->L[i], pc.C[i]);
        planes(pv->P[i], 512);
        planes(pv->O[i], pc.C[i]);
      }
      planes(pv->XP[i], 256);
      pv->X[i] = (i == 0) ? v->cond : c.take<float>(px * 256);
      if (i < pc.nlev - 1) {
        pv->UP[i] = c.take<float>(px * 256);
        if (pc.resample) pv->UPR[i] = c.take<float>(static_cast<size_t>(g.B) * 4 * pc.H[i + 1] * pc.W[i + 1] * 256);
      }
    }
  }
  if (e->rn.enabled) {
    const ResNetW& rc = e->rn;
    ResNetW* rv = &v->rn;
    const size_t pin = static_cast<size_t>(g.B) * rc.H * rc.W;
    const size_t p0 = static_cast<size_t>(g.B) * rc.Hs[0] * rc.Ws[0] * 64;  // largest stage tensor (elements)
    rv->IN.hi = c.take<__half>(pin * dd::GEN_BK);
    rv->IN.lo = c.take<__half>(pin * dd::GEN_BK);
    rv->T.hi = c.take<__half>(p0);
    rv->T.lo = c.take<__half>(p0);
    for (int k = 0; k < 2; ++k) {
      rv->Yp[k].hi = c.take<__half>(p0);
      rv->Yp[k].lo = c.take<__half>(p0);
      rv->Y32[k] = c.take<float>(p0);
    }
    rv->D32 = c.take<float>(p0);
  }
  if (e->bb.enabled) {
    const Backbone& bc = e->bb;
    Backbone* bv = &v->bb;
    const size_t m0 = (static_cast<size_t>(g.B) * bc.Hs[0] * bc.Ws[0] + 127) / 128 * 128 + 128;  // padded token count
    const size_t c0 = bc.E;
    bv->X[0] = c.take<float>(m0 * c0);
    bv->X[1] = c.take<float>(m0 * c0);
    bv->QKV = c.take<float>(m0 * c0 * 3);
    bv->AP.hi = c.take<__half>(m0 * c0);
    bv->AP.lo = c.take<__half>(m0 * c0);
    bv->HP.hi = c.take<__half>(m0 * c0 * 4);
    bv->HP.lo = c.take<__half>(m0 * c0 * 4);
  }
  if (e->mp.enabled) {
    const MPViTW& mc = e->mp;
    MPViTW* mv = &v->mp;
    const size_t pin = static_cast<size_t>(g.B) * mc.H * mc.W;
    size_t tok = 0, cat = 0, xs = pin * mc.dims[0];
    int cmax = 0;
    for (int s = 0; s < 4; ++s) {
      const size_t M = static_cast<size_t>(g.B) * mc.Hs[s] * mc.Ws[s] + 256;  // slack: the GEMM's token "image" is 16 wide
      tok = std::max(tok, M * mc.dims[s]);
      cat = std::max(cat, M * mc.dims[s] * (mc.paths[s] + 1));
      xs = std::max(xs, M * mc.out_dims[s]);
      cmax = std::max(cmax, mc.dims[s]);
    }
    auto planes = [&](Planes& pl, size_t n) {
      pl.hi = c.take<__half>(n);
      pl.lo = c.take<__half>(n);
    };
    planes(mv->IN, pin * dd::GEN_BK);
    planes(mv->S1, pin * (mc.dims[0] / 2));
    mv->XS = c.take<float>(xs);
    for (int i = 0; i < 4; ++i) mv->E[i] = c.take<float>(tok);
    mv->R1 = c.take<float>(tok);
    mv->QKV = c.take<float>(tok * 3);
    planes(mv->D, tok);
    planes(mv->EP0, tok);
    planes(mv->AP, tok);
    planes(mv->HP, tok * mc.mlp_ratio);
    planes(mv->CAT, cat);
    const size_t chm = static_cast<size_t>(cmax / mc.heads), nk = static_cast<size_t>(mc.heads) * chm * chm;
    mv->part_m = c.take<float>(static_cast<size_t>(g.B) * kMpChunksMax * cmax);
    mv->part_s = c.take<float>(static_cast<size_t>(g.B) * kMpChunksMax * cmax);
    mv->colinv = c.take<float>(static_cast<size_t>(g.B) * cmax);
    mv->part_ktv = c.take<float>(static_cast<size_t>(g.B) * kMpChunksMax * nk);
    mv->ktv = c.take<float>(static_cast<size_t>(g.B) * nk);
  }
  return align_up(c.off, 1024);
}

// One convolution on the engine's latent grid.  in planes have `cin` channels (scale in_scale).
// f8 bit 0: the INPUT planes are hi / a8 / l8 (in_lo = base of the e4m3 pair: a8, then l8 B*P*cin bytes further) and the
// conv runs with fp8 correction products; bit 1: the OUTPUT planes are written as hi / a8 / l8 (out_lo = their base).
constexpr int kF8In = 1, kF8Out = 2;
bool fp8_active(const dd_engine* e) {  // the wide convs of the Swin variant, on the CTA-pair halo kernel only
  const int need = DD_FLAG_FP8_CORR | DD_FLAG_HALO_CONV | DD_FLAG_PAIR_WIDE;
  return (e->cfg.flags & need) == need && !(e->cfg.flags & DD_FLAG_SIMT_CONV) && e->cfg.variant == DD_VARIANT_SWIN &&
         e->pair_mask < 0 && e->halo_mask < 0;
}
int run_conv(dd_engine* e, int layer, const __half* in_hi, const __half* in_lo, float in_scale, int epi, float* y32,
             float* stats_partial, __half* out_hi, __half* out_lo, cudaStream_t st, int f8 = 0) {
  const Geom g = geom_of(e->cfg);
  ConvLayer& L = e->L[layer];
  const ShapeInfo s = kShapes[L.sid];
  dd::ConvArgs a;
  a.B = g.B;
  a.H = g.h;
  a.W = g.w;
  a.tiles_x = g.tiles_x;
  a.tiles_y = g.tiles_y;
  a.num_tiles = g.tiles;
  a.bias = L.bias;
  a.acc_scale = 1.f / (in_scale * L.wscale);
  a.y32 = y32;
  a.stats_partial = stats_partial;
  a.out_hi = out_hi;
  a.out_lo = out_lo;
  a.out_a8 = a.out_l8 = nullptr;
  if (f8 & kF8Out) {
    a.out_a8 = reinterpret_cast<uint8_t*>(out_lo);
    a.out_l8 = a.out_a8 + static_cast<size_t>(g.B) * g.P * kShapes[e->L[layer].sid].cout;
  }
  a.split_scale = kActScale;
  a.status = e->status;
  a.fp8_probe = e->probe_fp8;
  a.clk_probe = e->clk_probe;
  cudaError_t err = cudaSuccess;
  e->launches++;
  int which = -1;
  for (int i = 0; i < 4; ++i)
    if (stats_partial == e->stats[i]) which = i;
  if (which >= 0) e->stats_tiles_img[which] = g.tiles_img;
  const bool swap_here = e->swap_mask >= 0 ? ((e->swap_mask >> L.sid) & 1) : kUseSwap[L.sid];
  const bool use_swap = (e->cfg.flags & DD_FLAG_SWAP_NARROW) && !(e->cfg.flags & DD_FLAG_SIMT_CONV) &&
                        swap_here && kSwapBK[L.sid] > 0 && epi != dd::EPI_SPLIT;
  const bool halo_here = e->halo_mask >= 0 ? ((e->halo_mask >> L.sid) & 1) : kUseHalo[L.sid];
  const bool use_halo = (e->cfg.flags & DD_FLAG_HALO_CONV) && !(e->cfg.flags & DD_FLAG_SIMT_CONV) && halo_here;
  if (!use_swap) {  // tile geometry of the kernel actually launched
    const int tw = use_halo ? dd::HALO_TW : dd::TILE_W, th = use_halo ? dd::HALO_TH : dd::TILE_H;
    a.tiles_x = (g.w + tw - 1) / tw;
    a.tiles_y = (g.h + th - 1) / th;
    a.num_tiles = a.tiles_x * a.tiles_y * g.B;
    if (which >= 0) e->stats_tiles_img[which] = a.tiles_x * a.tiles_y;
  }
  if (f8 && !use_halo) return fail(DD_ERR_INVALID, "fp8-correction planes need the row-halo CTA-pair kernel");
  if (use_swap) {
    a.tiles_x = (g.w + dd::SWAP_TW - 1) / dd::SWAP_TW;
    a.tiles_y = (g.h + dd::SWAP_TH - 1) / dd::SWAP_TH;
    a.num_tiles = a.tiles_x * a.tiles_y * g.B;
    if (which >= 0) e->stats_tiles_img[which] = a.tiles_x * a.tiles_y;
    CUtensorMap mp_hi, mp_lo;
    int rc;
    const int bk = kSwapBK[L.sid];
    // row-halo variant (three column-shifted strips per chunk instead of nine shifted patches) for the 32-channel-chunk
    // layers when the engine runs the halo kernels at all
    const bool swap_halo = (e->cfg.flags & DD_FLAG_HALO_CONV) && bk == 32 && e->swaphalo_mask != 0;
    if (swap_halo) {
      if ((rc = make_swap_strip_map(&mp_hi, in_hi, g.B, g.h, g.w, s.cin, bk))) return rc;
      if ((rc = make_swap_strip_map(&mp_lo, in_lo, g.B, g.h, g.w, s.cin, bk))) return rc;
    } else {
      if ((rc = make_patch_map(&mp_hi, in_hi, g.B, g.h, g.w, s.cin, bk))) return rc;
      if ((rc = make_patch_map(&mp_lo, in_lo, g.B, g.h, g.w, s.cin, bk))) return rc;
    }
    const bool st_ = (epi == dd::EPI_F32_STATS);
    if (swap_halo) {
      switch (L.sid) {
        case 3: err = st_ ? launch_swap<256, 64, 32, dd::EPI_F32_STATS, true>(mp_hi, mp_lo, L.mw_swap, a, e->sm_count, st)
                          : launch_swap<256, 64, 32, dd::EPI_F32, true>(mp_hi, mp_lo, L.mw_swap, a, e->sm_count, st); break;
        case 4: err = st_ ? launch_swap<64, 16, 32, dd::EPI_F32_STATS, true>(mp_hi, mp_lo, L.mw_swap, a, e->sm_count, st)
                          : launch_swap<64, 16, 32, dd::EPI_F32, true>(mp_hi, mp_lo, L.mw_swap, a, e->sm_count, st); break;
      }
    } else
    switch (L.sid) {
      case 0: err = st_ ? launch_swap<16, 64, 16, dd::EPI_F32_STATS>(mp_hi, mp_lo, L.mw_swap, a, e->sm_count, st)
                        : launch_swap<16, 64, 16, dd::EPI_F32>(mp_hi, mp_lo, L.mw_swap, a, e->sm_count, st); break;
      case 3: err = st_ ? launch_swap<256, 64, 32, dd::EPI_F32_STATS>(mp_hi, mp_lo, L.mw_swap, a, e->sm_count, st)
                        : launch_swap<256, 64, 32, dd::EPI_F32>(mp_hi, mp_lo, L.mw_swap, a, e->sm_count, st); break;
      case 4: err = st_ ? launch_swap<64, 16, 32, dd::EPI_F32_STATS>(mp_hi, mp_lo, L.mw_swap, a, e->sm_count, st)
                        : launch_swap<64, 16, 32, dd::EPI_F32>(mp_hi, mp_lo, L.mw_swap, a, e->sm_count, st); break;
    }
  } else if (e->cfg.flags & DD_FLAG_SIMT_CONV) {
    dd::SimtArgs sa;
    sa.in_hi = in_hi;
    sa.in_lo = in_lo;
    sa.in_inv_scale = 1.f / in_scale;
    sa.w = L.w_simt;
    sa.c = a;
#define SIMT_CASE(ID, CI, CO)                                                           \
  case ID:                                                                              \
    err = (epi == dd::EPI_F32_STATS) ? launch_simt<CI, CO, dd::EPI_F32_STATS>(sa, st)   \
          : (epi == dd::EPI_SPLIT)   ? launch_simt<CI, CO, dd::EPI_SPLIT>(sa, st)       \
                                     : launch_simt<CI, CO, dd::EPI_F32>(sa, st);        \
    break;
    switch (L.sid) {
      SIMT_CASE(0, 16, 64)
      SIMT_CASE(1, 64, 256)
      SIMT_CASE(2, 256, 256)
      SIMT_CASE(3, 256, 64)
      SIMT_CASE(4, 64, 16)
    }
#undef SIMT_CASE
  } else if (use_halo) {
    CUtensorMap ma_hi, ma_lo;
    int rc;
    const int hbk = kHaloBK[L.sid];
    if ((rc = make_strip_map(&ma_hi, in_hi, g.B, g.h, g.w, s.cin, hbk))) return rc;
    if (!(f8 & kF8In))
      if ((rc = make_strip_map(&ma_lo, in_lo, g.B, g.h, g.w, s.cin, hbk))) return rc;
    const bool use_pair = (e->cfg.flags & DD_FLAG_PAIR_WIDE) &&
                          (e->pair_mask >= 0 ? ((e->pair_mask >> L.sid) & 1) && s.cout == 256 : kUsePair[L.sid]);
    if ((f8 & kF8In) && !(use_pair && L.w8 && ((L.sid == 2 && epi != dd::EPI_F32_STATS) || (L.sid == 1 && epi == dd::EPI_F32_STATS))))
      return fail(DD_ERR_INVALID, "fp8-correction planes fed to a layer / kernel that does not take them");
    if ((f8 & kF8Out) && epi != dd::EPI_SPLIT) return fail(DD_ERR_INVALID, "fp8 output planes need the split epilogue");
    if (f8 & kF8In) {
      const uint8_t* a8 = reinterpret_cast<const uint8_t*>(in_lo);
      CUtensorMap m_hi64, m_a8, m_l8;
      if ((rc = make_strip_map(&m_hi64, in_hi, g.B, g.h, g.w, s.cin, 64))) return rc;
      if ((rc = make_strip_map8(&m_a8, a8, g.B, g.h, g.w, s.cin))) return rc;
      if ((rc = make_strip_map8(&m_l8, a8 + static_cast<size_t>(g.B) * g.P * s.cin, g.B, g.h, g.w, s.cin))) return rc;
      err = (L.sid == 1)
                ? launch_pair<64, 256, 64, dd::EPI_F32_STATS, true>(m_hi64, m_a8, L.m8_hi, L.m8_w, a, e->sm_count, st, &m_l8, &L.m8_lw)
            : (epi == dd::EPI_SPLIT)
                ? launch_pair<256, 256, 64, dd::EPI_SPLIT, true>(m_hi64, m_a8, L.m8_hi, L.m8_w, a, e->sm_count, st, &m_l8, &L.m8_lw)
                : launch_pair<256, 256, 64, dd::EPI_F32, true>(m_hi64, m_a8, L.m8_hi, L.m8_w, a, e->sm_count, st, &m_l8, &L.m8_lw);
    } else if (use_pair) {
#define PAIR_CASE(ID, CI, CO, BK)                                                                                   \
  case ID:                                                                                                          \
    err = (epi == dd::EPI_F32_STATS)                                                                                \
              ? launch_pair<CI, CO, BK, dd::EPI_F32_STATS>(ma_hi, ma_lo, L.mp_hi, L.mp_lo, a, e->sm_count, st)      \
          : (epi == dd::EPI_SPLIT)                                                                                  \
              ? launch_pair<CI, CO, BK, dd::EPI_SPLIT>(ma_hi, ma_lo, L.mp_hi, L.mp_lo, a, e->sm_count, st)          \
              : launch_pair<CI, CO, BK, dd::EPI_F32>(ma_hi, ma_lo, L.mp_hi, L.mp_lo, a, e->sm_count, st);           \
    break;
      switch (L.sid) {
        PAIR_CASE(1, 64, 256, 32)
        PAIR_CASE(2, 256, 256, 32)
      }
#undef PAIR_CASE
    } else {
#define HALO_CASE(ID, CI, CO, BK)                                                                                   \
  case ID:                                                                                                          \
    err = (epi == dd::EPI_F32_STATS)                                                                                \
              ? launch_halo<CI, CO, BK, dd::EPI_F32_STATS>(ma_hi, ma_lo, L.mh_hi, L.mh_lo, a, e->sm_count, st)      \
          : (epi == dd::EPI_SPLIT)                                                                                  \
              ? launch_halo<CI, CO, BK, dd::EPI_SPLIT>(ma_hi, ma_lo, L.mh_hi, L.mh_lo, a, e->sm_count, st)          \
              : launch_halo<CI, CO, BK, dd::EPI_F32>(ma_hi, ma_lo, L.mh_hi, L.mh_lo, a, e->sm_count, st);           \
    break;
    switch (L.sid) {
      HALO_CASE(0, 16, 64, 16)
      HALO_CASE(1, 64, 256, 32)
      HALO_CASE(2, 256, 256, 32)
      HALO_CASE(3, 256, 64, 32)
      HALO_CASE(4, 64, 16, 32)
    }
#undef HALO_CASE
    }
  } else {
    CUtensorMap ma_hi, ma_lo;
    int rc;
    if ((rc = make_act_map(&ma_hi, in_hi, g.B, g.h, g.w, s.cin, s.bk))) return rc;
    if ((rc = make_act_map(&ma_lo, in_lo, g.B, g.h, g.w, s.cin, s.bk))) return rc;
#define UMMA_CASE(ID, CI, CO, BK)                                                                                   \
  case ID:                                                                                                          \
    err = (epi == dd::EPI_F32_STATS)                                                                                \
              ? launch_umma<CI, CO, BK, dd::EPI_F32_STATS>(ma_hi, ma_lo, L.mb_hi, L.mb_lo, a, e->sm_count, st)      \
          : (epi == dd::EPI_SPLIT)                                                                                  \
              ? launch_umma<CI, CO, BK, dd::EPI_SPLIT>(ma_hi, ma_lo, L.mb_hi, L.mb_lo, a, e->sm_count, st)          \
              : launch_umma<CI, CO, BK, dd::EPI_F32>(ma_hi, ma_lo, L.mb_hi, L.mb_lo, a, e->sm_count, st);           \
    break;
    switch (L.sid) {
      UMMA_CASE(0, 16, 64, 16)
      UMMA_CASE(1, 64, 256, 32)
      UMMA_CASE(2, 256, 256, 32)
      UMMA_CASE(3, 256, 64, 64)
      UMMA_CASE(4, 64, 16, 64)
    }
#undef UMMA_CASE
  }
  if (err != cudaSuccess) return fail(DD_ERR_CUDA, std::string("conv launch: ") + cudaGetErrorString(err));
  return DD_OK;
}

int run_finalize(dd_engine* e, int which, int channels, cudaStream_t st) {
  const Geom g = geom_of(e->cfg);
  const double inv = 1.0 / (static_cast<double>(g.P) * (channels / 4));
  dd::gn_finalize_kernel<<<g.B * 4, 256, 0, st>>>(e->stats[which], e->stats_tiles_img[which], inv, 1e-5f, e->mr[which]);
  e->launches++;
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return fail(DD_ERR_CUDA, std::string("gn_finalize: ") + cudaGetErrorString(err));
  return DD_OK;
}

template <int C, int COND>
int run_apply(dd_engine* e, int which, const float* temb, int temb_bstride, __half* out_hi, __half* out_lo,
              cudaStream_t st, bool out_f8 = false) {
  const Geom g = geom_of(e->cfg);
  dd::ApplyArgs a;
  a.y = e->Y;
  a.mean_rstd = e->mr[which];
  a.gamma = e->gn_gamma[which];
  a.beta = e->gn_beta[which];
  a.cond = e->cond;
  a.temb = temb;
  a.temb_bstride = temb_bstride;
  a.H = g.h;
  a.W = g.w;
  a.ch = e->cfg.cond_h;
  a.cw = e->cfg.cond_w;
  a.ry = g.h > 1 ? static_cast<float>(a.ch - 1) / static_cast<float>(g.h - 1) : 0.f;
  a.rx = g.w > 1 ? static_cast<float>(a.cw - 1) / static_cast<float>(g.w - 1) : 0.f;
  a.out_hi = out_hi;
  a.out_lo = out_lo;
  a.out_a8 = a.out_l8 = nullptr;
  if (out_f8) {  // hi + e4m3 a8 / l8 planes; the e4m3 pair shares the fp16 lo plane's storage
    a.out_a8 = reinterpret_cast<uint8_t*>(out_lo);
    a.out_l8 = a.out_a8 + static_cast<size_t>(g.B) * g.P * C;
  }
  a.scale = kActScale;
  a.status = e->status;
  if (COND == 2 && C == 256) {
    // one 64-thread block per 2 x 2 output quad (rows 2i-1, 2i; columns 2j-1, 2j)
    if (e->up_qpb == 4) {
      dim3 grid((g.w / 2 + 1 + 3) / 4, g.h / 2 + 1, g.B);
      dd::gn_apply_up_split_kernel<4, 4><<<grid, 256, 0, st>>>(a);
    } else {
      dim3 grid(g.w / 2 + 1, g.h / 2 + 1, g.B);
      dd::gn_apply_up_split_kernel<4, 1><<<grid, 64, 0, st>>>(a);
    }
  } else {
    constexpr int PPB = 256 / (C / 8);
    dim3 grid((g.P + PPB - 1) / PPB, g.B);
    dd::gn_apply_split_kernel<C, COND><<<grid, 256, 0, st>>>(a);
  }
  e->launches++;
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return fail(DD_ERR_CUDA, std::string("gn_apply: ") + cudaGetErrorString(err));
  return DD_OK;
}

// One ScheduledCNNRefine.forward + (optionally) the DDIM update; z != nullptr adds sigma * z (stochastic DDIM).
int run_step(dd_engine* e, const float* temb, int temb_bstride, float cx, float ce, float* eps_out, cudaStream_t st,
             const float* z = nullptr, float sigma = 0.f) {
  const Geom g = geom_of(e->cfg);
  int rc;
  // noise_embedding.0 : x (16) -> 64, GN stats
  if ((rc = run_conv(e, 0, e->xs_hi, e->xs_lo, kXScale, dd::EPI_F32_STATS, e->Y, e->stats[0], nullptr, nullptr, st))) return rc;
  if ((rc = run_finalize(e, 0, 64, st))) return rc;
  // with DD_FLAG_FP8_CORR noise_embedding.3 takes hi / a8 / l8 planes too (fp16 hi*hi + two e4m3 correction products)
  const bool f8_ne3 = fp8_active(e) && e->f8_ne3;
  if ((rc = run_apply<64, 0>(e, 0, nullptr, 0, e->S_hi[0], e->S_lo[0], st, f8_ne3))) return rc;
  // noise_embedding.3 : 64 -> 256, GN stats
  if ((rc = run_conv(e, 1, e->S_hi[0], e->S_lo[0], kActScale, dd::EPI_F32_STATS, e->Y, e->stats[1], nullptr, nullptr, st,
                     f8_ne3 ? kF8In : 0))) return rc;
  if ((rc = run_finalize(e, 1, 256, st))) return rc;
  const __half *p_hi, *p_lo;
  if (e->cfg.variant == DD_VARIANT_SWIN) {
    // feat = up(cond + temb) + relu(gn(y2));  convA ; convB   (UpSample_add)
    // with DD_FLAG_FP8_CORR convA and convB take hi / a8 / l8 planes (fp8 correction products); convB's output feeds the
    // swapped-operand pred.0 kernel and stays fp16 hi / lo
    const bool f8 = fp8_active(e);
    if ((rc = run_apply<256, 2>(e, 1, temb, temb_bstride, e->S_hi[1], e->S_lo[1], st, f8))) return rc;
    if ((rc = run_conv(e, 2, e->S_hi[1], e->S_lo[1], kActScale, dd::EPI_SPLIT, nullptr, nullptr, e->S_hi[0], e->S_lo[0], st,
                       f8 ? (kF8In | kF8Out) : 0))) return rc;
    if ((rc = run_conv(e, 3, e->S_hi[0], e->S_lo[0], kActScale, dd::EPI_SPLIT, nullptr, nullptr, e->S_hi[1], e->S_lo[1], st,
                       f8 ? kF8In : 0))) return rc;
    p_hi = e->S_hi[1];
    p_lo = e->S_lo[1];
  } else {
    if ((rc = run_apply<256, 1>(e, 1, temb, temb_bstride, e->S_hi[1], e->S_lo[1], st))) return rc;
    p_hi = e->S_hi[1];
    p_lo = e->S_lo[1];
  }
  // pred.0 : 256 -> 64, GN stats
  if ((rc = run_conv(e, 4, p_hi, p_lo, kActScale, dd::EPI_F32_STATS, e->Y, e->stats[2], nullptr, nullptr, st))) return rc;
  if ((rc = run_finalize(e, 2, 64, st))) return rc;
  if ((rc = run_apply<64, 0>(e, 2, nullptr, 0, e->S_hi[0], e->S_lo[0], st))) return rc;
  // pred.3 : 64 -> 16, GN stats
  if ((rc = run_conv(e, 5, e->S_hi[0], e->S_lo[0], kActScale, dd::EPI_F32_STATS, e->Y, e->stats[3], nullptr, nullptr, st))) return rc;
  if ((rc = run_finalize(e, 3, 16, st))) return rc;
  dd::FinalArgs f;
  f.y = e->Y;
  f.mean_rstd = e->mr[3];
  f.gamma = e->gn_gamma[3];
  f.beta = e->gn_beta[3];
  f.x = e->x32;
  f.x_hi = e->xs_hi;
  f.x_lo = e->xs_lo;
  f.eps_out = eps_out;
  f.cx = cx;
  f.ce = ce;
  f.scale = kXScale;
  f.P = g.P;
  f.status = e->status;
  f.z = z;
  f.sigma = sigma;
  dim3 grid((g.P * 4 + 255) / 256, g.B);
  if (z)
    dd::gn_relu_ddim_stoch_kernel<<<grid, 256, 0, st>>>(f);
  else
    dd::gn_relu_ddim_kernel<<<grid, 256, 0, st>>>(f);
  e->launches++;
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return fail(DD_ERR_CUDA, std::string("gn_relu_ddim: ") + cudaGetErrorString(err));
  return DD_OK;
}

int transpose_in(const float* nchw, float* nhwc, int B, int C, int P, cudaStream_t st) {
  dim3 grid((P + 31) / 32, (C + 31) / 32, B), block(32, 8);
  dd::nchw_to_nhwc_kernel<<<grid, block, 0, st>>>(nchw, nhwc, C, P);
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return fail(DD_ERR_CUDA, std::string("nchw_to_nhwc: ") + cudaGetErrorString(err));
  return DD_OK;
}
int transpose_out(const float* nhwc, float* nchw, int B, int C, int P, cudaStream_t st) {
  dim3 grid((P + 31) / 32, (C + 31) / 32, B), block(32, 8);
  dd::nhwc_to_nchw_kernel<<<grid, block, 0, st>>>(nhwc, nchw, C, P);
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return fail(DD_ERR_CUDA, std::string("nhwc_to_nchw: ") + cudaGetErrorString(err));
  return DD_OK;
}
int split_planes(dd_engine* e, const float* x, __half* hi, __half* lo, size_t n, float scale, cudaStream_t st) {
  const size_t n4 = n / 4;
  int blocks = static_cast<int>((n4 + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  dd::split_planes_kernel<<<blocks, 256, 0, st>>>(x, hi, lo, n4, scale, e->status);
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return fail(DD_ERR_CUDA, std::string("split_planes: ") + cudaGetErrorString(err));
  return DD_OK;
}

int run_decoder(dd_engine* e, float* logit, float* depth, cudaStream_t st) {
  const Geom g = geom_of(e->cfg);
  dd::DecoderArgs a;
  a.x = e->x32;
  a.wt = e->dec_wt;
  a.bt = e->dec_bt;
  a.wc = e->dec_wc;
  a.bc = e->dec_bc;
  a.logit = logit;
  a.depth = depth;
  a.h = g.h;
  a.w = g.w;
  a.eps = 1e-6f;
  dim3 grid((2 * g.w + dd::DEC_TW - 1) / dd::DEC_TW, (2 * g.h + dd::DEC_TH - 1) / dd::DEC_TH, g.B);
  dd::decoder_kernel<<<grid, 256, dd::DEC_SMEM, st>>>(a);
  e->launches++;
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return fail(DD_ERR_CUDA, std::string("decoder: ") + cudaGetErrorString(err));
  return DD_OK;
}

int bind_workspace(dd_engine* e, void* ws, size_t bytes) {
  const size_t need = carve(e, nullptr);
  if (ws == nullptr || bytes < need) return fail(DD_ERR_INVALID, "workspace too small: need " + std::to_string(need));
  if ((reinterpret_cast<uintptr_t>(ws) & 1023) != 0) return fail(DD_ERR_INVALID, "workspace must be 1024-byte aligned");
  if (ws != e->ws) {
    carve(e, ws);
    e->ws = ws;
    drop_graphs(e);
  }
  return DD_OK;
}

const Raw* find(dd_engine* e, const std::string& k) {
  auto it = e->raw.find(k);
  return it == e->raw.end() ? nullptr : &it->second;
}

int dev_alloc(dd_engine* e, void** p, size_t bytes) {
  cudaError_t err = cudaMalloc(p, bytes);
  if (err != cudaSuccess) return fail(DD_ERR_CUDA, std::string("cudaMalloc: ") + cudaGetErrorString(err));
  e->owned.push_back(*p);
  return DD_OK;
}

int pack_layer(dd_engine* e, ConvLayer& L, const float* w, const float* b, int cout, int cin, cudaStream_t st,
               float* scratch_dev) {
  L.sid = shape_id(cin, cout);
  if (L.sid < 0) return fail(DD_ERR_UNSUPPORTED, "unsupported conv shape");
  const size_t n = static_cast<size_t>(cout) * cin * 9;
  int rc;
  if ((rc = dev_alloc(e, reinterpret_cast<void**>(&L.w_hi), n * 2))) return rc;
  if ((rc = dev_alloc(e, reinterpret_cast<void**>(&L.w_lo), n * 2))) return rc;
  if ((rc = dev_alloc(e, reinterpret_cast<void**>(&L.w_simt), n * 4))) return rc;
  if ((rc = dev_alloc(e, reinterpret_cast<void**>(&L.bias), cout * 4))) return rc;
  CUDA_TRY(cudaMemsetAsync(scratch_dev, 0, 4, st));
  dd::absmax_kernel<<<absmax_grid(n), 256, 0, st>>>(w, static_cast<int>(n), scratch_dev);
  float amax = 0.f;
  CUDA_TRY(cudaMemcpyAsync(&amax, scratch_dev, 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  // largest power of two with amax * scale < 2^15: hi stays finite, lo = O(2^4) stays normal
  float scale = 1.f;
  if (amax > 0.f && isfinite(amax)) scale = exp2f(floorf(log2f(32768.f / amax)) - 1.f);
  L.wscale = scale;
  dd::pack_conv_weight_kernel<<<128, 256, 0, st>>>(w, L.w_hi, L.w_lo, L.w_simt, cout, cin, scale);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(L.bias, b, cout * 4, cudaMemcpyDeviceToDevice, st));
  const ShapeInfo s = kShapes[L.sid];
  if ((rc = make_w_map(&L.mb_hi, L.w_hi, cout, cin, s.bk))) return rc;
  if ((rc = make_w_map(&L.mb_lo, L.w_lo, cout, cin, s.bk))) return rc;
  if ((rc = make_w_map(&L.mh_hi, L.w_hi, cout, cin, kHaloBK[L.sid]))) return rc;
  if ((rc = make_w_map(&L.mh_lo, L.w_lo, cout, cin, kHaloBK[L.sid]))) return rc;
  if (cout == 256) {
    if ((rc = make_w_map(&L.mp_hi, L.w_hi, cout, cin, kHaloBK[L.sid], cout / 2))) return rc;
    if ((rc = make_w_map(&L.mp_lo, L.w_lo, cout, cin, kHaloBK[L.sid], cout / 2))) return rc;
  }
  if (cout == 256 && cin % 64 == 0) {  // fp8-correction planes (used when the engine runs with DD_FLAG_FP8_CORR)
    if ((rc = dev_alloc(e, reinterpret_cast<void**>(&L.w8), n))) return rc;
    if ((rc = dev_alloc(e, reinterpret_cast<void**>(&L.lw8), n))) return rc;
    dd::pack_conv_weight8_kernel<<<128, 256, 0, st>>>(w, L.w8, L.lw8, cout, cin, scale);
    CUDA_TRY(cudaGetLastError());
    if ((rc = make_w_map(&L.m8_hi, L.w_hi, cout, cin, 64, cout / 2))) return rc;
    if ((rc = make_w_map8(&L.m8_w, L.w8, cout, cin, cout / 2))) return rc;
    if ((rc = make_w_map8(&L.m8_lw, L.lw8, cout, cin, cout / 2))) return rc;
  }
  if (kSwapBK[L.sid] > 0) {
    if ((rc = dev_alloc(e, reinterpret_cast<void**>(&L.w_swap), static_cast<size_t>(9) * 128 * cin * 2))) return rc;
    dd::pack_swap_weight_kernel<<<128, 256, 0, st>>>(w, L.w_swap, cout, cin, scale);
    CUDA_TRY(cudaGetLastError());
    if ((rc = make_w_map(&L.mw_swap, L.w_swap, 128, cin, kSwapBK[L.sid]))) return rc;
  }
  return DD_OK;
}


// ------------------------------------------------------------------------------------------------ producers
constexpr float kProdScale = 16.f;  // fp16-split pre-scale of every producer activation

// Fold eval-BN (prefix.{weight,bias,running_mean,running_var}) into per-channel (scale, shift) on the host.
int bn_fold(dd_engine* e, const std::string& bn, int ch, std::vector<float>& scale, std::vector<float>& shift,
            cudaStream_t st) {
  const char* parts[4] = {".weight", ".bias", ".running_mean", ".running_var"};
  std::vector<float> v[4];
  for (int i = 0; i < 4; ++i) {
    const Raw* r = find(e, bn + parts[i]);
    if (!r) return fail(DD_ERR_INVALID, "missing weights: " + bn + parts[i]);
    v[i].resize(ch);
    CUDA_TRY(cudaMemcpyAsync(v[i].data(), r->ptr, ch * 4, cudaMemcpyDeviceToHost, st));
  }
  CUDA_TRY(cudaStreamSynchronize(st));
  scale.resize(ch);
  shift.resize(ch);
  for (int c = 0; c < ch; ++c) {
    const double sc = static_cast<double>(v[0][c]) / sqrt(static_cast<double>(v[3][c]) + 1e-5);
    scale[c] = static_cast<float>(sc);
    shift[c] = static_cast<float>(static_cast<double>(v[1][c]) - static_cast<double>(v[2][c]) * sc);
  }
  return DD_OK;
}

// conv weight key `wkey` ([cout][cin][k][k], or ConvT [cin][co][2][2] when transposed) followed by eval-BN `bnkey`
// (folded), or — bnkey empty — by the plain bias `biaskey`.  cin_pad >= cin zero-pads the input-channel axis (RGB -> 32).
int pack_gen(dd_engine* e, GenLayer& L, const std::string& wkey, const std::string& bnkey, int cin, int cout_conv,
             int taps, bool transposed, cudaStream_t st, float* scratch, int cin_pad = 0,
             const std::string& biaskey = std::string()) {
  const Raw* w = find(e, wkey);
  if (!w) return fail(DD_ERR_INVALID, "missing weights: " + wkey);
  const int k = taps == 9 ? 3 : (transposed ? 2 : 1);
  std::vector<int64_t> want = transposed ? std::vector<int64_t>{cin, cout_conv, 2, 2}
                                         : std::vector<int64_t>{cout_conv, cin, k, k};
  if (w->shape != want) return fail(DD_ERR_INVALID, "weight shape mismatch: " + wkey);
  std::vector<float> scale(cout_conv, 1.f), shift(cout_conv, 0.f);
  int rc;
  if (!bnkey.empty()) {
    if ((rc = bn_fold(e, bnkey, cout_conv, scale, shift, st))) return rc;
  } else if (!biaskey.empty()) {
    const Raw* b = find(e, biaskey);
    if (!b) return fail(DD_ERR_INVALID, "missing weights: " + biaskey);
    CUDA_TRY(cudaMemcpyAsync(shift.data(), b->ptr, cout_conv * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
  }
  const int cp = cin_pad > 0 ? cin_pad : cin;
  L.cin = cp;
  L.taps = transposed ? 1 : taps;
  L.cout = transposed ? 4 * cout_conv : cout_conv;
  L.shuffle = transposed ? 1 : 0;
  L.relu = 1;
  // N tile: the width in {256, 192, 128} that wastes the fewest padded columns (ties -> wider); 64 for cout <= 64.
  // A last tile wider than the remaining channels reads zero weight rows (TMA out-of-bounds fill), the epilogue drops them.
  L.nt = 64;
  if (L.cout > 64) {
    int best = 1 << 30;
    for (int nt : {256, 192, 128}) {
      const int padded = (L.cout + nt - 1) / nt * nt;
      if (padded < best) { best = padded; L.nt = nt; }
    }
  }
  if (L.cout % 8 != 0 || cp % 8 != 0) return fail(DD_ERR_UNSUPPORTED, "producer conv channels must be multiples of 8: " + wkey);
  const int cout_pad = (L.cout + L.nt - 1) / L.nt * L.nt;
  const size_t n = static_cast<size_t>(L.cout) * cp * L.taps;
  float *d_scale = nullptr;
  if ((rc = dev_alloc(e, reinterpret_cast<void**>(&L.w_hi), n * 2))) return rc;
  if ((rc = dev_alloc(e, reinterpret_cast<void**>(&L.w_lo), n * 2))) return rc;
  if ((rc = dev_alloc(e, reinterpret_cast<void**>(&L.shift), cout_pad * 4))) return rc;
  if ((rc = dev_alloc(e, reinterpret_cast<void**>(&d_scale), cout_conv * 4))) return rc;
  if (cp != cin) {
    CUDA_TRY(cudaMemsetAsync(L.w_hi, 0, n * 2, st));
    CUDA_TRY(cudaMemsetAsync(L.w_lo, 0, n * 2, st));
  }
  CUDA_TRY(cudaMemcpyAsync(d_scale, scale.data(), cout_conv * 4, cudaMemcpyHostToDevice, st));
  std::vector<float> shift_full(cout_pad, 0.f);
  for (int i = 0; i < L.cout; ++i) shift_full[i] = shift[i % cout_conv];
  CUDA_TRY(cudaMemcpyAsync(L.shift, shift_full.data(), cout_pad * 4, cudaMemcpyHostToDevice, st));
  const int nraw = static_cast<int>(static_cast<size_t>(cout_conv) * cin * (transposed ? 4 : taps));
  CUDA_TRY(cudaMemsetAsync(scratch, 0, 4, st));
  dd::absmax_scaled_kernel<<<absmax_grid(nraw), 256, 0, st>>>(w->ptr, d_scale, nraw, cin * taps, cout_conv, transposed ? 1 : 0, scratch);
  float amax = 0.f;
  CUDA_TRY(cudaMemcpyAsync(&amax, scratch, 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  L.wscale = (amax > 0.f && isfinite(amax)) ? exp2f(floorf(log2f(32768.f / amax)) - 1.f) : 1.f;
  dd::pack_gen_weight_kernel<<<256, 256, 0, st>>>(w->ptr, d_scale, L.w_hi, L.w_lo, L.cout, cin, L.taps,
                                                  transposed ? 1 : 0, L.wscale, cp);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaStreamSynchronize(st));
  if ((rc = make_wgen_map(&L.mb_hi, L.w_hi, L.cout, cp, L.taps, L.nt))) return rc;
  if ((rc = make_wgen_map(&L.mb_lo, L.w_lo, L.cout, cp, L.taps, L.nt))) return rc;
  if ((rc = make_wgen_map(&L.mp_hi, L.w_hi, L.cout, cp, L.taps, L.nt / 2))) return rc;
  if ((rc = make_wgen_map(&L.mp_lo, L.w_lo, L.cout, cp, L.taps, L.nt / 2))) return rc;
  L.alt = (L.nt == 256 && L.cout % 256 == 0 && L.cout % 192 == 0 && !L.shuffle);
  if (L.alt) {
    if ((rc = make_wgen_map(&L.mb_hi_alt, L.w_hi, L.cout, cp, L.taps, 192))) return rc;
    if ((rc = make_wgen_map(&L.mb_lo_alt, L.w_lo, L.cout, cp, L.taps, 192))) return rc;
    if ((rc = make_wgen_map(&L.mp_hi_alt, L.w_hi, L.cout, cp, L.taps, 96))) return rc;
    if ((rc = make_wgen_map(&L.mp_lo_alt, L.w_lo, L.cout, cp, L.taps, 96))) return rc;
  }
  return DD_OK;
}

int pack_producers(dd_engine* e, cudaStream_t st, float* scratch) {
  Producers& p = e->prod;
  int rc;
  for (int i = 0; i < p.nlev; ++i) {
    const std::string si = std::to_string(i);
    if (p.neck) {
      const std::string h = "hahineck.";
      if ((rc = pack_gen(e, p.lat[i], h + "lateral_convs." + si + ".conv.weight", h + "lateral_convs." + si + ".bn",
                         p.C[i], p.C[i], 1, false, st, scratch))) return rc;
      const std::string pj = i == 0 ? h + "conv_proj.0" : h + "trans_proj." + std::to_string(i - 1);
      const std::string fs = i == 0 ? h + "conv_fusion.0" : h + "trans_fusion." + std::to_string(i - 1);
      if ((rc = pack_gen(e, p.proj[i], pj + ".conv.weight", pj + ".bn", p.C[i], 512, 1, false, st, scratch))) return rc;
      if ((rc = pack_gen(e, p.fus[i], fs + ".conv.weight", fs + ".bn", p.C[i] + 512, p.C[i], 9, false, st, scratch))) return rc;
    }
    if ((rc = pack_gen(e, p.fl[i], "conv_lateral." + si + ".0.weight", "conv_lateral." + si + ".1", p.C[i], 256, 9, false,
                       st, scratch))) return rc;
    if (i < p.nlev - 1)
      if ((rc = pack_gen(e, p.fu[i], "conv_up." + si + ".0.weight", "conv_up." + si + ".1", 256, 256, 1, true, st,
                         scratch))) return rc;
  }
  p.ready = true;
  return DD_OK;
}

template <int NT, bool PAIR>
cudaError_t launch_gen(int grid, cudaStream_t st, const CUtensorMap& m0h, const CUtensorMap& m0l, const CUtensorMap& m1h,
                       const CUtensorMap& m1l, const CUtensorMap& bh, const CUtensorMap& bl, const dd::GenConvArgs& a) {
  if constexpr (!PAIR) {
    dd::convgen_umma_kernel<NT, false><<<grid, dd::GenCfg<NT, false>::THREADS, dd::GenCfg<NT, false>::SMEM_BYTES, st>>>(m0h, m0l, m1h, m1l, bh, bl, a);
    return cudaGetLastError();
  } else {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(dd::GenCfg<NT, true>::THREADS);
    cfg.dynamicSmemBytes = dd::GenCfg<NT, true>::SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, dd::convgen_umma_kernel<NT, true>, m0h, m0l, m1h, m1l, bh, bl, a);
  }
}
// m_tiles x n_tiles work items of one producer conv / GEMM -> (use CTA pairs?, grid size).  Pairs (M = 256 per
// tcgen05.mma, half the weight bytes per SM) whenever there are at least two M tiles and the engine allows it.
bool gen_use_pair(const dd_engine* e, int m_tiles) {
  return (e->cfg.flags & DD_FLAG_PAIR_WIDE) && !(e->cfg.flags & DD_FLAG_SIMT_CONV) && m_tiles >= 2 && e->genpair_mask != 0;
}
int gen_grid(const dd_engine* e, bool pair, int m_tiles, int n_tiles) {
  if (!pair) return std::min(m_tiles * n_tiles, e->sm_count);
  return std::min(2 * ((m_tiles + 1) / 2) * n_tiles, e->sm_count & ~1);
}
cudaError_t launch_gen_nt(int nt, bool pair, int grid, cudaStream_t st, const CUtensorMap& m0h, const CUtensorMap& m0l,
                          const CUtensorMap& m1h, const CUtensorMap& m1l, const CUtensorMap& bh, const CUtensorMap& bl,
                          const dd::GenConvArgs& a) {
  switch (nt) {
    case 256: return pair ? launch_gen<256, true>(grid, st, m0h, m0l, m1h, m1l, bh, bl, a) : launch_gen<256, false>(grid, st, m0h, m0l, m1h, m1l, bh, bl, a);
    case 192: return pair ? launch_gen<192, true>(grid, st, m0h, m0l, m1h, m1l, bh, bl, a) : launch_gen<192, false>(grid, st, m0h, m0l, m1h, m1l, bh, bl, a);
    case 128: return pair ? launch_gen<128, true>(grid, st, m0h, m0l, m1h, m1l, bh, bl, a) : launch_gen<128, false>(grid, st, m0h, m0l, m1h, m1l, bh, bl, a);
    default: return pair ? launch_gen<64, true>(grid, st, m0h, m0l, m1h, m1l, bh, bl, a) : launch_gen<64, false>(grid, st, m0h, m0l, m1h, m1l, bh, bl, a);
  }
}

// H, W: OUTPUT grid.  With L.stride == 2 the sources live on a (src_h, src_w) grid.
int run_gen(dd_engine* e, const GenLayer& L, const Planes& a0, int c0, const Planes& a1, int c1, int H, int W,
            float* y32, const float* add32, const Planes* out, cudaStream_t st, int src_h = 0, int src_w = 0,
            int ld_out = 0, int ch_off = 0) {
  const int B = e->cfg.batch;
  dd::GenConvArgs a;
  a.B = B;
  a.H = H;
  a.W = W;
  a.tiles_x = (W + dd::TILE_W - 1) / dd::TILE_W;
  a.tiles_y = (H + dd::TILE_H - 1) / dd::TILE_H;
  a.m_tiles = a.tiles_x * a.tiles_y * B;
  // wave quantisation (as in run_gemm): with few M tiles pick the N-tile width whose last wave wastes least — the
  // level-2 fusion conv of the HAHI neck (768 channels, 30 tile pairs) runs 2 waves of 192 columns instead of 2 of 256
  const bool pair = gen_use_pair(e, a.m_tiles);
  int nt = L.nt;
  if (L.alt) {
    const int units = pair ? (a.m_tiles + 1) / 2 : a.m_tiles, slots = pair ? e->sm_count / 2 : e->sm_count;
    auto cost = [&](int w) { return ((units * (L.cout / w) + slots - 1) / slots) * w; };
    if (cost(192) < cost(256)) nt = 192;
  }
  a.n_tiles = (L.cout + nt - 1) / nt;
  a.kc0 = (c0 + dd::GEN_BK - 1) / dd::GEN_BK;  // a partial last chunk is zero-filled by TMA on both operands
  a.kc1 = (c1 + dd::GEN_BK - 1) / dd::GEN_BK;
  a.c0_ch = c0;
  a.taps = L.taps;
  a.cout = L.cout;
  a.ld_out = ld_out > 0 ? ld_out : L.cout;  // branches of a concatenation write straight into the concatenated planes
  a.ch_off = ch_off;
  a.shift = L.shift;
  a.acc_scale = 1.f / (kProdScale * L.wscale);
  a.relu = L.relu;
  a.m_valid = 0;
  a.stride = L.stride;
  a.add_first = L.add_first;
  a.shuffle = L.shuffle;
  a.y32 = y32;
  a.add32 = add32;
  a.out_hi = out ? out->hi : nullptr;
  a.out_lo = out ? out->lo : nullptr;
  a.split_scale = kProdScale;
  a.status = e->status;
  if (c0 + c1 != L.cin) return fail(DD_ERR_INVALID, "producer conv: source channels do not match the layer");
  CUtensorMap m0h, m0l, m1h, m1l;
  int rc;
  if (L.stride == 1) {
    if ((rc = make_act_map(&m0h, a0.hi, B, H, W, c0, dd::GEN_BK))) return rc;
    if ((rc = make_act_map(&m0l, a0.lo, B, H, W, c0, dd::GEN_BK))) return rc;
  } else {
    if ((rc = make_act_map_strided(&m0h, a0.hi, B, src_h, src_w, c0, dd::GEN_BK, L.stride))) return rc;
    if ((rc = make_act_map_strided(&m0l, a0.lo, B, src_h, src_w, c0, dd::GEN_BK, L.stride))) return rc;
  }
  if (c1 > 0) {
    if ((rc = make_act_map(&m1h, a1.hi, B, H, W, c1, dd::GEN_BK))) return rc;
    if ((rc = make_act_map(&m1l, a1.lo, B, H, W, c1, dd::GEN_BK))) return rc;
  } else {
    m1h = m0h;
    m1l = m0l;
  }
  const int grid = gen_grid(e, pair, a.m_tiles, a.n_tiles);
  const bool use_alt = nt != L.nt;
  const cudaError_t err = launch_gen_nt(nt, pair, grid, st, m0h, m0l, m1h, m1l,
                                        pair ? (use_alt ? L.mp_hi_alt : L.mp_hi) : (use_alt ? L.mb_hi_alt : L.mb_hi),
                                        pair ? (use_alt ? L.mp_lo_alt : L.mp_lo) : (use_alt ? L.mb_lo_alt : L.mb_lo), a);
  e->launches++;
  if (err != cudaSuccess) return fail(DD_ERR_CUDA, std::string("convgen launch: ") + cudaGetErrorString(err));
  return DD_OK;
}

// ------------------------------------------------------------------------------------------------ ResNet backbone
// ResNetForMMBEV with BasicBlocks and no stem (reference src/model/backbone/mmbev_resnet.py:124-160; block = mmdet
// BasicBlock): per stage, block 0 = conv3x3(s2)+BN+ReLU -> conv3x3+BN, skip = biased conv3x3(s2) without BN; other
// blocks are stride 1 with identity skips.  Stride-2 convs use TMA element strides on the same tensor-core conv kernel.
int pack_resnet(dd_engine* e, cudaStream_t st, float* scratch) {
  ResNetW& r = e->rn;
  int rc;
  for (int s = 0; s < 4; ++s) {
    r.blocks[s].assign(r.depths[s], ResBlockW());
    const int cprev = s == 0 ? 3 : r.C[s - 1];
    for (int b = 0; b < r.depths[s]; ++b) {
      ResBlockW& W = r.blocks[s][b];
      const std::string bp = "backbone.layers." + std::to_string(s) + "." + std::to_string(b) + ".";
      const int cin = b == 0 ? cprev : r.C[s];
      const int pad = (cin % dd::GEN_BK) ? dd::GEN_BK : 0;
      if ((rc = pack_gen(e, W.c1, bp + "conv1.weight", bp + "bn1", cin, r.C[s], 9, false, st, scratch, pad))) return rc;
      W.c1.stride = b == 0 ? 2 : 1;
      if ((rc = pack_gen(e, W.c2, bp + "conv2.weight", bp + "bn2", r.C[s], r.C[s], 9, false, st, scratch))) return rc;
      W.c2.add_first = 1;  // out = relu(bn2(conv2) + skip)
      W.has_ds = (b == 0);
      if (W.has_ds) {
        if ((rc = pack_gen(e, W.ds, bp + "downsample.weight", "", cin, r.C[s], 9, false, st, scratch, pad,
                           bp + "downsample.bias"))) return rc;
        W.ds.stride = 2;
        W.ds.relu = 0;
      }
    }
  }
  r.ready = true;
  return DD_OK;
}

int run_resnet(dd_engine* e, const float* rgb, float* const* feats_out, cudaStream_t st) {
  ResNetW& r = e->rn;
  const int B = e->cfg.batch;
  {
    const size_t n = static_cast<size_t>(B) * r.H * r.W * dd::GEN_BK;
    int blocks = static_cast<int>((n + 255) / 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    dd::rgb_to_planes_kernel<<<blocks, 256, 0, st>>>(rgb, r.IN.hi, r.IN.lo, B, r.H * r.W, kProdScale, e->status);
    e->launches++;
    CUDA_TRY(cudaGetLastError());
  }
  const Planes none;
  int rc;
  Planes src = r.IN;
  int src_c = dd::GEN_BK, src_h = r.H, src_w = r.W;
  for (int s = 0; s < 4; ++s) {
    const int C = r.C[s], H = r.Hs[s], W = r.Ws[s];
    int cur = 0;
    for (int b = 0; b < r.depths[s]; ++b) {
      const ResBlockW& Wt = r.blocks[s][b];
      const bool last = (b == r.depths[s] - 1);
      const int k = b & 1;
      const Planes& in = (b == 0) ? src : r.Yp[cur];
      const int in_c = (b == 0) ? src_c : C;
      if ((rc = run_gen(e, Wt.c1, in, in_c, none, 0, H, W, nullptr, nullptr, &r.T, st, src_h, src_w))) return rc;
      const float* skip;
      if (Wt.has_ds) {
        if ((rc = run_gen(e, Wt.ds, in, in_c, none, 0, H, W, r.D32, nullptr, nullptr, st, src_h, src_w))) return rc;
        skip = r.D32;
      } else {
        skip = r.Y32[cur];
      }
      const Planes& outp = last ? e->prod.F[s] : r.Yp[k];
      if ((rc = run_gen(e, Wt.c2, r.T, C, none, 0, H, W, r.Y32[k], skip, &outp, st))) return rc;
      cur = k;
    }
    if (feats_out && feats_out[s]) {
      if ((rc = transpose_out(r.Y32[cur], feats_out[s], B, C, H * W, st))) return rc;
      e->launches++;
    }
    src = e->prod.F[s];
    src_c = C;
    src_h = H;
    src_w = W;
  }
  return DD_OK;
}

// ------------------------------------------------------------------------------------------------ Swin backbone
constexpr float kTokScale = 16.f;  // fp16-split pre-scale of token activations (LayerNorm / GELU / attention outputs)

int copy_param(dd_engine* e, const std::string& key, size_t n, float** out, cudaStream_t st) {
  const Raw* r = find(e, key);
  if (!r) return fail(DD_ERR_INVALID, "missing weights: " + key);
  size_t have = 1;
  for (int64_t d : r->shape) have *= static_cast<size_t>(d);
  if (have != n) return fail(DD_ERR_INVALID, "weight shape mismatch: " + key);
  int rc;
  if ((rc = dev_alloc(e, reinterpret_cast<void**>(out), n * 4))) return rc;
  CUDA_TRY(cudaMemcpyAsync(*out, r->ptr, n * 4, cudaMemcpyDeviceToDevice, st));
  return DD_OK;
}

int pack_gemm(dd_engine* e, Gemm& G, const std::string& wkey, const std::string& bkey, int N, int K, cudaStream_t st,
              float* scratch) {
  const Raw* w = find(e, wkey);
  if (!w) return fail(DD_ERR_INVALID, "missing weights: " + wkey);
  if (w->shape != std::vector<int64_t>{N, K}) return fail(DD_ERR_INVALID, "weight shape mismatch: " + wkey);
  G.K = K;
  G.N = N;
  // N tile as in pack_gen: fewest padded columns among {256, 192, 128}, 64 for N <= 64; partial K chunks / N tiles are
  // completed with zeros by TMA (Swin-L: every N is a multiple of 256 or 192, every K of 64; MPViT: 216, 288, 648, 864 ...)
  G.nt = 64;
  if (N > 64) {
    int best = 1 << 30;
    for (int nt : {256, 192, 128}) {
      const int padded = (N + nt - 1) / nt * nt;
      if (padded < best) { best = padded; G.nt = nt; }
    }
  }
  if (N % 8 != 0 || K % 8 != 0) return fail(DD_ERR_UNSUPPORTED, "linear layer widths must be multiples of 8: " + wkey);
  const int n_pad = (N + G.nt - 1) / G.nt * G.nt;
  const size_t n = static_cast<size_t>(N) * K;
  int rc;
  if ((rc = dev_alloc(e, reinterpret_cast<void**>(&G.w_hi), n * 2))) return rc;
  if ((rc = dev_alloc(e, reinterpret_cast<void**>(&G.w_lo), n * 2))) return rc;
  if ((rc = dev_alloc(e, reinterpret_cast<void**>(&G.bias), n_pad * 4))) return rc;
  CUDA_TRY(cudaMemsetAsync(G.bias, 0, n_pad * 4, st));
  if (!bkey.empty()) {
    const Raw* b = find(e, bkey);
    if (!b) return fail(DD_ERR_INVALID, "missing weights: " + bkey);
    CUDA_TRY(cudaMemcpyAsync(G.bias, b->ptr, N * 4, cudaMemcpyDeviceToDevice, st));
  }
  CUDA_TRY(cudaMemsetAsync(scratch, 0, 4, st));
  dd::absmax_kernel<<<absmax_grid(n), 256, 0, st>>>(w->ptr, static_cast<int>(n), scratch);
  float amax = 0.f;
  CUDA_TRY(cudaMemcpyAsync(&amax, scratch, 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  G.wscale = (amax > 0.f && isfinite(amax)) ? exp2f(floorf(log2f(32768.f / amax)) - 1.f) : 1.f;
  dd::pack_gen_weight_kernel<<<256, 256, 0, st>>>(w->ptr, nullptr, G.w_hi, G.w_lo, N, K, 1, 0, G.wscale);
  CUDA_TRY(cudaGetLastError());
  if ((rc = make_wgen_map(&G.mb_hi, G.w_hi, N, K, 1, G.nt))) return rc;
  if ((rc = make_wgen_map(&G.mb_lo, G.w_lo, N, K, 1, G.nt))) return rc;
  if ((rc = make_wgen_map(&G.mp_hi, G.w_hi, N, K, 1, G.nt / 2))) return rc;
  if ((rc = make_wgen_map(&G.mp_lo, G.w_lo, N, K, 1, G.nt / 2))) return rc;
  G.alt = (G.nt == 256 && N % 256 == 0 && N % 192 == 0);
  if (G.alt) {
    if ((rc = make_wgen_map(&G.mb_hi_alt, G.w_hi, N, K, 1, 192))) return rc;
    if ((rc = make_wgen_map(&G.mb_lo_alt, G.w_lo, N, K, 1, 192))) return rc;
    if ((rc = make_wgen_map(&G.mp_hi_alt, G.w_hi, N, K, 1, 96))) return rc;
    if ((rc = make_wgen_map(&G.mp_lo_alt, G.w_lo, N, K, 1, 96))) return rc;
  }
  return DD_OK;
}

int pack_backbone(dd_engine* e, cudaStream_t st, float* scratch) {
  Backbone& b = e->bb;
  const std::string P = "backbone.";
  int rc;
  if ((rc = copy_param(e, P + "patch_embed.projection.weight", static_cast<size_t>(b.E) * 48, &b.pe_w, st))) return rc;
  if ((rc = copy_param(e, P + "patch_embed.projection.bias", b.E, &b.pe_b, st))) return rc;
  if ((rc = copy_param(e, P + "patch_embed.norm.weight", b.E, &b.pe_g, st))) return rc;
  if ((rc = copy_param(e, P + "patch_embed.norm.bias", b.E, &b.pe_beta, st))) return rc;
  for (int s = 0; s < 4; ++s) {
    const int C = b.E << s;
    SwinStageW& S = b.stage[s];
    S.blocks.assign(b.depths[s], SwinBlockW());
    for (int k = 0; k < b.depths[s]; ++k) {
      SwinBlockW& W = S.blocks[k];
      const std::string bp = P + "stages." + std::to_string(s) + ".blocks." + std::to_string(k) + ".";
      if ((rc = copy_param(e, bp + "norm1.weight", C, &W.ln1_g, st))) return rc;
      if ((rc = copy_param(e, bp + "norm1.bias", C, &W.ln1_b, st))) return rc;
      if ((rc = copy_param(e, bp + "norm2.weight", C, &W.ln2_g, st))) return rc;
      if ((rc = copy_param(e, bp + "norm2.bias", C, &W.ln2_b, st))) return rc;
      if ((rc = copy_param(e, bp + "attn.w_msa.relative_position_bias_table", static_cast<size_t>(169) * b.heads[s], &W.table, st))) return rc;
      if ((rc = pack_gemm(e, W.qkv, bp + "attn.w_msa.qkv.weight", bp + "attn.w_msa.qkv.bias", 3 * C, C, st, scratch))) return rc;
      if ((rc = pack_gemm(e, W.proj, bp + "attn.w_msa.proj.weight", bp + "attn.w_msa.proj.bias", C, C, st, scratch))) return rc;
      if ((rc = pack_gemm(e, W.ffn1, bp + "ffn.layers.0.0.weight", bp + "ffn.layers.0.0.bias", 4 * C, C, st, scratch))) return rc;
      if ((rc = pack_gemm(e, W.ffn2, bp + "ffn.layers.1.weight", bp + "ffn.layers.1.bias", C, 4 * C, st, scratch))) return rc;
    }
    const std::string np = P + "norm" + std::to_string(s) + ".";
    if ((rc = copy_param(e, np + "weight", C, &S.out_g, st))) return rc;
    if ((rc = copy_param(e, np + "bias", C, &S.out_b, st))) return rc;
    if (s < 3) {
      const std::string dp = P + "stages." + std::to_string(s) + ".downsample.";
      if ((rc = copy_param(e, dp + "norm.weight", 4 * C, &S.dn_g, st))) return rc;
      if ((rc = copy_param(e, dp + "norm.bias", 4 * C, &S.dn_b, st))) return rc;
      if ((rc = pack_gemm(e, S.reduction, dp + "reduction.weight", "", 2 * C, 4 * C, st, scratch))) return rc;
    }
  }
  CUDA_TRY(cudaStreamSynchronize(st));
  b.ready = true;
  return DD_OK;
}

// y = act(A[M][K] @ W^T + bias) (+ add32): tokens are laid out as a [ceil(M/16)][16] "image" for the conv kernel
int run_gemm(dd_engine* e, const Gemm& G, const Planes& A, int M, int act, float* y32, const float* add32,
             const Planes* out, cudaStream_t st, int ld_out = 0, int ch_off = 0) {
  dd::GenConvArgs a;
  a.B = 1;
  a.W = 16;
  a.H = (M + 15) / 16;
  a.tiles_x = 1;
  a.tiles_y = (a.H + dd::TILE_H - 1) / dd::TILE_H;
  a.m_tiles = a.tiles_y;
  // wave quantisation: with few M tiles (deep Swin stages) pick the N-tile width whose last wave wastes least
  const bool pair = gen_use_pair(e, a.m_tiles);
  const int units = pair ? (a.m_tiles + 1) / 2 : a.m_tiles, slots = pair ? e->sm_count / 2 : e->sm_count;
  int nt = G.nt;
  if (G.alt) {
    auto cost = [&](int w) { return ((units * (G.N / w) + slots - 1) / slots) * w; };
    if (cost(192) < cost(256)) nt = 192;
  }
  const CUtensorMap& mbh = pair ? ((nt == G.nt) ? G.mp_hi : G.mp_hi_alt) : ((nt == G.nt) ? G.mb_hi : G.mb_hi_alt);
  const CUtensorMap& mbl = pair ? ((nt == G.nt) ? G.mp_lo : G.mp_lo_alt) : ((nt == G.nt) ? G.mb_lo : G.mb_lo_alt);
  a.n_tiles = (G.N + nt - 1) / nt;
  a.kc0 = (G.K + dd::GEN_BK - 1) / dd::GEN_BK;
  a.kc1 = 0;
  a.c0_ch = G.K;
  a.taps = 1;
  a.cout = G.N;
  a.ld_out = ld_out > 0 ? ld_out : G.N;
  a.ch_off = ch_off;
  a.shift = G.bias;
  a.acc_scale = 1.f / (kTokScale * G.wscale);
  a.relu = act;
  a.m_valid = M;
  a.stride = 1;
  a.add_first = 0;
  a.shuffle = 0;
  a.y32 = y32;
  a.add32 = add32;
  a.out_hi = out ? out->hi : nullptr;
  a.out_lo = out ? out->lo : nullptr;
  a.split_scale = kTokScale;
  a.status = e->status;
  CUtensorMap mh, ml;
  int rc;
  if ((rc = make_act_map(&mh, A.hi, 1, a.H, 16, G.K, dd::GEN_BK))) return rc;
  if ((rc = make_act_map(&ml, A.lo, 1, a.H, 16, G.K, dd::GEN_BK))) return rc;
  const int grid = gen_grid(e, pair, a.m_tiles, a.n_tiles);
  const cudaError_t err = launch_gen_nt(nt, pair, grid, st, mh, ml, mh, ml, mbh, mbl, a);
  e->launches++;
  if (err != cudaSuccess) return fail(DD_ERR_CUDA, std::string("gemm launch: ") + cudaGetErrorString(err));
  return DD_OK;
}

int run_ln(dd_engine* e, int C, const float* x, const float* g, const float* b, const Planes& out, int M, float* nchw,
           int HW, cudaStream_t st) {
  const int grid = (M + 7) / 8;
  switch (C) {
    case 192: dd::ln_split_kernel<192><<<grid, 256, 0, st>>>(x, g, b, out.hi, out.lo, kTokScale, M, nchw, HW, e->status); break;
    case 384: dd::ln_split_kernel<384><<<grid, 256, 0, st>>>(x, g, b, out.hi, out.lo, kTokScale, M, nchw, HW, e->status); break;
    case 768: dd::ln_split_kernel<768><<<grid, 256, 0, st>>>(x, g, b, out.hi, out.lo, kTokScale, M, nchw, HW, e->status); break;
    case 1536: dd::ln_split_kernel<1536><<<grid, 256, 0, st>>>(x, g, b, out.hi, out.lo, kTokScale, M, nchw, HW, e->status); break;
    default: return fail(DD_ERR_UNSUPPORTED, "LayerNorm width not instantiated");
  }
  e->launches++;
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return fail(DD_ERR_CUDA, std::string("ln_split: ") + cudaGetErrorString(err));
  return DD_OK;
}

int run_swin(dd_engine* e, const float* rgb, float* const* feats_out, cudaStream_t st) {
  Backbone& b = e->bb;
  const int B = e->cfg.batch;
  {
    const int segs = (b.Ws[0] + dd::PE_TOK - 1) / dd::PE_TOK;
    dd::patch_embed_kernel<192><<<segs * b.Hs[0] * B, 192, 0, st>>>(rgb, b.pe_w, b.pe_b, b.pe_g, b.pe_beta, b.X[0], B, b.H,
                                                                     b.W, b.Hs[0], b.Ws[0]);
    e->launches++;
    CUDA_TRY(cudaGetLastError());
  }
  int rc;
  for (int s = 0; s < 4; ++s) {
    const int C = b.E << s, H = b.Hs[s], W = b.Ws[s], M = B * H * W, nH = b.heads[s];
    float* x = b.X[s & 1];
    const int ws = b.window;
    const int Hp = (H + ws - 1) / ws * ws, Wp = (W + ws - 1) / ws * ws;
    for (int k = 0; k < b.depths[s]; ++k) {
      const SwinBlockW& Wt = b.stage[s].blocks[k];
      if ((rc = run_ln(e, C, x, Wt.ln1_g, Wt.ln1_b, b.AP, M, nullptr, 0, st))) return rc;
      if ((rc = run_gemm(e, Wt.qkv, b.AP, M, 0, b.QKV, nullptr, nullptr, st))) return rc;
      dd::AttnArgs aa;
      aa.qkv = b.QKV;
      aa.qkv_bias = Wt.qkv.bias;
      aa.bias_table = Wt.table;
      aa.out_hi = b.AP.hi;
      aa.out_lo = b.AP.lo;
      aa.scale_out = kTokScale;
      aa.B = B; aa.H = H; aa.W = W; aa.C = C; aa.nH = nH;
      aa.shift = (k & 1) ? ws / 2 : 0;
      aa.Hp = Hp; aa.Wp = Wp; aa.nWx = Wp / ws; aa.nWy = Hp / ws;
      aa.status = e->status;
      if ((e->cfg.flags & DD_FLAG_SIMT_CONV) || (nH & 1) || e->attn_simt) {  // fp32 CUDA-core check path
        dd::window_attention_kernel<<<B * aa.nWx * aa.nWy * nH, 64, 0, st>>>(aa);
      } else {  // tcgen05: pairs of heads of one window per M = 128 tile, three persistent CTAs per SM
        const int pairs = B * aa.nWx * aa.nWy * (nH / 2);
        const int grid = pairs < 3 * e->sm_count ? pairs : 3 * e->sm_count;
        dd::window_attention_umma_kernel<<<grid, 128, dd::WAU_SMEM, st>>>(aa, pairs);
      }
      e->launches++;
      CUDA_TRY(cudaGetLastError());
      if ((rc = run_gemm(e, Wt.proj, b.AP, M, 0, x, x, nullptr, st))) return rc;      // x += proj(attn)
      if ((rc = run_ln(e, C, x, Wt.ln2_g, Wt.ln2_b, b.AP, M, nullptr, 0, st))) return rc;
      if ((rc = run_gemm(e, Wt.ffn1, b.AP, M, 2, nullptr, nullptr, &b.HP, st))) return rc;  // GELU(fc1) -> planes
      if ((rc = run_gemm(e, Wt.ffn2, b.HP, M, 0, x, x, nullptr, st))) return rc;      // x += fc2(...)
    }
    // per-stage output norm straight into the neck's input planes (+ NCHW copy on request)
    if ((rc = run_ln(e, C, x, b.stage[s].out_g, b.stage[s].out_b, e->prod.F[s], M, feats_out ? feats_out[s] : nullptr,
                     H * W, st))) return rc;
    if (s < 3) {
      const int M2 = B * b.Hs[s + 1] * b.Ws[s + 1];
      const int grid = (M2 + 7) / 8;
      const SwinStageW& S = b.stage[s];
      switch (C) {
        case 192: dd::merge_ln_split_kernel<192><<<grid, 256, 0, st>>>(x, S.dn_g, S.dn_b, b.AP.hi, b.AP.lo, kTokScale, B, H, W, e->status); break;
        case 384: dd::merge_ln_split_kernel<384><<<grid, 256, 0, st>>>(x, S.dn_g, S.dn_b, b.AP.hi, b.AP.lo, kTokScale, B, H, W, e->status); break;
        case 768: dd::merge_ln_split_kernel<768><<<grid, 256, 0, st>>>(x, S.dn_g, S.dn_b, b.AP.hi, b.AP.lo, kTokScale, B, H, W, e->status); break;
        default: return fail(DD_ERR_UNSUPPORTED, "patch merging width not instantiated");
      }
      e->launches++;
      CUDA_TRY(cudaGetLastError());
      if ((rc = run_gemm(e, S.reduction, b.AP, M2, 0, b.X[(s + 1) & 1], nullptr, nullptr, st))) return rc;
    }
  }
  return DD_OK;
}

#include "mpvit_host.inc"

}  // namespace

extern "C" {

int dd_abi_version(void) { return DD_ABI_VERSION; }
const char* dd_last_error(void) { return g_err.c_str(); }

int dd_create(const dd_config* cfg, dd_handle* out) {
  if (!cfg || !out) return fail(DD_ERR_INVALID, "null argument");
  if (cfg->abi_version != DD_ABI_VERSION) return fail(DD_ERR_INVALID, "ABI version mismatch");
  if (cfg->variant != DD_VARIANT_RES && cfg->variant != DD_VARIANT_SWIN) return fail(DD_ERR_INVALID, "bad variant");
  if (cfg->batch < 1 || cfg->latent_h < 1 || cfg->latent_w < 1 || cfg->num_inference_steps < 1)
    return fail(DD_ERR_INVALID, "bad geometry");
  if (cfg->variant == DD_VARIANT_RES && (cfg->cond_h != cfg->latent_h || cfg->cond_w != cfg->latent_w))
    return fail(DD_ERR_INVALID, "Res variant needs the condition map at latent resolution");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(DD_ERR_UNSUPPORTED, "no CUDA device: libddengine has no CPU path");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(DD_ERR_INVALID, "bad device ordinal");
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10) return fail(DD_ERR_UNSUPPORTED, "libddengine is built for sm_100a (Blackwell B200) only");
  CUDA_TRY(cudaSetDevice(cfg->device));
  int rc;
  if ((rc = load_driver())) return rc;
  dd_engine* e = new dd_engine();
  e->cfg = *cfg;
  e->sm_count = prop.multiProcessorCount;
#ifdef DD_PROBES
  if (const char* v = getenv("DD_FP8_PROBE")) e->probe_fp8 = atoi(v);
  if (const char* v = getenv("DD_SWAP_MASK")) e->swap_mask = atoi(v);
  if (const char* v = getenv("DD_HALO_MASK")) e->halo_mask = atoi(v);
  if (const char* v = getenv("DD_PAIR_MASK")) e->pair_mask = atoi(v);
  if (const char* v = getenv("DD_GENPAIR")) e->genpair_mask = atoi(v);
  if (const char* v = getenv("DD_SWAPHALO")) e->swaphalo_mask = atoi(v);
  if (const char* v = getenv("DD_ATTN_SIMT")) e->attn_simt = atoi(v);
  e->want_clk_probe = getenv("DD_CLK_PROBE") != nullptr;
  if (const char* v = getenv("DD_F8_NE3")) e->f8_ne3 = atoi(v) != 0;
  if (const char* v = getenv("DD_UP_QPB")) e->up_qpb = atoi(v);
#endif
  if (cudaMallocHost(&e->status_host, 64) != cudaSuccess ||
      cudaStreamCreateWithFlags(&e->cap_stream, cudaStreamNonBlocking) != cudaSuccess ||
      configure_all_kernels() != cudaSuccess || configure_halo_kernels() != cudaSuccess ||
      configure_swap_kernels() != cudaSuccess) {
    std::string msg = std::string("engine setup failed: ") + cudaGetErrorString(cudaGetLastError());
    if (e->status_host) cudaFreeHost(e->status_host);
    if (e->cap_stream) cudaStreamDestroy(e->cap_stream);
    delete e;
    return fail(DD_ERR_CUDA, msg);
  }
  *out = e;
  return DD_OK;
}

int dd_destroy(dd_handle h) {
  if (!h) return DD_OK;
  cudaSetDevice(h->cfg.device);
  drop_graphs(h);
  for (void* p : h->owned) cudaFree(p);
  if (h->status_host) cudaFreeHost(h->status_host);
  if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
  delete h;
  return DD_OK;
}

static const char* kKeys[] = {
    "model.noise_embedding.0.weight", "model.noise_embedding.0.bias", "model.noise_embedding.1.weight",
    "model.noise_embedding.1.bias", "model.noise_embedding.3.weight", "model.noise_embedding.3.bias",
    "model.noise_embedding.4.weight", "model.noise_embedding.4.bias", "model.upsample_fuse.convA.conv.weight",
    "model.upsample_fuse.convA.conv.bias", "model.upsample_fuse.convB.conv.weight",
    "model.upsample_fuse.convB.conv.bias", "model.time_embedding.weight", "model.pred.0.weight", "model.pred.0.bias",
    "model.pred.1.weight", "model.pred.1.bias", "model.pred.3.weight", "model.pred.3.bias", "model.pred.4.weight",
    "model.pred.4.bias", "depth_transform.conv_inv_transform.0.weight", "depth_transform.conv_inv_transform.0.bias",
    "depth_transform.conv_inv_transform.1.weight", "depth_transform.conv_inv_transform.1.bias",
    "depth_transform.conv_inv_transform.1.running_mean", "depth_transform.conv_inv_transform.1.running_var",
    "depth_transform.conv_inv_transform.3.0.weight", "depth_transform.conv_inv_transform.3.0.bias"};

int dd_set_weight(dd_handle h, const char* name, const float* dev_ptr, const int64_t* shape, int32_t ndim) {
  if (!h || !name || !dev_ptr || ndim < 0 || ndim > 4) return fail(DD_ERR_INVALID, "bad argument");
  bool known = strncmp(name, "hahineck.", 9) == 0 || strncmp(name, "conv_lateral.", 13) == 0 ||
               strncmp(name, "conv_up.", 8) == 0 ||  // step-invariant producers (optional, dd_enable_producers)
               strncmp(name, "backbone.", 9) == 0 ||  // native backbone (optional, dd_enable_backbone)
               strncmp(name, "depth_transform.conv_transform.", 31) == 0;  // encoder t() (optional, dd_encode)
  for (const char* k : kKeys) known |= (strcmp(k, name) == 0);
  if (!known) return fail(DD_ERR_INVALID, std::string("unknown weight key: ") + name);
  Raw r;
  r.ptr = dev_ptr;
  r.shape.assign(shape, shape + ndim);
  h->raw[name] = r;
  h->weights_ready = false;
  return DD_OK;
}

int dd_finalize_weights(dd_handle h, void* cuda_stream) {
  if (!h) return fail(DD_ERR_INVALID, "null handle");
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  const bool swin = h->cfg.variant == DD_VARIANT_SWIN;
  std::string missing;
  for (const char* k : kKeys) {
    if (!swin && strstr(k, "upsample_fuse")) continue;
    if (!find(h, k)) missing += std::string(missing.empty() ? "" : ", ") + k;
  }
  if (!missing.empty()) return fail(DD_ERR_INVALID, "missing weights: " + missing);
  auto expect = [&](const char* k, std::vector<int64_t> s) { return find(h, k)->shape == s; };
  if (!expect("model.noise_embedding.0.weight", {64, 16, 3, 3}) || !expect("model.noise_embedding.3.weight", {256, 64, 3, 3}) ||
      !expect("model.pred.0.weight", {64, 256, 3, 3}) || !expect("model.pred.3.weight", {16, 64, 3, 3}) ||
      !expect("model.time_embedding.weight", {DD_TIME_ROWS, 256}) ||
      !expect("depth_transform.conv_inv_transform.0.weight", {16, 16, 4, 4}) ||
      !expect("depth_transform.conv_inv_transform.3.0.weight", {1, 16, 3, 3}) ||
      (swin && (!expect("model.upsample_fuse.convA.conv.weight", {256, 256, 3, 3}) ||
                !expect("model.upsample_fuse.convB.conv.weight", {256, 256, 3, 3}))))
    return fail(DD_ERR_INVALID, "weight shape mismatch with the reference architecture");
  // drop any previous pack
  drop_graphs(h);
  for (void* p : h->owned) cudaFree(p);
  h->owned.clear();
  float* scratch = nullptr;
  int rc;
  if ((rc = dev_alloc(h, reinterpret_cast<void**>(&scratch), 64))) return rc;
  auto W = [&](const char* k) { return find(h, k)->ptr; };
  if ((rc = pack_layer(h, h->L[0], W("model.noise_embedding.0.weight"), W("model.noise_embedding.0.bias"), 64, 16, st, scratch))) return rc;
  if ((rc = pack_layer(h, h->L[1], W("model.noise_embedding.3.weight"), W("model.noise_embedding.3.bias"), 256, 64, st, scratch))) return rc;
  if (swin) {
    if ((rc = pack_layer(h, h->L[2], W("model.upsample_fuse.convA.conv.weight"), W("model.upsample_fuse.convA.conv.bias"), 256, 256, st, scratch))) return rc;
    if ((rc = pack_layer(h, h->L[3], W("model.upsample_fuse.convB.conv.weight"), W("model.upsample_fuse.convB.conv.bias"), 256, 256, st, scratch))) return rc;
  }
  if ((rc = pack_layer(h, h->L[4], W("model.pred.0.weight"), W("model.pred.0.bias"), 64, 256, st, scratch))) return rc;
  if ((rc = pack_layer(h, h->L[5], W("model.pred.3.weight"), W("model.pred.3.bias"), 16, 64, st, scratch))) return rc;
  const char* gnk[4] = {"model.noise_embedding.1", "model.noise_embedding.4", "model.pred.1", "model.pred.4"};
  const int gnc[4] = {64, 256, 64, 16};
  for (int i = 0; i < 4; ++i) {
    if ((rc = dev_alloc(h, reinterpret_cast<void**>(&h->gn_gamma[i]), gnc[i] * 4))) return rc;
    if ((rc = dev_alloc(h, reinterpret_cast<void**>(&h->gn_beta[i]), gnc[i] * 4))) return rc;
    CUDA_TRY(cudaMemcpyAsync(h->gn_gamma[i], W((std::string(gnk[i]) + ".weight").c_str()), gnc[i] * 4, cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(h->gn_beta[i], W((std::string(gnk[i]) + ".bias").c_str()), gnc[i] * 4, cudaMemcpyDeviceToDevice, st));
  }
  if ((rc = dev_alloc(h, reinterpret_cast<void**>(&h->temb), DD_TIME_ROWS * 256 * 4))) return rc;
  CUDA_TRY(cudaMemcpyAsync(h->temb, W("model.time_embedding.weight"), DD_TIME_ROWS * 256 * 4, cudaMemcpyDeviceToDevice, st));
  // decoder: fold eval-BN into the transposed conv (tiny: do it on the host in fp64)
  std::vector<float> wt(16 * 16 * 16), bt(16), g(16), be(16), mu(16), var(16), wc(16 * 9), bc(1);
  CUDA_TRY(cudaMemcpyAsync(wt.data(), W("depth_transform.conv_inv_transform.0.weight"), wt.size() * 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(bt.data(), W("depth_transform.conv_inv_transform.0.bias"), 64, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(g.data(), W("depth_transform.conv_inv_transform.1.weight"), 64, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(be.data(), W("depth_transform.conv_inv_transform.1.bias"), 64, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(mu.data(), W("depth_transform.conv_inv_transform.1.running_mean"), 64, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(var.data(), W("depth_transform.conv_inv_transform.1.running_var"), 64, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(wc.data(), W("depth_transform.conv_inv_transform.3.0.weight"), wc.size() * 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(bc.data(), W("depth_transform.conv_inv_transform.3.0.bias"), 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  std::vector<float> wt_f(4 * 4 * 16 * 16), bt_f(16), wc_f(9 * 16);
  for (int co = 0; co < 16; ++co) {
    const double sc = static_cast<double>(g[co]) / sqrt(static_cast<double>(var[co]) + 1e-5);
    bt_f[co] = static_cast<float>((static_cast<double>(bt[co]) - mu[co]) * sc + be[co]);
    for (int ci = 0; ci < 16; ++ci)
      for (int ky = 0; ky < 4; ++ky)
        for (int kx = 0; kx < 4; ++kx)  // ConvTranspose2d weight layout: [Cin][Cout][kh][kw]
          wt_f[((ky * 4 + kx) * 16 + ci) * 16 + co] =
              static_cast<float>(static_cast<double>(wt[((ci * 16 + co) * 4 + ky) * 4 + kx]) * sc);
  }
  for (int ci = 0; ci < 16; ++ci)
    for (int tap = 0; tap < 9; ++tap) wc_f[tap * 16 + ci] = wc[ci * 9 + tap];
  if ((rc = dev_alloc(h, reinterpret_cast<void**>(&h->dec_wt), wt_f.size() * 4))) return rc;
  if ((rc = dev_alloc(h, reinterpret_cast<void**>(&h->dec_bt), 64))) return rc;
  if ((rc = dev_alloc(h, reinterpret_cast<void**>(&h->dec_wc), wc_f.size() * 4))) return rc;
  CUDA_TRY(cudaMemcpyAsync(h->dec_wt, wt_f.data(), wt_f.size() * 4, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(h->dec_bt, bt_f.data(), 64, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(h->dec_wc, wc_f.data(), wc_f.size() * 4, cudaMemcpyHostToDevice, st));
  h->dec_bc = bc[0];
  CUDA_TRY(cudaStreamSynchronize(st));
  h->enc_w1 = nullptr;
  if (find(h, "depth_transform.conv_transform.0.0.weight")) {
    const std::string P = "depth_transform.conv_transform.";
    const Raw *w1 = find(h, P + "0.0.weight"), *w2 = find(h, P + "1.0.weight");
    if (!w2 || w1->shape != std::vector<int64_t>{16, 1, 3, 3} || w2->shape != std::vector<int64_t>{16, 16, 3, 3})
      return fail(DD_ERR_INVALID, "encoder weights missing / wrong shape");
    std::vector<float> s1, t1, s2, t2, hw1(144), hw2(2304);
    if ((rc = bn_fold(h, P + "0.1", 16, s1, t1, st))) return rc;
    if ((rc = bn_fold(h, P + "1.1", 16, s2, t2, st))) return rc;
    CUDA_TRY(cudaMemcpyAsync(hw1.data(), w1->ptr, 144 * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaMemcpyAsync(hw2.data(), w2->ptr, 2304 * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    std::vector<float> f1(144), f2(2304);
    for (int co = 0; co < 16; ++co)
      for (int tap = 0; tap < 9; ++tap) f1[tap * 16 + co] = static_cast<float>(static_cast<double>(hw1[co * 9 + tap]) * s1[co]);
    for (int co = 0; co < 16; ++co)
      for (int ci = 0; ci < 16; ++ci)
        for (int tap = 0; tap < 9; ++tap)
          f2[(tap * 16 + ci) * 16 + co] = static_cast<float>(static_cast<double>(hw2[(co * 16 + ci) * 9 + tap]) * s2[co]);
    if ((rc = dev_alloc(h, reinterpret_cast<void**>(&h->enc_w1), 144 * 4))) return rc;
    if ((rc = dev_alloc(h, reinterpret_cast<void**>(&h->enc_b1), 64))) return rc;
    if ((rc = dev_alloc(h, reinterpret_cast<void**>(&h->enc_w2), 2304 * 4))) return rc;
    if ((rc = dev_alloc(h, reinterpret_cast<void**>(&h->enc_b2), 64))) return rc;
    CUDA_TRY(cudaMemcpyAsync(h->enc_w1, f1.data(), 144 * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(h->enc_b1, t1.data(), 64, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(h->enc_w2, f2.data(), 2304 * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(h->enc_b2, t2.data(), 64, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));
  }
  h->prod.ready = false;
  if (h->prod.enabled)
    if ((rc = pack_producers(h, st, scratch))) return rc;
  h->bb.ready = false;
  if (h->bb.enabled)
    if ((rc = pack_backbone(h, st, scratch))) return rc;
  h->rn.ready = false;
  if (h->rn.enabled)
    if ((rc = pack_resnet(h, st, scratch))) return rc;
  h->mp.ready = false;
  if (h->mp.enabled)
    if ((rc = pack_mpvit(h, st, scratch))) return rc;
  // the registered pointers were borrowed for this call only (include/dd_engine.h): forget them, so a later finalize
  // cannot read memory the caller has freed in the meantime — every key has to be registered again
  h->raw.clear();
  h->weights_ready = true;
  return DD_OK;
}

int dd_set_schedule(dd_handle h, const int64_t* timesteps, const double* c_x, const double* c_eps, int32_t n) {
  if (!h || !timesteps || !c_x || !c_eps) return fail(DD_ERR_INVALID, "null argument");
  if (n != h->cfg.num_inference_steps) return fail(DD_ERR_INVALID, "schedule length != num_inference_steps");
  h->ts.assign(timesteps, timesteps + n);
  h->cx.resize(n);
  h->ce.resize(n);
  for (int i = 0; i < n; ++i) {
    if (timesteps[i] < 0 || timesteps[i] >= DD_TIME_ROWS) return fail(DD_ERR_INVALID, "timestep outside time_embedding");
    h->cx[i] = static_cast<float>(c_x[i]);
    h->ce[i] = static_cast<float>(c_eps[i]);
  }
  h->sg.assign(n, 0.f);
  drop_graphs(h);
  return DD_OK;
}

int dd_set_schedule_eta(dd_handle h, const int64_t* timesteps, const double* c_x, const double* c_eps,
                        const double* sigma, int32_t n) {
  if (!h || !sigma) return fail(DD_ERR_INVALID, "null argument");
  for (int i = 0; i < n; ++i)
    if (!(sigma[i] >= 0.0)) return fail(DD_ERR_INVALID, "sigma must be finite and >= 0");
  int rc;
  if ((rc = dd_set_schedule(h, timesteps, c_x, c_eps, n))) return rc;
  for (int i = 0; i < n; ++i) h->sg[i] = static_cast<float>(sigma[i]);
  return DD_OK;
}

size_t dd_workspace_bytes(dd_handle h) { return h ? carve(h, nullptr) : 0; }

static int poll_status(dd_handle h, cudaStream_t st) {
  CUDA_TRY(cudaMemcpyAsync(h->status_host, h->status, 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  if (*h->status_host & 1)
    return fail(DD_ERR_RANGE, "an activation exceeded the operand split's range (16 |v| > 6e4; with fp8 corrections, "
                              "DD_FLAG_FP8_CORR, 16 |v| > 1792: create the engine without that flag / set "
                              "head.fp8_corrections = False)");
  return DD_OK;
}

// dd_denoise_decode and dd_denoise_decode_steps: the T-step loop (+ a decode after every step when depth_steps_out
// is given: the *Vis heads' `pred_inter`, reference ..._swin_addHAHI_vis.py:130-149,289-304), then the final decode.
// step_noise (stochastic engines only, then required): NCHW [T][B][16][h][w]; latent_steps_out (nullable, stochastic
// engines only): NCHW [T][B][16][h][w], the latent after every step.
static int denoise_impl(dd_handle h, const float* cond, const float* noise, const float* step_noise, float* latent_out,
                        float* latent_steps_out, float* logit_out, float* depth_out, float* depth_steps_out,
                        void* workspace, size_t workspace_bytes, void* cuda_stream) {
  if (!h || !noise || (!depth_out && !depth_steps_out)) return fail(DD_ERR_INVALID, "null argument");
  const bool stoch = (h->cfg.flags & DD_FLAG_STOCHASTIC) != 0;
  if (stoch != (step_noise != nullptr))
    return fail(DD_ERR_INVALID, stoch ? "engine was created with DD_FLAG_STOCHASTIC: it needs step noise "
                                        "(dd_denoise_decode_stochastic)"
                                      : "dd_denoise_decode_stochastic needs an engine created with DD_FLAG_STOCHASTIC");
  if (!cond && !h->cond_ready) return fail(DD_ERR_INVALID, "cond is NULL but dd_build_condition has not run");
  if (!h->weights_ready) return fail(DD_ERR_INVALID, "dd_finalize_weights has not been called");
  if (static_cast<int>(h->ts.size()) != h->cfg.num_inference_steps) return fail(DD_ERR_INVALID, "dd_set_schedule has not been called");
  if (depth_steps_out && !(h->cfg.flags & DD_FLAG_STEP_DECODE))
    return fail(DD_ERR_INVALID, "dd_denoise_decode_steps needs an engine created with DD_FLAG_STEP_DECODE");
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  int rc;
  if ((rc = bind_workspace(h, workspace, workspace_bytes))) return rc;
  const Geom g = geom_of(h->cfg);
  if (cond) {
    h->launches = 0;
    CUDA_TRY(cudaMemsetAsync(h->status, 0, 64, st));
    if ((rc = transpose_in(cond, h->cond, g.B, 256, h->cfg.cond_h * h->cfg.cond_w, st))) return rc;
    h->launches += 1;
  }  // else: dd_build_condition left the NHWC condition map (and the launch / status counters) in place
  h->cond_ready = false;
  if ((rc = transpose_in(noise, h->x32, g.B, 16, g.P, st))) return rc;
  if ((rc = split_planes(h, h->x32, h->xs_hi, h->xs_lo, static_cast<size_t>(g.B) * g.P * 16, kXScale, st))) return rc;
  h->launches += 2;
  const int T = h->cfg.num_inference_steps;
  const size_t map_elems = static_cast<size_t>(g.B) * g.P * 4;  // one decoded batch [B][2h][2w]
  const size_t lat_elems = static_cast<size_t>(g.B) * g.P * 16;  // one latent batch [B][P][16]
  const bool steps = depth_steps_out != nullptr;
  const bool lsteps = latent_steps_out != nullptr;
  if (stoch) {
    // the graph reads the noise from the workspace only: stage the caller's NCHW [T][B][16][P] as NHWC, T*B "images"
    if ((rc = transpose_in(step_noise, h->step_noise, T * g.B, 16, g.P, st))) return rc;
    h->launches++;
  }
  auto loop = [&](cudaStream_t s) -> int {
    for (int i = 0; i < T; ++i) {
      int r = stoch ? run_step(h, h->temb + h->ts[i] * 256, 0, h->cx[i], h->ce[i], nullptr, s, h->step_noise + i * lat_elems,
                               h->sg[i])
                    : run_step(h, h->temb + h->ts[i] * 256, 0, h->cx[i], h->ce[i], nullptr, s);
      if (r == DD_OK && steps) r = run_decoder(h, nullptr, h->inter + i * map_elems, s);
      if (r == DD_OK && lsteps) {
        r = transpose_out(h->x32, h->lat_steps + i * lat_elems, g.B, 16, g.P, s);
        h->launches++;
      }
      if (r != DD_OK) return r;
    }
    return DD_OK;
  };
  if (h->cfg.flags & DD_FLAG_CUDA_GRAPH) {
    const int which = stoch ? dd_engine::G_STOCH + (steps ? 1 : 0) + (lsteps ? 2 : 0)
                            : (steps ? dd_engine::G_LOOP_STEPS : dd_engine::G_LOOP);
    if ((rc = graph_run(h, which, st, loop))) return rc;
  } else if ((rc = loop(st))) {
    return rc;
  }
  if (lsteps)
    CUDA_TRY(cudaMemcpyAsync(latent_steps_out, h->lat_steps, static_cast<size_t>(T) * lat_elems * 4,
                             cudaMemcpyDeviceToDevice, st));
  if (steps) {
    CUDA_TRY(cudaMemcpyAsync(depth_steps_out, h->inter, static_cast<size_t>(T) * map_elems * 4, cudaMemcpyDeviceToDevice, st));
    if (depth_out)
      CUDA_TRY(cudaMemcpyAsync(depth_out, h->inter + static_cast<size_t>(T - 1) * map_elems, map_elems * 4,
                               cudaMemcpyDeviceToDevice, st));
    if (logit_out)  // the logits of the final map only: one more (cheap) decode, its depth lands in the scratch slot
      if ((rc = run_decoder(h, logit_out, h->inter + static_cast<size_t>(T - 1) * map_elems, st))) return rc;
  } else if ((rc = run_decoder(h, logit_out, depth_out, st))) {
    return rc;
  }
  if (latent_out) {
    if ((rc = transpose_out(h->x32, latent_out, g.B, 16, g.P, st))) return rc;
    h->launches++;
  }
  if (h->cfg.flags & DD_FLAG_CHECK_RANGE) return poll_status(h, st);
  return DD_OK;
}

int dd_denoise_decode(dd_handle h, const float* cond, const float* noise, float* latent_out, float* logit_out,
                      float* depth_out, void* workspace, size_t workspace_bytes, void* cuda_stream) {
  if (!depth_out) return fail(DD_ERR_INVALID, "null argument");
  return denoise_impl(h, cond, noise, nullptr, latent_out, nullptr, logit_out, depth_out, nullptr, workspace,
                      workspace_bytes, cuda_stream);
}

int dd_denoise_decode_steps(dd_handle h, const float* cond, const float* noise, float* latent_out, float* logit_out,
                            float* depth_steps_out, void* workspace, size_t workspace_bytes, void* cuda_stream) {
  if (!depth_steps_out) return fail(DD_ERR_INVALID, "null argument");
  return denoise_impl(h, cond, noise, nullptr, latent_out, nullptr, logit_out, nullptr, depth_steps_out, workspace,
                      workspace_bytes, cuda_stream);
}

int dd_denoise_decode_stochastic(dd_handle h, const float* cond, const float* noise, const float* step_noise,
                                 float* latent_out, float* latent_steps_out, float* logit_out, float* depth_out,
                                 float* depth_steps_out, void* workspace, size_t workspace_bytes, void* cuda_stream) {
  if (!step_noise || (!depth_out && !depth_steps_out)) return fail(DD_ERR_INVALID, "null argument");
  return denoise_impl(h, cond, noise, step_noise, latent_out, latent_steps_out, logit_out, depth_out, depth_steps_out,
                      workspace, workspace_bytes, cuda_stream);
}

int dd_denoiser_forward(dd_handle h, const float* cond, const float* noisy, const int64_t* t_host, float* eps_out,
                        void* workspace, size_t workspace_bytes, void* cuda_stream) {
  if (!h || !cond || !noisy || !t_host || !eps_out) return fail(DD_ERR_INVALID, "null argument");
  if (!h->weights_ready) return fail(DD_ERR_INVALID, "dd_finalize_weights has not been called");
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  int rc;
  if ((rc = bind_workspace(h, workspace, workspace_bytes))) return rc;
  const Geom g = geom_of(h->cfg);
  h->launches = 0;
  CUDA_TRY(cudaMemsetAsync(h->status, 0, 64, st));
  for (int b = 0; b < g.B; ++b) {
    if (t_host[b] < 0 || t_host[b] >= DD_TIME_ROWS) return fail(DD_ERR_INVALID, "timestep outside time_embedding");
    CUDA_TRY(cudaMemcpyAsync(h->temb_sel + b * 256, h->temb + t_host[b] * 256, 1024, cudaMemcpyDeviceToDevice, st));
  }
  if ((rc = transpose_in(cond, h->cond, g.B, 256, h->cfg.cond_h * h->cfg.cond_w, st))) return rc;
  if ((rc = transpose_in(noisy, h->x32, g.B, 16, g.P, st))) return rc;
  if ((rc = split_planes(h, h->x32, h->xs_hi, h->xs_lo, static_cast<size_t>(g.B) * g.P * 16, kXScale, st))) return rc;
  // eps (NHWC) lands in the tail of Y's storage: Y holds y6 in its first B*P*16 floats at that point
  float* eps_nhwc = h->Y + static_cast<size_t>(g.B) * g.P * 16;
  if ((rc = run_step(h, h->temb_sel, 256, 0.f, 0.f, eps_nhwc, st))) return rc;
  if ((rc = transpose_out(eps_nhwc, eps_out, g.B, 16, g.P, st))) return rc;
  if (h->cfg.flags & DD_FLAG_CHECK_RANGE) return poll_status(h, st);
  return DD_OK;
}

int dd_decode(dd_handle h, const float* latent, float* logit_out, float* depth_out, void* workspace,
              size_t workspace_bytes, void* cuda_stream) {
  if (!h || !latent || !depth_out) return fail(DD_ERR_INVALID, "null argument");
  if (!h->weights_ready) return fail(DD_ERR_INVALID, "dd_finalize_weights has not been called");
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  int rc;
  if ((rc = bind_workspace(h, workspace, workspace_bytes))) return rc;
  const Geom g = geom_of(h->cfg);
  if ((rc = transpose_in(latent, h->x32, g.B, 16, g.P, st))) return rc;
  return run_decoder(h, logit_out, depth_out, st);
}

int dd_enable_producers(dd_handle h, const dd_producer_config* pc) {
  if (!h || !pc) return fail(DD_ERR_INVALID, "null argument");
  if (pc->num_levels < 2 || pc->num_levels > 4) return fail(DD_ERR_INVALID, "producers need 2..4 pyramid levels");
  Producers p;
  p.enabled = true;
  p.neck = pc->has_neck != 0;
  p.nlev = pc->num_levels;
  for (int i = 0; i < p.nlev; ++i) {
    p.C[i] = pc->channels[i];
    p.H[i] = pc->heights[i];
    p.W[i] = pc->widths[i];
    // 16-byte rows for TMA and the vector stores of the epilogues; nothing else constrains the counts (MPViT: 128/216/288/288)
    if (p.C[i] % 8 != 0 || p.C[i] <= 0) return fail(DD_ERR_UNSUPPORTED, "feature channels must be positive multiples of 8");
    // the FPN's adaptive_avg_pool2d (reference head :121) is the identity only for exact 2x pyramids; otherwise the
    // ConvT output (2x the coarser level) is average-pooled down to the lateral's size by a dedicated kernel
    if (i > 0 && (p.H[i - 1] != 2 * p.H[i] || p.W[i - 1] != 2 * p.W[i])) {
      p.resample = true;
      if (p.H[i - 1] > 2 * p.H[i] || p.W[i - 1] > 2 * p.W[i])
        return fail(DD_ERR_UNSUPPORTED, "feature pyramid level is more than 2x its coarser neighbour");
    }
  }
  if (p.H[0] != h->cfg.cond_h || p.W[0] != h->cfg.cond_w)
    return fail(DD_ERR_INVALID, "level-0 feature size must equal the condition map size");
  h->prod = p;
  h->weights_ready = false;  // producer weights are packed by dd_finalize_weights
  h->ws = nullptr;           // workspace layout changed
  drop_graphs(h);
  return DD_OK;
}

int dd_build_condition(dd_handle h, const float* const* feats, float* cond_out, void* workspace, size_t workspace_bytes,
                       void* cuda_stream) {
  if (!h) return fail(DD_ERR_INVALID, "null argument");
  if (!feats && !h->feats_ready) return fail(DD_ERR_INVALID, "feats is NULL but dd_run_backbone has not run");
  if (!h->prod.enabled || !h->weights_ready || !h->prod.ready)
    return fail(DD_ERR_INVALID, "producers not enabled / weights not finalized");
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  int rc;
  if ((rc = bind_workspace(h, workspace, workspace_bytes))) return rc;
  Producers& p = h->prod;
  const int B = h->cfg.batch;
  if (feats) {
    CUDA_TRY(cudaMemsetAsync(h->status, 0, 64, st));
    h->launches = 0;
  }  // else: dd_run_backbone already wrote the input planes F[i] (and owns the status / launch counters)
  h->feats_ready = false;
  for (int i = 0; feats && i < p.nlev; ++i) {
    if (!feats[i]) return fail(DD_ERR_INVALID, "null feature map");
    const int P = p.H[i] * p.W[i];
    dim3 grid((P + 31) / 32, (p.C[i] + 31) / 32, B), block(32, 8);
    dd::nchw_to_nhwc_split_kernel<<<grid, block, 0, st>>>(feats[i], p.F[i].hi, p.F[i].lo, p.C[i], P, kProdScale, h->status);
    h->launches++;
  }
  CUDA_TRY(cudaGetLastError());
  auto build = [&](cudaStream_t s) -> int {
  const Planes none;
  for (int i = 0; i < p.nlev; ++i) {
    if (!p.neck) {
      p.O[i] = p.F[i];
      continue;
    }
    // HAHI neck, attention gates off (reference necks/hahi.py:173-176, 226-250, 253-272)
    if ((rc = run_gen(h, p.lat[i], p.F[i], p.C[i], none, 0, p.H[i], p.W[i], nullptr, nullptr, &p.L[i], s))) return rc;
    if ((rc = run_gen(h, p.proj[i], p.L[i], p.C[i], none, 0, p.H[i], p.W[i], nullptr, nullptr, &p.P[i], s))) return rc;
    if (i == 0) {  // cat([conv_proj(lat), lat])
      if ((rc = run_gen(h, p.fus[i], p.P[i], 512, p.L[i], p.C[i], p.H[i], p.W[i], nullptr, nullptr, &p.O[i], s))) return rc;
    } else {       // cat([lat, trans_proj(lat)])
      if ((rc = run_gen(h, p.fus[i], p.L[i], p.C[i], p.P[i], 512, p.H[i], p.W[i], nullptr, nullptr, &p.O[i], s))) return rc;
    }
  }
  // FPN top-down (reference head :112-122): x_i = relu(bn(conv3x3(O_i))) + relu(bn(convT2x2(x_{i+1})))
  for (int i = p.nlev - 1; i >= 0; --i) {
    const float* add = (i < p.nlev - 1) ? p.UP[i] : nullptr;
    if ((rc = run_gen(h, p.fl[i], p.O[i], p.C[i], none, 0, p.H[i], p.W[i], p.X[i], add, i > 0 ? &p.XP[i] : nullptr, s)))
      return rc;
    if (i > 0) {
      float* up_raw = p.resample ? p.UPR[i - 1] : p.UP[i - 1];
      if ((rc = run_gen(h, p.fu[i - 1], p.XP[i], 256, none, 0, p.H[i], p.W[i], up_raw, nullptr, nullptr, s))) return rc;
      if (p.resample) {  // F.adaptive_avg_pool2d(conv_up(pre_x), output_size = lateral size)  (reference head :121)
        const size_t n = static_cast<size_t>(B) * p.H[i - 1] * p.W[i - 1] * 256;
        int blocks = static_cast<int>((n + 255) / 256);
        if (blocks > 148 * 16) blocks = 148 * 16;
        dd::adaptive_avg_pool_nhwc_kernel<<<blocks, 256, 0, s>>>(up_raw, p.UP[i - 1], B, 2 * p.H[i], 2 * p.W[i], p.H[i - 1],
                                                                 p.W[i - 1], 256);
        h->launches++;
        CUDA_TRY(cudaGetLastError());
      }
    }
  }
  return DD_OK;
  };
  // every pointer of the neck / FPN kernels lives in the workspace -> replayable as a graph
  if (h->cfg.flags & DD_FLAG_CUDA_GRAPH) {
    if ((rc = graph_run(h, dd_engine::G_COND, st, build))) return rc;
  } else if ((rc = build(st))) {
    return rc;
  }
  h->cond_ready = true;
  if (cond_out) {
    if ((rc = transpose_out(h->cond, cond_out, B, 256, p.H[0] * p.W[0], st))) return rc;
    h->launches++;
  }
  return DD_OK;
}

int dd_enable_backbone(dd_handle h, const dd_backbone_config* bc) {
  if (!h || !bc) return fail(DD_ERR_INVALID, "null argument");
  if (bc->kind == DD_BACKBONE_RESNET) {
    if (!h->prod.enabled || h->prod.neck || h->prod.nlev != 4)
      return fail(DD_ERR_INVALID, "dd_enable_producers (4 levels, no neck) must be called first");
    ResNetW r;
    r.enabled = true;
    r.H = bc->height;
    r.W = bc->width;
    int hh = bc->height, ww = bc->width;
    for (int s = 0; s < 4; ++s) {
      r.depths[s] = bc->depths[s];
      if (r.depths[s] < 1) return fail(DD_ERR_INVALID, "bad ResNet depth");
      hh = (hh - 1) / 2 + 1;  // 3x3, stride 2, pad 1
      ww = (ww - 1) / 2 + 1;
      r.Hs[s] = hh;
      r.Ws[s] = ww;
      if (hh != h->prod.H[s] || ww != h->prod.W[s] || r.C[s] != h->prod.C[s])
        return fail(DD_ERR_INVALID, "backbone stage geometry does not match the producer pyramid");
    }
    h->rn = r;
    h->bb.enabled = false;
    h->mp.enabled = false;
    h->weights_ready = false;
    h->ws = nullptr;
    drop_graphs(h);
    return DD_OK;
  }
  if (bc->kind == DD_BACKBONE_MPVIT) {
    if (!h->prod.enabled || h->prod.nlev != 4)
      return fail(DD_ERR_INVALID, "dd_enable_producers (4 levels) must be called first");
    MPViTW m;
    m.enabled = true;
    m.H = bc->height;
    m.W = bc->width;
    m.heads = 8;  // every MPViT variant (reference mpvit.py:743-870)
    m.mlp_ratio = bc->mlp_ratio;
    if (m.mlp_ratio < 1 || m.mlp_ratio > 8) return fail(DD_ERR_INVALID, "bad MPViT mlp_ratio");
    int hh = bc->height, ww = bc->width;
    for (int s = 0; s < 4; ++s) {
      m.dims[s] = bc->mp_dims[s];
      m.layers[s] = bc->depths[s];
      m.paths[s] = bc->mp_paths[s];
      if (m.layers[s] < 1 || m.paths[s] < 1 || m.paths[s] > 3) return fail(DD_ERR_UNSUPPORTED, "MPViT: 1..3 paths, >= 1 layer per stage");
      if (m.dims[s] <= 0 || m.dims[s] % 8 != 0 || m.dims[s] / m.heads > dd::KTV_CH_MAX || m.dims[s] > 512)
        return fail(DD_ERR_UNSUPPORTED, "MPViT: stage widths must be multiples of 8 (8 heads), at most 512");
      hh = (hh - 1) / 2 + 1;  // depthwise 3x3, stride 2, pad 1
      ww = (ww - 1) / 2 + 1;
      m.Hs[s] = hh;
      m.Ws[s] = ww;
    }
    if (m.dims[0] % 16 != 0) return fail(DD_ERR_UNSUPPORTED, "MPViT: stem width must be a multiple of 16");
    for (int s = 0; s < 4; ++s) {
      m.out_dims[s] = s < 3 ? m.dims[s + 1] : m.dims[s];
      if (m.Hs[s] != h->prod.H[s] || m.Ws[s] != h->prod.W[s] || m.out_dims[s] != h->prod.C[s])
        return fail(DD_ERR_INVALID, "backbone stage geometry does not match the producer pyramid");
    }
    h->mp = m;
    h->bb.enabled = false;
    h->rn.enabled = false;
    h->weights_ready = false;
    h->ws = nullptr;
    drop_graphs(h);
    return DD_OK;
  }
  if (bc->kind != DD_BACKBONE_SWIN) return fail(DD_ERR_UNSUPPORTED, "unknown backbone kind");
  if (!h->prod.enabled || h->prod.nlev != 4)
    return fail(DD_ERR_INVALID, "dd_enable_producers (4 levels) must be called first");
  if (bc->embed_dims != 192 || bc->window != 7)
    return fail(DD_ERR_UNSUPPORTED, "native Swin is instantiated for embed_dims 192 (Swin-L), window 7");
  Backbone b;
  b.enabled = true;
  b.E = bc->embed_dims;
  b.window = bc->window;
  b.H = bc->height;
  b.W = bc->width;
  int hh = (bc->height + 3) / 4, ww = (bc->width + 3) / 4;
  for (int s = 0; s < 4; ++s) {
    b.depths[s] = bc->depths[s];
    b.heads[s] = bc->num_heads[s];
    if (b.depths[s] < 1 || (b.E << s) != 32 * b.heads[s]) return fail(DD_ERR_UNSUPPORTED, "Swin head_dim must be 32");
    b.Hs[s] = hh;
    b.Ws[s] = ww;
    if (hh != h->prod.H[s] || ww != h->prod.W[s] || (b.E << s) != h->prod.C[s])
      return fail(DD_ERR_INVALID, "backbone stage geometry does not match the producer pyramid");
    hh = (hh + 1) / 2;
    ww = (ww + 1) / 2;
  }
  h->bb = b;
  h->rn.enabled = false;
  h->mp.enabled = false;
  h->weights_ready = false;
  h->ws = nullptr;
  drop_graphs(h);
  return DD_OK;
}

int dd_run_backbone(dd_handle h, const float* rgb, float* const* feats_out, void* workspace, size_t workspace_bytes,
                    void* cuda_stream) {
  if (!h || !rgb) return fail(DD_ERR_INVALID, "null argument");
  const bool swin = h->bb.enabled && h->bb.ready, resnet = h->rn.enabled && h->rn.ready, mpvit = h->mp.enabled && h->mp.ready;
  if (!h->weights_ready || !(swin || resnet || mpvit)) return fail(DD_ERR_INVALID, "backbone not enabled / weights not finalized");
  auto run = [&](const float* img, float* const* outs, cudaStream_t s) {
    return swin ? run_swin(h, img, outs, s) : (resnet ? run_resnet(h, img, outs, s) : run_mpvit(h, img, outs, s));
  };
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  int rc;
  if ((rc = bind_workspace(h, workspace, workspace_bytes))) return rc;
  CUDA_TRY(cudaMemsetAsync(h->status, 0, 64, st));
  h->launches = 0;
  bool want_out = false;
  for (int i = 0; feats_out && i < 4; ++i) want_out |= (feats_out[i] != nullptr);
  if ((h->cfg.flags & DD_FLAG_CUDA_GRAPH) && !want_out) {
    // the graph's kernels read the image from the workspace: stage the caller's batch there first (20 MB at C3)
    const size_t n = static_cast<size_t>(h->cfg.batch) * 3 *
                     (swin ? h->bb.H * h->bb.W : (resnet ? h->rn.H * h->rn.W : h->mp.H * h->mp.W));
    CUDA_TRY(cudaMemcpyAsync(h->rgb_stage, rgb, n * 4, cudaMemcpyDeviceToDevice, st));
    if ((rc = graph_run(h, dd_engine::G_BACKBONE, st, [&](cudaStream_t s) { return run(h->rgb_stage, nullptr, s); }))) return rc;
  } else if ((rc = run(rgb, feats_out, st))) {
    return rc;
  }
  h->feats_ready = true;
  return DD_OK;
}

// Debug / tuning aid: time the GEMM-mode kernel on synthetic planes.  mode: 0 fp32 out, 1 fp32 out + residual add,
// 2 GELU -> planes, 3 no output at all (mainloop + TMEM drain only).
int dd_bench_gemm(dd_handle h, int32_t M, int32_t K, int32_t N, int32_t mode, int32_t iters, float* ms_out) {
  if (!h || !ms_out || M < 1 || K % dd::GEN_BK || N % 192 && N % 256) return fail(DD_ERR_INVALID, "bad argument");
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  cudaStream_t st = h->cap_stream;
  const size_t Mp = (static_cast<size_t>(M) + 127) / 128 * 128 + 128;
  Planes A, O;
  Gemm G;
  float *y = nullptr, *bias = nullptr;
  int* status = nullptr;
  CUDA_TRY(cudaMalloc(&A.hi, Mp * K * 2));
  CUDA_TRY(cudaMalloc(&A.lo, Mp * K * 2));
  CUDA_TRY(cudaMalloc(&O.hi, Mp * N * 2));
  CUDA_TRY(cudaMalloc(&O.lo, Mp * N * 2));
  CUDA_TRY(cudaMalloc(&y, Mp * N * 4));
  CUDA_TRY(cudaMalloc(&G.w_hi, static_cast<size_t>(N) * K * 2));
  CUDA_TRY(cudaMalloc(&G.w_lo, static_cast<size_t>(N) * K * 2));
  CUDA_TRY(cudaMalloc(&bias, N * 4));
  CUDA_TRY(cudaMalloc(&status, 64));
  CUDA_TRY(cudaMemsetAsync(A.hi, 0x11, Mp * K * 2, st));
  CUDA_TRY(cudaMemsetAsync(A.lo, 0x01, Mp * K * 2, st));
  CUDA_TRY(cudaMemsetAsync(G.w_hi, 0x11, static_cast<size_t>(N) * K * 2, st));
  CUDA_TRY(cudaMemsetAsync(G.w_lo, 0x01, static_cast<size_t>(N) * K * 2, st));
  CUDA_TRY(cudaMemsetAsync(bias, 0, N * 4, st));
  CUDA_TRY(cudaMemsetAsync(y, 0, Mp * N * 4, st));
  G.K = K;
  G.N = N;
  G.nt = (N % 256 == 0) ? 256 : 192;
  G.bias = bias;
  G.wscale = 1.f;
  int rc;
  if ((rc = make_wgen_map(&G.mb_hi, G.w_hi, N, K, 1, G.nt))) return rc;
  if ((rc = make_wgen_map(&G.mb_lo, G.w_lo, N, K, 1, G.nt))) return rc;
  if ((rc = make_wgen_map(&G.mp_hi, G.w_hi, N, K, 1, G.nt / 2))) return rc;
  if ((rc = make_wgen_map(&G.mp_lo, G.w_lo, N, K, 1, G.nt / 2))) return rc;
  int* saved = h->status;
  h->status = status;
  auto once = [&]() {
    return run_gemm(h, G, A, M, mode == 2 ? 2 : 0, (mode == 0 || mode == 1) ? y : nullptr, mode == 1 ? y : nullptr,
                    mode == 2 ? &O : nullptr, st);
  };
  for (int i = 0; i < 3; ++i)
    if ((rc = once())) return rc;
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0));
  CUDA_TRY(cudaEventCreate(&e1));
  CUDA_TRY(cudaEventRecord(e0, st));
  for (int i = 0; i < iters; ++i)
    if ((rc = once())) return rc;
  CUDA_TRY(cudaEventRecord(e1, st));
  CUDA_TRY(cudaEventSynchronize(e1));
  float ms = 0.f;
  CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
  *ms_out = ms / iters;
  h->status = saved;
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  for (void* p : {(void*)A.hi, (void*)A.lo, (void*)O.hi, (void*)O.lo, (void*)y, (void*)G.w_hi, (void*)G.w_lo, (void*)bias, (void*)status})
    cudaFree(p);
  return DD_OK;
}

int dd_encode(dd_handle h, const float* depth, int32_t height, int32_t width, float* latent_out, void* cuda_stream) {
  if (!h || !depth || !latent_out) return fail(DD_ERR_INVALID, "null argument");
  if (!h->weights_ready || !h->enc_w1) return fail(DD_ERR_INVALID, "encoder weights (depth_transform.conv_transform.*) not registered");
  if ((height + 1) / 2 != h->cfg.latent_h || (width + 1) / 2 != h->cfg.latent_w)
    return fail(DD_ERR_INVALID, "depth map size does not match the engine's latent grid");
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  dd::EncoderArgs a;
  a.depth = depth;
  a.w1 = h->enc_w1;
  a.b1 = h->enc_b1;
  a.w2 = h->enc_w2;
  a.b2 = h->enc_b2;
  a.out = latent_out;
  a.H = height;
  a.W = width;
  a.h = h->cfg.latent_h;
  a.w = h->cfg.latent_w;
  dim3 grid((a.w + 15) / 16, (a.h + 15) / 16, h->cfg.batch);
  dd::encoder_kernel<<<grid, 256, 0, st>>>(a);
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) return fail(DD_ERR_CUDA, std::string("encoder: ") + cudaGetErrorString(err));
  return DD_OK;
}

int64_t dd_last_launch_count(dd_handle h) { return h ? h->launches : 0; }

int dd_poll_status(dd_handle h, void* cuda_stream) {
  if (!h) return fail(DD_ERR_INVALID, "null handle");
  if (!h->status) return DD_OK;  // nothing has run yet
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  return poll_status(h, static_cast<cudaStream_t>(cuda_stream));
}

// ---------------------------------------------------------------- standalone conv (tests / roofline)
size_t dd_conv3x3_workspace_bytes(int32_t batch, int32_t cin, int32_t cout, int32_t height, int32_t width) {
  const size_t BP = static_cast<size_t>(batch) * height * width;
  const size_t nw = static_cast<size_t>(cin) * cout * 9;
  size_t off = 0;
  auto add = [&](size_t bytes) { off = align_up(off, 1024) + bytes; };
  add(64);            // status + scratch
  add(BP * cin * 4);  // x nhwc
  add(BP * cin * 2);  // hi
  add(BP * cin * 2);  // lo
  add(BP * cout * 4); // y nhwc
  add(nw * 2);
  add(nw * 2);
  add(nw * 4);
  add(static_cast<size_t>(9) * 128 * cin * 2);  // swapped-operand weight tile
  return align_up(off, 1024);
}

int dd_conv3x3(dd_handle h, const float* x, const float* w, const float* b, float* y, int32_t batch, int32_t cin,
               int32_t cout, int32_t height, int32_t width, void* workspace, size_t workspace_bytes, void* cuda_stream) {
  if (!h || !x || !w || !b || !y) return fail(DD_ERR_INVALID, "null argument");
  const int sid = shape_id(cin, cout);
  if (sid < 0) return fail(DD_ERR_UNSUPPORTED, "conv shape not on the DiffusionDepth hot path");
  if (workspace_bytes < dd_conv3x3_workspace_bytes(batch, cin, cout, height, width) ||
      (reinterpret_cast<uintptr_t>(workspace) & 1023))
    return fail(DD_ERR_INVALID, "conv workspace too small or misaligned");
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  const size_t BP = static_cast<size_t>(batch) * height * width;
  const size_t nw = static_cast<size_t>(cin) * cout * 9;
  Carver c{reinterpret_cast<uint8_t*>(workspace)};
  int* status = c.take<int>(16);
  float* xn = c.take<float>(BP * cin);
  __half* hi = c.take<__half>(BP * cin);
  __half* lo = c.take<__half>(BP * cin);
  float* yn = c.take<float>(BP * cout);
  __half* whi = c.take<__half>(nw);
  __half* wlo = c.take<__half>(nw);
  float* wsimt = c.take<float>(nw);
  __half* wswap = c.take<__half>(static_cast<size_t>(9) * 128 * cin);
  CUDA_TRY(cudaMemsetAsync(status, 0, 64, st));
  int rc;
  if ((rc = transpose_in(x, xn, batch, cin, height * width, st))) return rc;
  float* amax_dev = reinterpret_cast<float*>(status) + 8;
  dd::absmax_kernel<<<absmax_grid(BP * cin), 256, 0, st>>>(xn, static_cast<int>(std::min<size_t>(BP * cin, 1u << 30)), amax_dev);  // zeroed with status
  dd::absmax_kernel<<<absmax_grid(nw), 256, 0, st>>>(w, static_cast<int>(nw), amax_dev + 1);
  float am[2] = {0.f, 0.f};
  CUDA_TRY(cudaMemcpyAsync(am, amax_dev, 8, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  auto pow2_scale = [](float amax) {
    return (amax > 0.f && isfinite(amax)) ? exp2f(floorf(log2f(32768.f / amax)) - 1.f) : 1.f;
  };
  const float sx = pow2_scale(am[0]), sw = pow2_scale(am[1]);
  dd::split_planes_kernel<<<148 * 8, 256, 0, st>>>(xn, hi, lo, BP * cin / 4, sx, status);
  dd::pack_conv_weight_kernel<<<128, 256, 0, st>>>(w, whi, wlo, wsimt, cout, cin, sw);
  CUDA_TRY(cudaGetLastError());
  dd::ConvArgs a;
  a.B = batch;
  a.H = height;
  a.W = width;
  a.tiles_x = (width + dd::TILE_W - 1) / dd::TILE_W;
  a.tiles_y = (height + dd::TILE_H - 1) / dd::TILE_H;
  a.num_tiles = a.tiles_x * a.tiles_y * batch;
  a.bias = b;
  a.acc_scale = 1.f / (sx * sw);
  a.y32 = yn;
  a.stats_partial = nullptr;
  a.out_hi = nullptr;
  a.out_lo = nullptr;
  a.out_a8 = a.out_l8 = nullptr;
  a.split_scale = 1.f;
  a.status = status;
  a.fp8_probe = 0;
  a.clk_probe = nullptr;
  cudaError_t err = cudaSuccess;
  const ShapeInfo s = kShapes[sid];
  if (h->cfg.flags & DD_FLAG_SIMT_CONV) {
    dd::SimtArgs sa;
    sa.in_hi = hi;
    sa.in_lo = lo;
    sa.in_inv_scale = 1.f / sx;
    sa.w = wsimt;
    sa.c = a;
    switch (sid) {
      case 0: err = launch_simt<16, 64, dd::EPI_F32>(sa, st); break;
      case 1: err = launch_simt<64, 256, dd::EPI_F32>(sa, st); break;
      case 2: err = launch_simt<256, 256, dd::EPI_F32>(sa, st); break;
      case 3: err = launch_simt<256, 64, dd::EPI_F32>(sa, st); break;
      case 4: err = launch_simt<64, 16, dd::EPI_F32>(sa, st); break;
    }
  } else if ((h->cfg.flags & DD_FLAG_SWAP_NARROW) && kSwapBK[sid] > 0) {
    CUtensorMap mp_hi, mp_lo, mw;
    const int bk = kSwapBK[sid];
    a.tiles_x = (width + dd::SWAP_TW - 1) / dd::SWAP_TW;
    a.tiles_y = (height + dd::SWAP_TH - 1) / dd::SWAP_TH;
    a.num_tiles = a.tiles_x * a.tiles_y * batch;
    __half* wsw = wswap;
    dd::pack_swap_weight_kernel<<<128, 256, 0, st>>>(w, wsw, cout, cin, sw);
    CUDA_TRY(cudaGetLastError());
    const bool swap_halo = (h->cfg.flags & DD_FLAG_HALO_CONV) && bk == 32 && h->swaphalo_mask != 0;
    if (swap_halo) {
      if ((rc = make_swap_strip_map(&mp_hi, hi, batch, height, width, cin, bk))) return rc;
      if ((rc = make_swap_strip_map(&mp_lo, lo, batch, height, width, cin, bk))) return rc;
    } else {
      if ((rc = make_patch_map(&mp_hi, hi, batch, height, width, cin, bk))) return rc;
      if ((rc = make_patch_map(&mp_lo, lo, batch, height, width, cin, bk))) return rc;
    }
    if ((rc = make_w_map(&mw, wsw, 128, cin, bk))) return rc;
    if (swap_halo) {
      err = sid == 3 ? launch_swap<256, 64, 32, dd::EPI_F32, true>(mp_hi, mp_lo, mw, a, h->sm_count, st)
                     : launch_swap<64, 16, 32, dd::EPI_F32, true>(mp_hi, mp_lo, mw, a, h->sm_count, st);
    } else
    switch (sid) {
      case 0: err = launch_swap<16, 64, 16, dd::EPI_F32>(mp_hi, mp_lo, mw, a, h->sm_count, st); break;
      case 3: err = launch_swap<256, 64, 32, dd::EPI_F32>(mp_hi, mp_lo, mw, a, h->sm_count, st); break;
      case 4: err = launch_swap<64, 16, 32, dd::EPI_F32>(mp_hi, mp_lo, mw, a, h->sm_count, st); break;
    }
  } else if (fp8_active(h) && cin == 256 && cout == 256) {
    // fp8-correction kernel on a standalone layer (tests): the e4m3 planes reuse the fp16 lo plane's storage, the
    // weight planes that of the SIMT copy; x is re-split with a scale that keeps |s x| / 4 inside e4m3
    const float sx8 = (am[0] > 0.f && isfinite(am[0])) ? exp2f(floorf(log2f(1024.f / am[0]))) : 1.f;
    uint8_t* a8 = reinterpret_cast<uint8_t*>(lo);
    uint8_t* l8 = a8 + BP * cin;
    uint8_t* w8 = reinterpret_cast<uint8_t*>(wsimt);
    uint8_t* lw8 = w8 + nw;
    dd::split_planes8_kernel<<<148 * 8, 256, 0, st>>>(xn, hi, a8, l8, BP * cin / 8, sx8, status);
    dd::pack_conv_weight8_kernel<<<128, 256, 0, st>>>(w, w8, lw8, cout, cin, sw);
    CUDA_TRY(cudaGetLastError());
    a.acc_scale = 1.f / (sx8 * sw);
    a.tiles_x = (width + dd::HALO_TW - 1) / dd::HALO_TW;
    a.tiles_y = (height + dd::HALO_TH - 1) / dd::HALO_TH;
    a.num_tiles = a.tiles_x * a.tiles_y * batch;
    CUtensorMap ma_hi, m_a8, m_l8, mb_hi, m_w8, m_lw8;
    if ((rc = make_strip_map(&ma_hi, hi, batch, height, width, cin, 64))) return rc;
    if ((rc = make_strip_map8(&m_a8, a8, batch, height, width, cin))) return rc;
    if ((rc = make_strip_map8(&m_l8, l8, batch, height, width, cin))) return rc;
    if ((rc = make_w_map(&mb_hi, whi, cout, cin, 64, cout / 2))) return rc;
    if ((rc = make_w_map8(&m_w8, w8, cout, cin, cout / 2))) return rc;
    if ((rc = make_w_map8(&m_lw8, lw8, cout, cin, cout / 2))) return rc;
    err = launch_pair<256, 256, 64, dd::EPI_F32, true>(ma_hi, m_a8, mb_hi, m_w8, a, h->sm_count, st, &m_l8, &m_lw8);
  } else if (h->cfg.flags & DD_FLAG_HALO_CONV) {
    CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
    const int hbk = kHaloBK[sid];
    a.tiles_x = (width + dd::HALO_TW - 1) / dd::HALO_TW;
    a.tiles_y = (height + dd::HALO_TH - 1) / dd::HALO_TH;
    a.num_tiles = a.tiles_x * a.tiles_y * batch;
    if ((rc = make_strip_map(&ma_hi, hi, batch, height, width, cin, hbk))) return rc;
    if ((rc = make_strip_map(&ma_lo, lo, batch, height, width, cin, hbk))) return rc;
    const bool pair = (h->cfg.flags & DD_FLAG_PAIR_WIDE) && cout == 256;
    if ((rc = make_w_map(&mb_hi, whi, cout, cin, hbk, pair ? cout / 2 : 0))) return rc;
    if ((rc = make_w_map(&mb_lo, wlo, cout, cin, hbk, pair ? cout / 2 : 0))) return rc;
    if (pair) {
      err = sid == 1 ? launch_pair<64, 256, 32, dd::EPI_F32>(ma_hi, ma_lo, mb_hi, mb_lo, a, h->sm_count, st)
                     : launch_pair<256, 256, 32, dd::EPI_F32>(ma_hi, ma_lo, mb_hi, mb_lo, a, h->sm_count, st);
    } else
    switch (sid) {
      case 0: err = launch_halo<16, 64, 16, dd::EPI_F32>(ma_hi, ma_lo, mb_hi, mb_lo, a, h->sm_count, st); break;
      case 1: err = launch_halo<64, 256, 32, dd::EPI_F32>(ma_hi, ma_lo, mb_hi, mb_lo, a, h->sm_count, st); break;
      case 2: err = launch_halo<256, 256, 32, dd::EPI_F32>(ma_hi, ma_lo, mb_hi, mb_lo, a, h->sm_count, st); break;
      case 3: err = launch_halo<256, 64, 32, dd::EPI_F32>(ma_hi, ma_lo, mb_hi, mb_lo, a, h->sm_count, st); break;
      case 4: err = launch_halo<64, 16, 32, dd::EPI_F32>(ma_hi, ma_lo, mb_hi, mb_lo, a, h->sm_count, st); break;
    }
  } else {
    CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
    if ((rc = make_act_map(&ma_hi, hi, batch, height, width, cin, s.bk))) return rc;
    if ((rc = make_act_map(&ma_lo, lo, batch, height, width, cin, s.bk))) return rc;
    if ((rc = make_w_map(&mb_hi, whi, cout, cin, s.bk))) return rc;
    if ((rc = make_w_map(&mb_lo, wlo, cout, cin, s.bk))) return rc;
    switch (sid) {
      case 0: err = launch_umma<16, 64, 16, dd::EPI_F32>(ma_hi, ma_lo, mb_hi, mb_lo, a, h->sm_count, st); break;
      case 1: err = launch_umma<64, 256, 32, dd::EPI_F32>(ma_hi, ma_lo, mb_hi, mb_lo, a, h->sm_count, st); break;
      case 2: err = launch_umma<256, 256, 32, dd::EPI_F32>(ma_hi, ma_lo, mb_hi, mb_lo, a, h->sm_count, st); break;
      case 3: err = launch_umma<256, 64, 64, dd::EPI_F32>(ma_hi, ma_lo, mb_hi, mb_lo, a, h->sm_count, st); break;
      case 4: err = launch_umma<64, 16, 64, dd::EPI_F32>(ma_hi, ma_lo, mb_hi, mb_lo, a, h->sm_count, st); break;
    }
  }
  if (err != cudaSuccess) return fail(DD_ERR_CUDA, std::string("conv launch: ") + cudaGetErrorString(err));
  return transpose_out(yn, y, batch, cout, height * width, st);
}

int dd_bench_conv(dd_handle h, int32_t cin, int32_t cout, int32_t iters, float* ms_out, void* workspace,
                  size_t workspace_bytes, void* cuda_stream) {
  if (!h || !ms_out || iters < 1) return fail(DD_ERR_INVALID, "bad argument");
  if (!h->weights_ready) return fail(DD_ERR_INVALID, "dd_finalize_weights has not been called");
  cudaStream_t st = static_cast<cudaStream_t>(cuda_stream);
  CUDA_TRY(cudaSetDevice(h->cfg.device));
  int rc;
  if ((rc = bind_workspace(h, workspace, workspace_bytes))) return rc;
  int layer = -1;
  for (int i = 0; i < 6; ++i)
    if (h->L[i].sid >= 0 && kShapes[h->L[i].sid].cin == cin && kShapes[h->L[i].sid].cout == cout) layer = i;
  if (layer < 0) return fail(DD_ERR_UNSUPPORTED, "no packed layer with that shape in this engine variant");
  const bool split_out = (cin == 256 && cout == 256);
  const int f8 = ((split_out || (cin == 64 && cout == 256 && h->f8_ne3)) && fp8_active(h)) ? kF8In : 0;  // time the kernel the loop actually runs
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0));
  CUDA_TRY(cudaEventCreate(&e1));
  // whatever the planes currently hold is fine for timing: MMA time is data independent
  const __half* in_hi = cin == 16 ? h->xs_hi : h->S_hi[1];
  const __half* in_lo = cin == 16 ? h->xs_lo : h->S_lo[1];
  for (int w = 0; w < 2; ++w)
    if ((rc = run_conv(h, layer, in_hi, in_lo, kActScale, split_out ? dd::EPI_SPLIT : dd::EPI_F32_STATS, h->Y,
                       h->stats[0], h->S_hi[0], h->S_lo[0], st, f8)))
      return rc;
  if (h->want_clk_probe && !h->clk_probe) CUDA_TRY(cudaMalloc(&h->clk_probe, 16));
  if (h->clk_probe) CUDA_TRY(cudaMemsetAsync(h->clk_probe, 0, 16, st));
  CUDA_TRY(cudaEventRecord(e0, st));
  for (int i = 0; i < iters; ++i)
    if ((rc = run_conv(h, layer, in_hi, in_lo, kActScale, split_out ? dd::EPI_SPLIT : dd::EPI_F32_STATS, h->Y,
                       h->stats[0], h->S_hi[0], h->S_lo[0], st, f8)))
      return rc;
  CUDA_TRY(cudaEventRecord(e1, st));
  CUDA_TRY(cudaEventSynchronize(e1));
  float ms = 0.f;
  CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (h->clk_probe) {
    unsigned long long v[2] = {0, 0};
    CUDA_TRY(cudaMemcpy(v, h->clk_probe, 16, cudaMemcpyDeviceToHost));
    if (v[1])
      fprintf(stderr, "[clk_probe] conv %d->%d: %.0f SM cycles, %.1f us per launch (CTA 0) => %.0f MHz\n", cin, cout,
              double(v[0]) / iters, double(v[1]) / iters * 1e-3, double(v[0]) / double(v[1]) * 1e3);
    cudaFree(h->clk_probe);
    h->clk_probe = nullptr;
  }
  *ms_out = ms / iters;
  return DD_OK;
}

}  // extern "C"
