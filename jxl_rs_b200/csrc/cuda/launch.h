// Host-side entry points into kernels.cu.
#pragma once
#include <cuda_runtime.h>

#include "device_types.h"

namespace jxgpu {
cudaError_t upload_constants(const float* wc, const float* rdct_scale);
cudaError_t configure_kernels();
// Enqueues the K1..K2 part of the pipeline on `stream`: block plan, entropy and transform kernels (debug_stop 1: the
// block plan and entropy kernels only); returns the number of kernel launches. lean_S (4 or 8) and lean_ctas come from
// the host's schedule of k_entropy_lean.
int launch_pipeline(const BatchDev& B, cudaStream_t stream, int debug_stop, cudaEvent_t* ev, bool lean_all_420,
                    uint32_t lean_S, uint32_t lean_ctas, bool lean_ctx_smem);
constexpr int kFusedTileW = 64, kFusedTileH = 32;
int launch_filter_range(const BatchDev& B, const uint32_t* fused_prefix, uint32_t tile_begin, uint32_t tile_count,
                        uint32_t filter_cfg_mask, cudaStream_t stream);
// Parity tap (jxg_batch_read_coeffs): lists of one frame -> dense [groups][3][65536] i32 (zeroed by the caller).
void launch_expand_coeffs(const BatchDev& B, uint32_t frame, uint32_t num_groups, int32_t* dense, cudaStream_t stream);
// Orientation post-pass of one frame: coded w x h image at `src` (row stride src_stride) -> display orientation at `dst`.
void launch_orient(const void* src, size_t src_stride, void* dst, size_t dst_stride, uint32_t w, uint32_t h, uint32_t bpp,
                   uint32_t orientation, cudaStream_t stream);
constexpr int kNumStages = 8;  // memset, entropy, dequant_idct, gaborish, epf0, epf1, epf2, xyb_store
}  // namespace jxgpu
