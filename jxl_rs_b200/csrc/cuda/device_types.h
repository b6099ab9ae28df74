// Device-visible layout of a decode batch. One "blob" (uploaded with a single
// H2D copy from pinned staging) carries every per-frame table and plane the
// kernels read; FrameDev holds byte offsets into it. Large intermediates
// (coefficients, XYB planes) live in separate device-only allocations.
#pragma once
#include <stdint.h>
#include <vector_types.h>

namespace jxgpu {

constexpr int kMaxPasses = 11;
constexpr uint32_t kGroupCoeffs = 65536;  // per channel per group (group.rs:53-55)

// Coefficients travel from the entropy kernels to the transform kernels as one list of NON-ZERO entries per
// (pass, group) stream, in decode order (varblocks in raster order, channels Y, X, B inside a varblock, coefficient
// order inside a channel). Entry of a varblock with 2^n coefficients per channel (n = 6 .. 16):
//     position in the storage layout (low n bits) | value << n (two's complement in the remaining 32 - n bits),
// i.e. +-2^25 for an 8x8 block down to +-2^15 for DCT256X256. A value outside that range is refused
// (JXG_ERR_UNSUPPORTED for the stream): quantised coefficients of that size do not occur in real streams, and refusing
// keeps both sides branch-free. Behind the entries (and 4 words of padding: the writer stores every decoded coefficient
// at the cursor and only advances it for non-zero ones) sit the offset words: offw[seq * 3 + ci] = index of the first
// entry of channel ci (0 = Y, 1 = X, 2 = B) of the seq-th varblock, offw[nblk * 3] = total. The dense
// [groups][3][65536] i32 array of round 1 (12 B/px written once, read once, >= 90 % zeros, plus a memset) is gone;
// a list is written and read sequentially.
// A pass of one group decodes at most 3 x 1024 non-zero counts + 3 x 65536 coefficients, fewer than the reference's
// 2^20-symbol LZ77 window: the window never wraps and is addressed linearly.
constexpr uint32_t kLzWindow = 3 * kGroupCoeffs + 3 * 1024;
constexpr uint32_t kListCap = 3 * kGroupCoeffs;        // entries: every coefficient of the group non-zero
constexpr uint32_t kListPad = 4;
constexpr uint32_t kOffBase = kListCap + kListPad;     // first offset word
constexpr uint32_t kOffWords = 3 * 1024 + 4;           // offsets of <= 1024 varblocks x 3 channels + end, 16-byte multiple
constexpr uint32_t kListStride = kOffBase + kOffWords;  // u32 words per list

struct PassDev {
  uint32_t shift, use_prefix, log_alpha_size, num_clusters;
  uint32_t lz77_enabled, lz77_min_symbol, lz77_min_length, lz77_length_uint, lz_dist_cluster;
  uint32_t custom_orders;
  uint64_t context_map_off;   // u8[]
  uint64_t uint_configs_off;  // u32[num_clusters]
  uint64_t ans_off;           // u64[num_clusters << log_alpha_size]
  uint64_t huff_off;          // u32[] entries
  uint64_t huff_offset_off;   // u32[num_clusters]
  uint64_t order_off;         // u32[] custom orders
  uint32_t order_offset[39];
};

struct FrameDev {
  uint32_t width, height, xb, yb, xg, yg, num_groups, num_passes;
  uint32_t plane_stride, plane_rows;     // padded XYB plane geometry (xb*8, yb*8)
  uint32_t cxb;                          // ceil(xb/8): CfL map stride
  // entropy / contexts
  uint32_t num_histograms, num_block_contexts, num_lf_contexts, num_qf_thresholds;
  uint32_t qf_thresholds[15];
  uint64_t block_ctx_map_off;
  PassDev passes[kMaxPasses];
  // dequant
  float inv_global_scale, x_dm, b_dm;
  float quant_biases[4];
  float base_correlation_x, base_correlation_b, inv_color_factor_unused;
  uint32_t color_factor;
  int64_t dequant_off[17];  // byte offset into blob, or -1 = library default table
  // planes in the blob
  uint64_t lf_off[3];  // f32 xb*yb
  uint64_t transform_off, raw_quant_off, epf_off, quant_lf_off, ytox_off, ytob_off;
  // HF sections: index of this frame's first section in the batch section table
  uint32_t section_base;
  uint32_t first_stream;      // index of group 0 in the batch stream list
  // persistent entropy lanes (k_entropy_lean): this frame's range in streams_lean (longest first) and its CTAs
  uint32_t lean_first, lean_count, lean_cta_first, lean_ctas;
  uint32_t lean_lanes;        // lanes of this frame that start with a stream of their own; the rest is queued
  // LZ77 inside the HF streams (entropy_coding/decode.rs:286-330): such frames take the one-lane-per-warp kernel and own
  // one window of decoded symbols per section in BatchDev::lzwin
  uint32_t has_lz, lz_win_base;
  // device-only buffers (element offsets)
  uint64_t coeff_group_base;  // group index base into coeffs
  uint64_t block_base;        // block index base into block_off
  uint64_t plane_base;        // float index base into plane sets (per channel: + c * plane_size)
  uint64_t plane_size;        // plane_stride * plane_rows
  uint64_t out_off;           // byte offset into device output buffer (or absolute pointer if out_is_ptr)
  uint64_t out_row_stride;
  void* out_ptr;              // device pointer for this frame's output
  // filters / colour
  uint32_t gab, epf_iters;
  float gab_k0[3], gab_k1[3], gab_k2[3];  // normalised weights (gaborish.rs:20-27)
  float epf_sharp_lut[8], epf_channel_scale[3];
  float epf_quant_mul, epf_pass0_sigma_scale, epf_pass2_sigma_scale, epf_border_sad_mul;
  float quant_scale;  // 1 / inv_global_scale (features/epf.rs:55)
  float opsin[9], bias_cbrt[3], scaled_bias[3], intensity_scale;
  uint32_t output_tf, output_format;
  float tf_gamma;        // JXG_TF_GAMMA exponent
  float tf_lum[3];       // JXG_TF_HLG: luminances of the output primaries
  float tf_hlg_exp;      // JXG_TF_HLG: (1 - system_gamma) / system_gamma (color/tf.rs:458-470), 0 = OOTF skipped
  float tf_pq_mul;       // JXG_TF_PQ: intensity_target / 10000
};

struct SectionDev {
  uint64_t off;  // byte offset in blob (8-byte aligned, zero padded)
  uint32_t len;
  uint32_t pad;
};

struct StreamDev {  // one (frame, group) unit of entropy-decode work
  uint32_t frame, group;
};

struct BatchDev {
  const uint8_t* blob;
  const FrameDev* frames;
  const SectionDev* sections;
  const StreamDev* streams;       // all (frame, group) units, ordered by frame then group
  const StreamDev* streams_lean;  // single-pass ANS frames: k_entropy_lean
  const StreamDev* streams_fast;  // single-pass prefix-coded frames: k_entropy_fast
  const StreamDev* streams_slow;  // multi-pass frames: k_entropy
  uint32_t num_frames, num_streams, num_lean, num_fast, num_slow;
  uint32_t* nzlist;     // [sections][kListStride]: list of section (pass * num_groups + group) of a frame, see above
  uint32_t* lzwin;      // [lz sections][kLzWindow] LZ77 windows (decode.rs:86-146), frames with has_lz only
  uint32_t* block_off;  // per 8x8 block: ordinal (raster order) of the varblock starting there within its group
  uint8_t* nz;          // [streams][passes][3][1024]
  uint64_t* nz_base;    // per stream offset into nz (bytes)
  float* planes_a;
  int32_t* status;      // per stream
  uint32_t* queue;      // [frames] work-queue cursors of the persistent entropy kernel
  const uint32_t* lean_cta_first;  // [frames] first CTA of each frame in k_entropy_lean's grid
  const uint2* lean_warp;          // [lean CTAs * 4] per warp: first stream (relative to the frame's list), lanes
  uint4* desc;           // [num_streams][1024] varblock descriptors written by k_block_plan
  uint32_t* nblk;        // [num_streams] varblocks per stream (0xffffffff: invalid transform id)
  // context-wide tables
  const float* dequant_default;       // 17 tables concatenated
  const uint32_t* dequant_default_off;  // [17] float offsets
  const uint32_t* natural_orders;     // 13 orders concatenated
  const uint32_t* natural_order_off;  // [13]
};

}  // namespace jxgpu
