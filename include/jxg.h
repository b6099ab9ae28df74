/*
 * jxg.h — C ABI of libjxgpu.so: the B200 (sm_100a) replacement for the
 * per-group VarDCT decode + render hot path of libjxl/jxl-rs.
 *
 * The reference crate exposes no FFI (jxl/src/lib.rs:6 `#![deny(unsafe_code)]`);
 * the seam these entry points sit behind is internal:
 *
 *   Frame::decode_and_render_hf_groups        jxl/src/frame/render.rs:143
 *     (fan-out `parallel_runner.run(...)`     jxl/src/frame/render.rs:461-479)
 *       -> Frame::decode_hf_group             jxl/src/frame/decode.rs:790
 *       -> decode_vardct_group                jxl/src/frame/group.rs:383
 *       -> render stages Gaborish/EPF/XYB/FromLinear/Convert/Save
 *                                             jxl/src/frame/render.rs:579-620,757-905
 *
 * A Rust host keeps doing what jxl-rs does today up to that point (container,
 * headers, TOC, LfGlobal, LfGroups, HfGlobal) and hands the parsed frame state
 * plus the raw HF section bytes to `jxg_batch_add_frame`. INTEGRATION.md shows
 * the `extern "C"` block a maintainer would add.
 *
 * Conventions: every function returns 0 (JXG_OK) or a negative JXG_ERR_*.
 * All pointers in a JxgFrameDesc are HOST pointers that must stay valid until
 * jxg_batch_add_frame returns (the library copies what it needs into pinned
 * staging memory). One host thread per context; distinct contexts are
 * independent. No torch types cross this boundary.
 */
#ifndef JXG_H_
#define JXG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define JXG_ABI_VERSION 2

/* Error codes; names mirror jxl/src/error.rs variants raised on this path. */
enum {
  JXG_OK = 0,
  JXG_ERR_BITSTREAM = -1,              /* generic malformed input (host front-end)  */
  JXG_ERR_UNSUPPORTED = -2,            /* feature outside the hot-path scope        */
  JXG_ERR_OUT_OF_BOUNDS = -3,          /* Error::OutOfBounds: section over-read     */
  JXG_ERR_INVALID_HISTOGRAM_INDEX = -4,/* Error::InvalidHistogramIndex group.rs:339 */
  JXG_ERR_INVALID_NUM_NONZEROS = -5,   /* Error::InvalidNumNonZeros   group.rs:544  */
  JXG_ERR_RESIDUAL_NONZEROS = -6,      /* Error::EndOfBlockResidualNonZeros :575    */
  JXG_ERR_ANS_CHECKSUM = -7,           /* Error::AnsChecksumMismatch  ans.rs:441    */
  JXG_ERR_INVALID_TRANSFORM = -8,      /* Error::InvalidVarDCTTransform             */
  JXG_ERR_INVALID_OUTPUT = -9,         /* Error::InvalidOutputBufferSize            */
  JXG_ERR_LZ77 = -10,                  /* UnexpectedLz77Repeat / ArithmeticOverflow */
  JXG_ERR_CUDA = -20,                  /* CUDA runtime failure                      */
  JXG_ERR_NO_DEVICE = -21,             /* no CUDA device: there is NO CPU fallback  */
  JXG_ERR_ARGUMENT = -22
};

/* Output pixel formats (JxlPixelFormat, jxl/src/api/data_types.rs:154). */
enum {
  JXG_FORMAT_RGB_U8 = 0,   /* interleaved sRGB-encoded u8, 3 B/px  (convert.rs:548) */
  JXG_FORMAT_RGBA_U8 = 1,  /* + opaque alpha 255 (fill_opaque_alpha, render.rs:858) */
  JXG_FORMAT_RGB_F32 = 2,  /* interleaved f32, 12 B/px; linear sRGB unless tf set   */
  JXG_FORMAT_XYB_F32_PLANAR = 3, /* debug/parity tap: the 3 XYB planes after filters */
  JXG_FORMAT_RGB_U16 = 4,  /* interleaved u16 (native endian), 6 B/px: clamp to [0,1], x 65535, round
                              (ConvertF32ToU16Stage, convert.rs:717-786, bit_depth 16; no dither) */
  JXG_FORMAT_RGB_F16 = 5   /* interleaved IEEE half, 6 B/px (ConvertF32ToF16Stage, convert.rs:789-857); PQ output
                              is clamped to [0,1], HLG to [-0.074, 1.1] first (frame/render.rs:746-750) */
};

/* Output transfer function (render/stages/from_linear.rs). */
enum {
  JXG_TF_LINEAR = 0, /* no curve (the reference adds no stage for a linear output, frame/render.rs:761)      */
  JXG_TF_SRGB = 1,   /* color/tf.rs:13-44                                                                     */
  JXG_TF_GAMMA = 2,  /* |v|^output_gamma, sign kept (from_linear.rs:97-109; DCI is gamma 1/2.6)               */
  JXG_TF_BT709 = 3,  /* color/tf.rs:114-150                                                                   */
  JXG_TF_PQ = 4,     /* color/tf.rs:261-304, 1.0 = intensity_target nits                                      */
  JXG_TF_HLG = 5     /* inverse OOTF with output_luminances, then the HLG OETF (color/tf.rs:458-470, 481-497) */
};

/* One entropy-coded histogram set + coefficient orders, per pass
 * (HfGlobalState.passes[i], jxl/src/frame/decode.rs:519-545). */
typedef struct JxgPassDesc {
  uint32_t shift;                 /* frame_header.passes.shift[pass] (group.rs:350) */
  uint32_t use_prefix;            /* 1: prefix codes, 0: ANS                         */
  uint32_t log_alpha_size;        /* ANS only: 5..8                                  */
  uint32_t num_clusters;
  uint32_t num_contexts;          /* length of context_map (incl. +16 padding)       */
  uint32_t lz77_enabled, lz77_min_symbol, lz77_min_length;
  uint32_t lz77_length_uint;      /* packed hybrid-uint config                       */
  uint32_t lz_dist_cluster;
  const uint8_t* context_map;     /* [num_contexts] context -> cluster (decode.rs:547)*/
  const uint32_t* uint_configs;   /* [num_clusters] split_exp | msb<<8 | lsb<<16     */
  const uint64_t* ans_buckets;    /* [num_clusters << log_alpha_size], ans.rs:31-39:
                                     alias_symbol u8 | alias_cutoff u8 <<8 | dist u16 <<16
                                     | alias_offset u16 <<32 | alias_dist_xor u16 <<48 */
  const uint32_t* huff_entries;   /* bits | value<<16, concatenated 2-level LUTs     */
  const uint32_t* huff_offset;    /* [num_clusters] start of each LUT                */
  uint32_t huff_entries_len;
  /* 13 shapes x 3 channels coefficient orders (coeff_order.rs:122). NULL = all
   * natural orders (used_orders == 0). Otherwise order i starts at
   * coeff_order_offset[i] (index = shape*3 + c). */
  const uint32_t* coeff_order;
  uint32_t coeff_order_offset[39];
  uint32_t coeff_order_len;
} JxgPassDesc;

typedef struct JxgFrameDesc {
  uint32_t abi_version;           /* JXG_ABI_VERSION                                  */
  uint32_t width, height;         /* frame_header.size() in pixels                    */
  /* ---- quantiser / CfL (LfGlobal) ---- */
  uint32_t global_scale;          /* quantizer.rs:55                                  */
  uint32_t x_qm_scale, b_qm_scale;/* group.rs:395-396                                 */
  float quant_biases[4];          /* transform_data.rs:30-31                          */
  float base_correlation_x, base_correlation_b; uint32_t color_factor; /* color_correlation_map.rs:21 */
  /* ---- block context map (block_context_map.rs:46-53) ---- */
  uint32_t num_qf_thresholds; uint32_t qf_thresholds[15];
  uint32_t num_lf_contexts;       /* product of (lf thresholds + 1)                   */
  uint32_t num_block_contexts;    /* max(ctx_map)+1, <= 16                            */
  uint32_t block_ctx_map_len;     /* 39 * (num_qf_thresholds+1) * num_lf_contexts     */
  const uint8_t* block_ctx_map;
  uint32_t num_histograms;        /* HfGlobal, frame/decode.rs:512                    */
  uint32_t num_passes;
  const JxgPassDesc* passes;      /* [num_passes]                                     */
  /* ---- dequant matrices (quant_weights.rs:1081): NULL entry = library default ---- */
  const float* dequant_tables[17];
  /* ---- per-frame planes, dimensions in 8x8 blocks: xb = ceil(width/8) ---- */
  const float* lf[3];             /* X, Y, B dequantised (and smoothed) LF, stride xb */
  const uint8_t* transform_map;   /* HfTransformType | 128 for first block of varblock*/
  const int32_t* raw_quant_map;   /* 1..256                                           */
  const uint8_t* epf_map;         /* sharpness 0..7                                   */
  const uint8_t* quant_lf;        /* LF context bucket per block (modular/mod.rs:895) */
  const int8_t* ytox_map;         /* ceil(xb/8) x ceil(yb/8)                          */
  const int8_t* ytob_map;
  /* ---- restoration filter (frame_header.rs:146-234) ---- */
  uint32_t gab;                   float gab_w1[3], gab_w2[3];   /* per X,Y,B */
  uint32_t epf_iters;
  float epf_sharp_lut[8]; float epf_channel_scale[3];
  float epf_quant_mul, epf_pass0_sigma_scale, epf_pass2_sigma_scale, epf_border_sad_mul;
  /* ---- colour (xyb.rs:145-241) ---- */
  float opsin_inverse_matrix[9]; float opsin_biases[3]; float intensity_target;
  uint32_t output_tf;             /* JXG_TF_*                                         */
  uint32_t output_format;         /* JXG_FORMAT_*                                     */
  /* ImageMetadata.orientation 1..8 (headers/image_metadata.rs:41-50), applied by the store as the reference's save stage
   * does (render/save.rs, api/options.rs:39 adjust_orientation = true): the output buffer holds the image in display
   * orientation, i.e. height x width swap for values 5..8. The XYB debug tap ignores it. */
  uint32_t orientation;
  /* Output encoding as OutputColorInfo::from_header derives it (render/stages/xyb.rs:65-140): opsin_inverse_matrix above
   * is already re-targeted to the output primaries / white point (grey: three luminance rows). */
  float output_gamma;             /* JXG_TF_GAMMA exponent                             */
  float output_luminances[3];     /* Y row of the output primaries (JXG_TF_HLG)        */
} JxgFrameDesc;

/* PCI bus id of a CUDA device in the spelling of /sys/bus/pci/devices ("0000:1b:00.0"): lets the host bind its
 * threads and pinned allocations to the GPU's NUMA node before jxg_init. buf: >= 16 bytes. */
int jxg_device_pci_bus_id(int device, char* buf, int len);

/* Context: one per device/rank. Owns streams, pinned staging and device pools. */
int jxg_init(int device, void** ctx);
void jxg_shutdown(void* ctx);

/* Batch of frames decoded together (one kernel pipeline over all groups of
 * all frames). Replaces N calls of decode_and_render_hf_groups. */
int jxg_batch_begin(void* ctx, uint32_t n_frames_hint, void** batch);

/* hf_bytes: the frame's HF section bytes, any layout; section s (pass-major:
 * s = pass * num_groups + group, frame/mod.rs:326-338) lives at
 * hf_bytes[sec_off[s] .. sec_off[s] + sec_len[s]). n_sections = passes * groups.
 * out/out_row_stride: destination for the frame's pixels; `out_is_device` says
 * whether it is a device pointer (left in HBM) or a host pointer (D2H copy is
 * part of jxg_batch_run + jxg_batch_wait). */
int jxg_batch_add_frame(void* batch, const JxgFrameDesc* desc, const uint8_t* hf_bytes,
                        const uint64_t* sec_off, const uint32_t* sec_len, uint32_t n_sections,
                        void* out, size_t out_row_stride, int out_is_device);

/* Uploads (H2D from pinned staging), launches the kernels, queues D2H for host
 * outputs. Asynchronous on the context's stream (or `cuda_stream` if non-NULL). */
int jxg_batch_run(void* batch, void* cuda_stream);
/* Blocks until the batch finished; returns the first error (per-stream status
 * words written by the entropy kernel, check_final_state decode.rs:400). */
int jxg_batch_wait(void* batch, uint32_t* first_bad_frame, uint32_t* first_bad_group);
/* Re-run the same batch (inputs already resident in HBM): device-only timing. */
int jxg_batch_rerun_device(void* batch, void* cuda_stream);
void jxg_batch_end(void* batch);

/* Parity taps: copy intermediate planes of frame `f` of a finished batch to
 * host. coeffs: 3 planes of i32, dense per group in decode order (group.rs:53).
 * xyb: the three padded XYB planes after dequant + IDCT; `stage` must be 0
 * (any other value returns JXG_ERR_ARGUMENT). */
int jxg_batch_read_coeffs(void* batch, uint32_t f, int32_t* out, size_t out_len);
int jxg_batch_read_xyb(void* batch, uint32_t f, int stage, float* out, size_t out_len);

/* Opt-in host-side staging speed-up: copies of the large inputs (LF planes, per-block maps, HF sections) into the
 * pinned staging blob are postponed to jxg_batch_run and spread over `threads` host threads. Every pointer passed to
 * jxg_batch_add_frame / jxg_batch_add_parsed afterwards must stay valid until jxg_batch_run returns. 0 = immediate
 * copies (default; the contract a `&[u8]`-borrowing Rust caller gets, frame/render.rs:143). */
int jxg_batch_set_deferred_copy(void* batch, int threads);

/* Debug/parity: 0 = run everything (default), 1 = stop after the entropy kernel,
 * 2 = stop after dequant+IDCT (planes readable with jxg_batch_read_xyb stage 0).
 * Any other value returns JXG_ERR_ARGUMENT. */
int jxg_batch_set_debug_stop(void* batch, int stage);

/* Per-stage device timing with CUDA events on the launching stream (bench.py roofline):
 * stages = memset, entropy, dequant_idct, gaborish, epf0, epf1, epf2, xyb_store. */
int jxg_batch_set_profile(void* batch, int on);
int jxg_batch_stage_times(void* batch, float* ms, int n);
/* Absolute device times (ms since a process-wide reference event set at the first call) of the 9 stage events of the
 * last run: the timeline of several batches in flight. With n >= 11, ms[9] and ms[10] are the run's first event (before
 * the H2D copy of the staging blob) and its last one (behind the D2H copies of the outputs). */
int jxg_batch_stage_marks(void* batch, float* ms, int n);

/* Counters for bench.py (kernels launched by the last run, bytes moved). */
int jxg_batch_stats(void* batch, uint64_t* kernel_launches, uint64_t* h2d_bytes, uint64_t* d2h_bytes,
                    float* last_device_ms);

/* ---------------- convenience front-end (host parse + batch) ----------------
 * Parses complete .jxl files (container or bare codestream) on the host with
 * the in-tree C++ front-end (the stand-in for the Rust host: headers, TOC,
 * LfGlobal, LfGroups, HfGlobal), then feeds the batch API above. Mirrors
 * JxlDecoder::process for whole files (jxl/src/api/decoder.rs:258).
 * Frames with extra channels (alpha ...) are accepted and decode to their colour channels — the output of the
 * reference when JxlPixelFormat::extra_channel_format holds None (api/data_types.rs:154); patches, splines,
 * upsampling, non-regular / blended frames and JPEG recompression return JXG_ERR_UNSUPPORTED. */
typedef struct JxgImageInfo {
  uint32_t width, height; /* size of the OUTPUT (display orientation): what the caller allocates */
  uint32_t num_groups, num_passes;
  uint32_t encoding;      /* 0 VarDCT, 1 Modular */
  uint64_t hf_bytes;      /* sum of HF section sizes */
  uint32_t coded_width, coded_height; /* frame size as coded (swapped against width/height for orientation 5..8) */
  uint32_t orientation;   /* 1..8 */
} JxgImageInfo;

int jxg_parse_file(const uint8_t* data, size_t size, void** parsed, JxgImageInfo* info);
/* Same, decoding the frame's LF groups (independent TOC sections, frame/decode.rs:429 decode_lf_group) on `threads`
 * host threads, the fan-out jxl-rs does over its parallel runner (api/inner/codestream_parser/frame_info.rs:505-520):
 * the latency path for one large image. The parsed state does not depend on `threads`. */
int jxg_parse_file_mt(const uint8_t* data, size_t size, int threads, void** parsed, JxgImageInfo* info);
void jxg_parsed_free(void* parsed);
/* Adds a parsed frame to a batch with the given output. */
int jxg_batch_add_parsed(void* batch, void* parsed, uint32_t output_format, void* out, size_t out_row_stride,
                         int out_is_device);
/* Exposes the parsed frame as the (desc, sections) tuple jxg_batch_add_frame takes;
 * pointers stay valid until jxg_parsed_free. */
int jxg_parsed_desc(void* parsed, uint32_t output_format, JxgFrameDesc* desc, const uint8_t** hf_bytes,
                    const uint64_t** sec_off, const uint32_t** sec_len, uint32_t* n_sections);

/* ---- Modular frames (BASELINE config 5; SURVEY §8 rows a18 / a19) ------------------------------------------------
 * Seam: FullModularImage::read_stream for ModularHF sections (jxl/src/frame/modular/mod.rs:567,
 * decode/bitstream.rs:134, decode/channel.rs:220) plus the inverse transforms (transforms/{rct,squeeze}.rs) and
 * ConvertI32ToU8 (render/stages/convert.rs:642). The host front end (headers, LfGlobal incl. the global MA tree,
 * section 0, ModularLF streams, group headers / local trees) is jxg_modular_parse_file; a Rust host would hand over
 * the same state from Frame::decode_lf_global / decode_lf_group (frame/decode.rs:307-497).
 * Device scope: 8-bit RGB / grey, one pass, global transforms RCT and Squeeze, group-local RCT, ANS or prefix codes,
 * all 14 predictors incl. the weighted one, all properties incl. those of reference channels, the global palette
 * transform without delta entries (transforms/palette.rs:165-199). Delta palettes and LZ77 in group streams return
 * JXG_ERR_UNSUPPORTED (no CPU fallback). Output: interleaved RGB u8 (grey replicated). */
int jxg_modular_parse_file(const uint8_t* data, size_t size, void** parsed, JxgImageInfo* info);
void jxg_modular_parsed_free(void* parsed);
int jxg_modular_batch_begin(void* ctx, void** batch);
/* `parsed` must stay alive until jxg_modular_batch_end. */
int jxg_modular_batch_add(void* batch, void* parsed, void* out, size_t out_row_stride, int out_is_device);
/* Streams per warp of the decode kernel (1, 2 or 4; default 1). */
int jxg_modular_batch_set_lanes(void* batch, int lanes_per_warp);
int jxg_modular_batch_run(void* batch, void* cuda_stream);
int jxg_modular_batch_wait(void* batch, uint32_t* first_bad_frame, uint32_t* first_bad_group);
int jxg_modular_batch_rerun_device(void* batch, void* cuda_stream);
/* Parity tap: final colour planes of frame f (3 x H x W i32, before the u8 conversion). */
int jxg_modular_batch_read_planes(void* batch, uint32_t f, int32_t* out, size_t out_len);
/* ms[0]: whole batch on the device, ms[1]: group-stream decode kernel (+ local RCT). */
int jxg_modular_batch_stats(void* batch, uint64_t* h2d_bytes, uint64_t* d2h_bytes, uint64_t* kernel_launches, float* ms);
void jxg_modular_batch_end(void* batch);
/* Parity tap (no device needed): the table form of one channel's MA-tree walk as the Modular path builds it - the device
 * counterpart of the single-property specialisations of frame/modular/decode/specialized_trees.rs:197-372.
 * nodes: n_nodes x 5 ints {property (< 0: leaf), split value | offset, left child | predictor, right child | multiplier,
 * leaf context}; context_map: leaf context -> cluster. Returns 1 and fills lut[2048] (index = property value clamped to
 * [-1024, 1023] + 1024; entry = predictor | cluster << 4 | plain << 12 | leaf node << 16) and *property (0xff: single leaf,
 * every entry equal) when the tree left after the channel / stream decisions has a table form, 0 when the channel needs
 * the generic walk, JXG_ERR_ARGUMENT on malformed input. */
int jxg_modular_walk_table(const int32_t* nodes, uint32_t n_nodes, const uint8_t* context_map, uint32_t n_contexts,
                           uint32_t channel, uint32_t stream_id, uint32_t* lut, uint32_t* property);

const char* jxg_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* JXG_H_ */
