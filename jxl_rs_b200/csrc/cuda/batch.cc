// C ABI of libjxgpu.so (include/jxg.h): context + batch management around the
// sm_100a kernels. There is NO CPU fallback: without a CUDA device jxg_init
// fails with JXG_ERR_NO_DEVICE and nothing else can be called.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../../include/jxg.h"
#include "../host/frame.h"
#include "device_types.h"
#include "batch_common.h"
#include "launch.h"

using namespace jxgpu;

namespace jxgpu {
namespace detail {
thread_local std::string g_error;
std::atomic<int> g_live_contexts[64];  // per device: contexts between jxg_init and jxg_shutdown

cudaStream_t device_d2h_stream(int device) {
  static std::mutex mu;
  static cudaStream_t table[64];
  std::lock_guard<std::mutex> lk(mu);
  if (device < 0 || device >= 64) return nullptr;
  cudaStream_t& s = table[device];
  if (!s) {
    cudaSetDevice(device);
    if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) s = nullptr;
  }
  return s;
}
}
}  // namespace jxgpu
using namespace jxgpu::detail;

namespace {

struct FrameOut {
  void* user_ptr;
  size_t row_stride, rows, bytes;  // bytes: rows * row_stride (device staging), copy_bytes: what the user buffer must hold
  bool is_device;
  size_t dev_off;  // offset in d_out when !is_device
  size_t copy_bytes;
  // orientation != 1: the kernels store the coded image tightly into d_orient, k_orient writes the final place
  uint32_t orientation, coded_w, coded_h, bpp;
  size_t stage_off, stage_stride;
};

struct Batch {
  Context* ctx;
  PinnedArena& blob;
  explicit Batch(Context* c)
      : ctx(c), blob(c->blob), d_blob(c->d_blob), d_coeffs(c->d_coeffs), d_block_off(c->d_block_off), d_nz(c->d_nz),
        d_planes_a(c->d_planes_a), d_status(c->d_status), d_out(c->d_out) {}
  std::vector<FrameDev> frames;
  std::vector<SectionDev> sections;
  std::vector<StreamDev> streams, streams_lean, streams_fast, streams_slow;
  bool lean_all_420 = true;
  bool lean_ctx_smem = true;  // every lean frame's context map (+64 spill) fits k_entropy_lean's 16 KB staging area
  uint32_t lean_S = 1, lean_ctas = 0;  // k_entropy_lean schedule (see schedule_lean)
  std::vector<uint32_t> lean_cta_first;
  std::vector<uint2> lean_warps;  // per warp of k_entropy_lean: first stream (relative to its frame's list), lanes
  std::vector<uint64_t> nz_base;
  std::vector<uint32_t> fused_prefix{0};
  std::vector<FrameOut> outs;
  uint64_t total_groups = 0, total_blocks = 0, total_plane_floats = 0, nz_bytes = 0, out_bytes = 0, orient_bytes = 0;
  uint32_t lz_windows = 0;
  uint32_t filter_cfg_mask = 0;  // bit (gab * 4 + min(epf_iters, 3))
  int debug_stop = 0;
  // device
  DevBuf &d_blob, &d_coeffs, &d_block_off, &d_nz, &d_planes_a, &d_status, &d_out;
  bool uploaded = false;
  // byte offsets of the batch tables inside the blob (they ride on the one pinned H2D copy: a cudaMemcpyAsync from
  // pageable std::vector storage blocks the calling thread until earlier device work drains — 100+ ms with other
  // batches in flight, profiles/r02c_e2e_trace.log)
  struct {
    uint64_t frames = 0, sections = 0, streams = 0, lean_cta = 0, lean_warp = 0, streams_lean = 0, streams_fast = 0, streams_slow = 0,
             nz_base = 0, ftiles = 0;
  } tab;
  int32_t* status_host = nullptr;  // pinned (context-owned): a D2H copy into pageable memory would block jxg_batch_run
  size_t status_n = 0;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaStream_t last_stream = nullptr;  // stream of the last run / rerun (the context's or the caller's)
  bool profile = false;
  cudaEvent_t stage_ev[kNumStages + 1] = {nullptr};
  uint64_t launches = 0, h2d = 0, d2h = 0;
  float last_ms = 0;
};

// The kernels index device tables with fields of the descriptor and never bounds-check them, so everything a
// foreign host could get wrong is checked here (the in-tree front-end guarantees all of it by construction).
static int validate_desc(const JxgFrameDesc* d, const uint32_t* sec_len, uint32_t n_sections) {
  auto bad = [](const char* what) { return set_error(JXG_ERR_ARGUMENT, std::string("frame descriptor: ") + what); };
  static const uint8_t kCovX[27] = {1, 1, 1, 1, 2, 4, 1, 2, 1, 4, 2, 4, 1, 1, 1, 1, 1, 1, 8, 4, 8, 16, 8, 16, 32, 16, 32};
  static const uint8_t kCovY[27] = {1, 1, 1, 1, 2, 4, 2, 1, 4, 1, 4, 2, 1, 1, 1, 1, 1, 1, 8, 8, 4, 16, 16, 8, 32, 32, 16};
  static const uint32_t kShapeCoeffs[13] = {64, 64, 256, 1024, 128, 256, 512, 4096, 2048, 16384, 8192, 65536, 32768};
  if (!d->width || !d->height || d->width > (1u << 30) || d->height > (1u << 30)) return bad("bad dimensions");
  if (!d->global_scale || !d->color_factor || !(d->intensity_target > 0.0f)) return bad("zero global_scale / color_factor / intensity_target");
  if (!d->block_ctx_map || !d->passes || !d->transform_map || !d->raw_quant_map || !d->epf_map || !d->quant_lf || !d->ytox_map ||
      !d->ytob_map || !d->lf[0] || !d->lf[1] || !d->lf[2])
    return bad("null table pointer");
  if (d->num_qf_thresholds > 15 || !d->num_lf_contexts || d->num_lf_contexts > 64) return bad("bad qf / lf context counts");
  if (!d->num_block_contexts || d->num_block_contexts > 16) return bad("num_block_contexts must be 1..16");
  if (d->block_ctx_map_len != 39u * (d->num_qf_thresholds + 1) * d->num_lf_contexts) return bad("block_ctx_map_len");
  for (uint32_t i = 0; i < d->block_ctx_map_len; i++)
    if (d->block_ctx_map[i] >= d->num_block_contexts) return bad("block_ctx_map entry >= num_block_contexts");
  if (!d->num_histograms || d->num_histograms > 4096) return bad("num_histograms");
  if (d->output_tf > JXG_TF_HLG) return bad("unknown output_tf");
  if (d->output_tf == JXG_TF_GAMMA && !(d->output_gamma > 0.0f && d->output_gamma <= 1.0f)) return bad("output_gamma must be in (0, 1]");
  const uint64_t need_ctx = uint64_t(d->num_histograms) * d->num_block_contexts * 495;
  for (uint32_t p = 0; p < d->num_passes; p++) {
    const JxgPassDesc& s = d->passes[p];
    if (!s.context_map || !s.uint_configs) return bad("null pass table");
    if (!s.num_clusters || s.num_clusters > 256) return bad("num_clusters must be 1..256");
    if (s.num_contexts < need_ctx) return bad("context map shorter than num_histograms * num_block_contexts * 495");
    for (uint32_t i = 0; i < s.num_contexts; i++)
      if (s.context_map[i] >= s.num_clusters) return bad("context_map entry >= num_clusters");
    if (s.shift > 31) return bad("pass shift");
    if (s.lz77_enabled && s.lz_dist_cluster >= s.num_clusters) return bad("lz_dist_cluster >= num_clusters");
    if (s.use_prefix) {
      if (!s.huff_entries || !s.huff_offset) return bad("null prefix tables");
      for (uint32_t c = 0; c < s.num_clusters; c++) {
        const uint64_t o = s.huff_offset[c];
        if (o + 256 > s.huff_entries_len) return bad("prefix LUT root outside huff_entries");
        for (uint32_t r = 0; r < 256; r++) {  // 2nd-level reach of every root entry (huffman.rs:446-457)
          const uint32_t e = s.huff_entries[o + r], nb = e & 0xff;
          if (nb > 8 && (nb > 15 || o + r + (e >> 16) + (1u << (nb - 8)) > s.huff_entries_len)) return bad("prefix LUT 2nd level outside huff_entries");
        }
      }
    } else {
      if (!s.ans_buckets) return bad("null ANS table");
      if (s.log_alpha_size < 5 || s.log_alpha_size > 8) return bad("log_alpha_size must be 5..8");
    }
    if (s.coeff_order) {
      for (int i = 0; i < 39; i++) {
        const uint64_t o = s.coeff_order_offset[i], n = kShapeCoeffs[i / 3];
        if (o + n > s.coeff_order_len) return bad("coefficient order outside coeff_order");
        for (uint64_t k = 0; k < n; k++)
          if (s.coeff_order[o + k] >= n) return bad("coefficient order entry out of range");
      }
    }
  }
  const uint32_t xb = (d->width + 7) / 8, yb = (d->height + 7) / 8;
  for (uint32_t by = 0; by < yb; by++)
    for (uint32_t bx = 0; bx < xb; bx++) {
      const size_t i = size_t(by) * xb + bx;
      if (d->quant_lf[i] >= d->num_lf_contexts) return bad("quant_lf entry >= num_lf_contexts");
      if (d->epf_map[i] > 7) return bad("epf sharpness > 7");
      const uint32_t t = d->transform_map[i];
      if (t < 128) continue;
      if ((t & 127) >= 27) return bad("unknown transform type");
      const uint32_t cx = kCovX[t & 127], cy = kCovY[t & 127];
      if ((bx & 31) + cx > 32 || (by & 31) + cy > 32 || bx + cx > xb || by + cy > yb) return bad("varblock crosses its group or the frame");
      if (d->raw_quant_map[i] < 1) return bad("raw_quant < 1");
    }
  for (uint32_t i = 0; i < n_sections; i++)
    if (sec_len[i] > (1u << 30)) return bad("HF section too large");
  return 0;
}

}  // namespace

extern "C" {

const char* jxg_last_error(void) { return g_error.c_str(); }

// PCI bus id of a CUDA device ("0000:1b:00.0", lower case, as under /sys/bus/pci/devices), so that a host can find the
// NUMA node the GPU hangs off and keep its threads and pinned buffers there. No context is created.
int jxg_device_pci_bus_id(int device, char* buf, int len) {
  if (!buf || len < 16) return JXG_ERR_ARGUMENT;
  CUDA_TRY(cudaDeviceGetPCIBusId(buf, len, device));
  for (char* p = buf; *p; p++)
    if (*p >= 'A' && *p <= 'Z') *p = char(*p - 'A' + 'a');
  return JXG_OK;
}

int jxg_init(int device, void** out_ctx) {
  if (!out_ctx) return JXG_ERR_ARGUMENT;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0)
    return set_error(JXG_ERR_NO_DEVICE, "no CUDA device: libjxgpu has no CPU fallback");
  if (device < 0 || device >= n) return set_error(JXG_ERR_ARGUMENT, "bad device index");
  CUDA_TRY(cudaSetDevice(device));
  auto ctx = std::make_unique<Context>();
  ctx->device = device;
  CUDA_TRY(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  ctx->d2h_stream = device_d2h_stream(device);
  if (!ctx->d2h_stream) return set_error(JXG_ERR_CUDA, "cannot create the device's D2H stream");
  for (auto& e : ctx->range_done) CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming | cudaEventBlockingSync));
  CUDA_TRY(cudaEventCreateWithFlags(&ctx->copy_done, cudaEventDisableTiming | cudaEventBlockingSync));
  // constant tables
  std::vector<float> wc(9 * 128, 0.0f), rs(6 * 32, 0.0f);
  for (int l = 1; l <= 8; l++) {
    int nn = 1 << l;
    for (int i = 0; i < nn / 2; i++) wc[l * 128 + i] = float(1.0 / (2.0 * std::cos((i + 0.5) * M_PI / nn)));
  }
  for (int l = 0; l <= 5; l++) {
    int nn = 1 << l;
    for (int i = 0; i < nn; i++) {
      double s = std::cos(i / (16.0 * nn) * M_PI) * std::cos(i / (8.0 * nn) * M_PI) * std::cos(i / (4.0 * nn) * M_PI) * nn;
      rs[l * 32 + i] = float(std::round(1e6 / s) / 1e6);  // 6-decimal literals of the generated reference code
    }
  }
  CUDA_TRY(upload_constants(wc.data(), rs.data()));
  CUDA_TRY(configure_kernels());
  // library dequant tables and natural coefficient orders
  std::vector<float> dq;
  std::vector<uint32_t> dq_off(17);
  for (int i = 0; i < 17; i++) {
    const std::vector<float>& t = jxg::library_dequant_table(i);
    dq_off[i] = uint32_t(dq.size());
    dq.insert(dq.end(), t.begin(), t.end());
  }
  std::vector<uint32_t> no, no_off(13);
  for (int i = 0; i < 13; i++) {
    std::vector<uint32_t> o = jxg::natural_coeff_order(i);
    no_off[i] = uint32_t(no.size());
    no.insert(no.end(), o.begin(), o.end());
  }
  if (int r = upload(ctx->dequant_default, dq, ctx->stream, nullptr)) return r;
  if (int r = upload(ctx->dequant_default_off, dq_off, ctx->stream, nullptr)) return r;
  if (int r = upload(ctx->natural_orders, no, ctx->stream, nullptr)) return r;
  if (int r = upload(ctx->natural_order_off, no_off, ctx->stream, nullptr)) return r;
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  g_live_contexts[device & 63].fetch_add(1);
  *out_ctx = ctx.release();
  return JXG_OK;
}

void jxg_shutdown(void* c) {
  Context* ctx = static_cast<Context*>(c);
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  for (auto& e : ctx->range_done)
    if (e) cudaEventDestroy(e);
  if (ctx->copy_done) cudaEventDestroy(ctx->copy_done);
  if (ctx->status_host) cudaFreeHost(ctx->status_host);
  g_live_contexts[ctx->device & 63].fetch_sub(1);
  delete ctx;
}

int jxg_batch_begin(void* c, uint32_t n_frames_hint, void** out_batch) {
  if (!c || !out_batch) return JXG_ERR_ARGUMENT;
  Context* cx = static_cast<Context*>(c);
  if (cx->batch_live) return set_error(JXG_ERR_ARGUMENT, "one live batch per context: call jxg_batch_end first");
  auto b = std::make_unique<Batch>(cx);
  CUDA_TRY(cudaSetDevice(b->ctx->device));
  cx->blob.size = 0;
  cx->blob.pending.clear();
  cx->blob.deferred_threads = 0;
  b->frames.reserve(n_frames_hint);
  CUDA_TRY(cudaEventCreate(&b->ev0));
  if (cudaError_t e = cudaEventCreate(&b->ev1); e != cudaSuccess) {
    cudaEventDestroy(b->ev0);
    return set_error(JXG_ERR_CUDA, std::string("cudaEventCreate: ") + cudaGetErrorString(e));
  }
  cx->batch_live = true;  // only once nothing can fail any more
  *out_batch = b.release();
  return JXG_OK;
}

void jxg_batch_end(void* bp) {
  Batch* b = static_cast<Batch*>(bp);
  if (!b) return;
  cudaSetDevice(b->ctx->device);
  if (b->uploaded && b->ev1) cudaEventSynchronize(b->ev1);
  if (b->ev0) cudaEventDestroy(b->ev0);
  if (b->ev1) cudaEventDestroy(b->ev1);
  for (auto& e : b->stage_ev)
    if (e) cudaEventDestroy(e);
  b->ctx->batch_live = false;
  delete b;
}

int jxg_batch_set_profile(void* bp, int on) {
  Batch* b = static_cast<Batch*>(bp);
  if (!b) return JXG_ERR_ARGUMENT;
  if (on && !b->stage_ev[0])
    for (auto& e : b->stage_ev) CUDA_TRY(cudaEventCreate(&e));
  b->profile = on != 0;
  return JXG_OK;
}

// ms per stage of the last run (memset, entropy, dequant_idct, gaborish, epf0, epf1, epf2, xyb_store); 0 if skipped.
int jxg_batch_stage_times(void* bp, float* ms, int n) {
  Batch* b = static_cast<Batch*>(bp);
  if (!b || !ms || n < kNumStages || !b->profile) return JXG_ERR_ARGUMENT;
  CUDA_TRY(cudaEventSynchronize(b->ev1));
  for (int i = 0; i < kNumStages; i++) {
    ms[i] = 0.0f;
    if (cudaEventElapsedTime(&ms[i], b->stage_ev[i], b->stage_ev[i + 1]) != cudaSuccess) ms[i] = 0.0f;
  }
  cudaGetLastError();
  return JXG_OK;
}

// Absolute device times of the stage events of the last run, in ms since a process-wide reference event (recorded at the
// first call): ms[i] = time of event i (before stage i; ms[kNumStages] = end), 0 for events that were not recorded.
// Lets a host draw the timeline of several batches in flight (tools/e2e_profile4.py).
int jxg_batch_stage_marks(void* bp, float* ms, int n) {
  Batch* b = static_cast<Batch*>(bp);
  if (!b || !ms || n < kNumStages + 1 || !b->profile) return JXG_ERR_ARGUMENT;
  static cudaEvent_t ref = nullptr;
  if (!ref) {
    CUDA_TRY(cudaEventCreate(&ref));
    CUDA_TRY(cudaEventRecord(ref, 0));
    CUDA_TRY(cudaEventSynchronize(ref));
  }
  CUDA_TRY(cudaEventSynchronize(b->ev1));
  for (int i = 0; i <= kNumStages; i++)
    if (cudaEventElapsedTime(&ms[i], ref, b->stage_ev[i]) != cudaSuccess) ms[i] = 0.0f;
  if (n >= kNumStages + 3) {  // + the run's first event (before the H2D copy) and its last (behind the D2H copies)
    if (cudaEventElapsedTime(&ms[kNumStages + 1], ref, b->ev0) != cudaSuccess) ms[kNumStages + 1] = 0.0f;
    if (cudaEventElapsedTime(&ms[kNumStages + 2], ref, b->ev1) != cudaSuccess) ms[kNumStages + 2] = 0.0f;
  }
  cudaGetLastError();
  return JXG_OK;
}

// Opt-in: copies of large inputs (LF planes, maps, HF sections) into the pinned staging blob are postponed to
// jxg_batch_run and spread over `threads` host threads. Every pointer handed to jxg_batch_add_frame /
// jxg_batch_add_parsed must then stay valid until jxg_batch_run returns.
int jxg_batch_set_deferred_copy(void* bp, int threads) {
  Batch* b = static_cast<Batch*>(bp);
  if (!b || threads < 0) return JXG_ERR_ARGUMENT;
  if (b->uploaded) return set_error(JXG_ERR_ARGUMENT, "batch already submitted");
  b->blob.deferred_threads = threads;
  return JXG_OK;
}

int jxg_batch_set_debug_stop(void* bp, int stage) {
  Batch* b = static_cast<Batch*>(bp);
  if (!b) return JXG_ERR_ARGUMENT;
  if (stage < 0 || stage > 2) return set_error(JXG_ERR_ARGUMENT, "debug stop must be 0, 1 or 2");
  b->debug_stop = stage;
  return JXG_OK;
}

// `trusted`: the descriptor comes from the in-tree front-end, which guarantees every invariant validate_desc checks by
// construction (the scan costs ~0.45 ms per 4K frame, 30 ms per 64-frame batch on the dispatcher's critical path).
static int add_frame_impl(void* bp, const JxgFrameDesc* d, const uint8_t* hf_bytes, const uint64_t* sec_off,
                          const uint32_t* sec_len, uint32_t n_sections, void* out, size_t out_row_stride,
                          int out_is_device, bool trusted) {
  Batch* b = static_cast<Batch*>(bp);
  if (!b || !d || !hf_bytes || !sec_off || !sec_len || !out) return JXG_ERR_ARGUMENT;
  if (d->abi_version != JXG_ABI_VERSION) return set_error(JXG_ERR_ARGUMENT, "ABI version mismatch");
  if (b->uploaded) return set_error(JXG_ERR_ARGUMENT, "batch already submitted");
  if (d->num_passes == 0 || d->num_passes > kMaxPasses) return set_error(JXG_ERR_ARGUMENT, "bad num_passes");
  FrameDev F;
  memset(&F, 0, sizeof(F));
  F.width = d->width;
  F.height = d->height;
  F.xb = (d->width + 7) / 8;
  F.yb = (d->height + 7) / 8;
  F.xg = (d->width + 255) / 256;
  F.yg = (d->height + 255) / 256;
  F.num_groups = F.xg * F.yg;
  F.num_passes = d->num_passes;
  if (n_sections != F.num_groups * F.num_passes) return set_error(JXG_ERR_ARGUMENT, "n_sections != groups * passes");
  F.plane_stride = F.xb * 8;
  F.plane_rows = F.yb * 8;
  F.cxb = (F.xb + 7) / 8;
  const size_t nb = size_t(F.xb) * F.yb, ncm = size_t(F.cxb) * ((F.yb + 7) / 8);
  if (d->output_format > JXG_FORMAT_RGB_F16) return set_error(JXG_ERR_ARGUMENT, "unknown output format");
  size_t bpp = d->output_format == JXG_FORMAT_RGB_U8 ? 3
               : d->output_format == JXG_FORMAT_RGBA_U8 ? 4
               : d->output_format == JXG_FORMAT_RGB_F32 ? 12
               : (d->output_format == JXG_FORMAT_RGB_U16 || d->output_format == JXG_FORMAT_RGB_F16) ? 6 : 4;
  if (d->orientation > 8) return set_error(JXG_ERR_ARGUMENT, "orientation must be 1..8");
  const uint32_t orientation = (d->orientation == 0 || d->output_format == JXG_FORMAT_XYB_F32_PLANAR) ? 1u : d->orientation;
  const uint32_t disp_w = orientation >= 5 ? F.height : F.width, disp_h = orientation >= 5 ? F.width : F.height;
  if (out_row_stride < size_t(disp_w) * bpp) return set_error(JXG_ERR_INVALID_OUTPUT, "output row stride too small");
  if (!trusted)
    if (int r = validate_desc(d, sec_len, n_sections)) return r;
  F.num_histograms = d->num_histograms;
  F.num_block_contexts = d->num_block_contexts;
  F.num_lf_contexts = d->num_lf_contexts;
  F.num_qf_thresholds = d->num_qf_thresholds;
  if (F.num_qf_thresholds > 15) return set_error(JXG_ERR_ARGUMENT, "too many qf thresholds");
  memcpy(F.qf_thresholds, d->qf_thresholds, sizeof(F.qf_thresholds));
#define APPEND(dst, src, bytes, align)                                         \
  do {                                                                         \
    int64_t o__ = b->blob.append(src, bytes, align);                           \
    if (o__ < 0) return set_error(JXG_ERR_CUDA, "pinned staging allocation failed"); \
    dst = uint64_t(o__);                                                       \
  } while (0)
  APPEND(F.block_ctx_map_off, d->block_ctx_map, d->block_ctx_map_len, 16);
  for (uint32_t p = 0; p < d->num_passes; p++) {
    const JxgPassDesc& s = d->passes[p];
    PassDev& P = F.passes[p];
    if (s.lz77_enabled) F.has_lz = 1;  // routed to the one-lane-per-warp kernel, which carries the LZ77 window
    P.lz77_enabled = s.lz77_enabled;
    P.lz77_min_symbol = s.lz77_min_symbol;
    P.lz77_min_length = s.lz77_min_length;
    P.lz77_length_uint = s.lz77_length_uint;
    P.lz_dist_cluster = s.lz_dist_cluster;
    P.shift = s.shift;
    P.use_prefix = s.use_prefix;
    P.log_alpha_size = s.log_alpha_size;
    P.num_clusters = s.num_clusters;
    P.custom_orders = s.coeff_order != nullptr;
    APPEND(P.context_map_off, s.context_map, s.num_contexts, 16);
    APPEND(P.uint_configs_off, s.uint_configs, size_t(s.num_clusters) * 4, 16);
    if (s.use_prefix) {
      APPEND(P.huff_off, s.huff_entries, size_t(s.huff_entries_len) * 4, 16);
      APPEND(P.huff_offset_off, s.huff_offset, size_t(s.num_clusters) * 4, 16);
    } else {
      APPEND(P.ans_off, s.ans_buckets, (size_t(s.num_clusters) << s.log_alpha_size) * 8, 16);
    }
    if (P.custom_orders) {
      APPEND(P.order_off, s.coeff_order, size_t(s.coeff_order_len) * 4, 16);
      memcpy(P.order_offset, s.coeff_order_offset, sizeof(P.order_offset));
    }
  }
  F.inv_global_scale = 65536.0f / float(d->global_scale);
  F.x_dm = std::pow(1.0f / 1.25f, float(d->x_qm_scale) - 2.0f);  // group.rs:395-396
  F.b_dm = std::pow(1.0f / 1.25f, float(d->b_qm_scale) - 2.0f);
  memcpy(F.quant_biases, d->quant_biases, sizeof(F.quant_biases));
  F.base_correlation_x = d->base_correlation_x;
  F.base_correlation_b = d->base_correlation_b;
  F.color_factor = d->color_factor;
  for (int i = 0; i < 17; i++) {
    F.dequant_off[i] = -1;
    if (d->dequant_tables[i]) {
      size_t n = 3 * 64 * size_t(jxg::kQuantTableRows[i]) * jxg::kQuantTableCols[i];
      uint64_t o;
      APPEND(o, d->dequant_tables[i], n * 4, 16);
      F.dequant_off[i] = int64_t(o);
    }
  }
  for (int c = 0; c < 3; c++) APPEND(F.lf_off[c], d->lf[c], nb * 4, 16);
  APPEND(F.transform_off, d->transform_map, nb, 16);
  APPEND(F.raw_quant_off, d->raw_quant_map, nb * 4, 16);
  APPEND(F.epf_off, d->epf_map, nb, 16);
  APPEND(F.quant_lf_off, d->quant_lf, nb, 16);
  APPEND(F.ytox_off, d->ytox_map, ncm, 16);
  APPEND(F.ytob_off, d->ytob_map, ncm, 16);
  F.section_base = uint32_t(b->sections.size());
  for (uint32_t s = 0; s < n_sections; s++) {
    SectionDev sd;
    uint64_t o;
    // 8-byte aligned copy followed by >= 8 zero bytes: the device bit reader
    // refills with aligned 32-bit words and may look one word past the end.
    int64_t oo = b->blob.append(hf_bytes + sec_off[s], sec_len[s], 8, 8);
    if (oo < 0) return set_error(JXG_ERR_CUDA, "pinned staging allocation failed");
    o = uint64_t(oo);
    sd.off = o;
    sd.len = sec_len[s];
    sd.pad = 0;
    b->sections.push_back(sd);
  }
#undef APPEND
  if (F.has_lz) {
    F.lz_win_base = b->lz_windows;
    b->lz_windows += F.num_passes * F.num_groups;
  }
  if (F.num_passes == 1 && !F.has_lz && !F.passes[0].use_prefix && F.passes[0].shift == 0 &&
      size_t(F.num_histograms) * F.num_block_contexts * 495 + 64 > 16384)
    b->lean_ctx_smem = false;
  if (F.num_passes == 1 && !F.has_lz && !F.passes[0].use_prefix)
    for (uint32_t c = 0; c < d->passes[0].num_clusters; c++)
      if (d->passes[0].uint_configs[c] != (4u | (2u << 8))) b->lean_all_420 = false;
  F.first_stream = uint32_t(b->streams.size());
  for (uint32_t g = 0; g < F.num_groups; g++) {
    b->streams.push_back(StreamDev{uint32_t(b->frames.size()), g});
    ((F.num_passes != 1 || F.has_lz) ? b->streams_slow : ((F.passes[0].use_prefix || F.passes[0].shift != 0) ? b->streams_fast : b->streams_lean)).push_back(StreamDev{uint32_t(b->frames.size()), g});
    b->nz_base.push_back(b->nz_bytes);
    b->nz_bytes += size_t(F.num_passes) * 3072;
  }
  F.coeff_group_base = b->total_groups;
  b->total_groups += F.num_groups;
  F.block_base = b->total_blocks;
  b->total_blocks += nb;
  F.plane_size = size_t(F.plane_stride) * F.plane_rows;
  F.plane_base = b->total_plane_floats;
  b->total_plane_floats += 3 * F.plane_size;
  F.out_row_stride = out_row_stride;
  size_t rows = d->output_format == JXG_FORMAT_XYB_F32_PLANAR ? size_t(F.height) * 3 : disp_h;
  FrameOut fo{};
  fo.user_ptr = out;
  fo.row_stride = out_row_stride;
  fo.rows = rows;
  fo.bytes = rows * out_row_stride;
  fo.copy_bytes = (rows - 1) * out_row_stride + size_t(disp_w) * bpp;  // the last row of a user buffer may be unpadded
  fo.is_device = out_is_device != 0;
  fo.orientation = orientation;
  fo.coded_w = F.width;
  fo.coded_h = F.height;
  fo.bpp = uint32_t(bpp);
  if (!fo.is_device) {
    fo.dev_off = (b->out_bytes + 255) / 256 * 256;
    b->out_bytes = fo.dev_off + fo.bytes;
  }
  if (orientation != 1) {  // coded image, tight rows (16-byte multiples: the vector store path stays usable)
    fo.stage_stride = (size_t(F.width) * bpp + 15) / 16 * 16;
    fo.stage_off = (b->orient_bytes + 255) / 256 * 256;
    b->orient_bytes = fo.stage_off + fo.stage_stride * F.height;
    F.out_row_stride = fo.stage_stride;
  }
  b->outs.push_back(fo);
  F.gab = d->gab;
  for (int c = 0; c < 3; c++) {  // gaborish.rs:20-27
    float total = 1.0f + d->gab_w1[c] * 4.0f + d->gab_w2[c] * 4.0f;
    F.gab_k0[c] = 1.0f / total;
    F.gab_k1[c] = d->gab_w1[c] / total;
    F.gab_k2[c] = d->gab_w2[c] / total;
  }
  F.epf_iters = d->epf_iters;
  memcpy(F.epf_sharp_lut, d->epf_sharp_lut, sizeof(F.epf_sharp_lut));
  memcpy(F.epf_channel_scale, d->epf_channel_scale, sizeof(F.epf_channel_scale));
  F.epf_quant_mul = d->epf_quant_mul;
  F.epf_pass0_sigma_scale = d->epf_pass0_sigma_scale;
  F.epf_pass2_sigma_scale = d->epf_pass2_sigma_scale;
  F.epf_border_sad_mul = d->epf_border_sad_mul;
  F.quant_scale = 1.0f / F.inv_global_scale;
  memcpy(F.opsin, d->opsin_inverse_matrix, sizeof(F.opsin));
  F.intensity_scale = 255.0f / d->intensity_target;
  for (int i = 0; i < 3; i++) {  // xyb.rs:147-160
    F.bias_cbrt[i] = std::cbrt(d->opsin_biases[i]);
    F.scaled_bias[i] = d->opsin_biases[i] * F.intensity_scale;
  }
  F.output_tf = d->output_tf;
  F.output_format = d->output_format;
  F.tf_gamma = d->output_gamma;
  memcpy(F.tf_lum, d->output_luminances, sizeof(F.tf_lum));
  {  // color/tf.rs:458-470 hlg_display_to_scene: exponent of the inverse OOTF; |exp| < 0.1 skips it (tf.rs:381-383)
    const float system_gamma = 1.2f * std::pow(1.111f, std::log2(d->intensity_target / 1e3f));
    const float e = (1.0f - system_gamma) / system_gamma;
    F.tf_hlg_exp = std::fabs(e) < 0.1f ? 0.0f : e;
  }
  F.tf_pq_mul = d->intensity_target * (1.0f / 10000.0f);
  b->filter_cfg_mask |= 1u << ((d->gab ? 4 : 0) + std::min<uint32_t>(d->epf_iters, 3));
  b->fused_prefix.push_back(b->fused_prefix.back() + ((F.width + kFusedTileW - 1) / kFusedTileW) * ((F.height + kFusedTileH - 1) / kFusedTileH));
  b->frames.push_back(F);
  return JXG_OK;
}

int jxg_batch_add_frame(void* bp, const JxgFrameDesc* d, const uint8_t* hf_bytes, const uint64_t* sec_off,
                        const uint32_t* sec_len, uint32_t n_sections, void* out, size_t out_row_stride,
                        int out_is_device) {
  return add_frame_impl(bp, d, hf_bytes, sec_off, sec_len, n_sections, out, out_row_stride, out_is_device, false);
}

// Schedule of the persistent entropy lanes (k_entropy_lean). A stream's cost is proportional to its section length
// and a stream is one serial chain; each frame's streams are ordered longest first and handed to the frame's lanes in
// that order (longest-processing-time rule), streams beyond the initial assignment are queued and pulled by whichever
// lane finishes first. All CTAs of one frame stay on that frame so that its tables stay in L1 / shared memory.
// Measured on B200 (64 x 4K, profiles/r02_entropy_schedule.md): every stream on a lane of its own from the start, four
// lanes to a warp, is the fastest (33.1 ms); giving the longest streams warps of their own is slower (38.6 - 41.4 ms)
// because a lone lane still costs a full warp's issue slots, and so are fewer lanes with queued streams (43.9 ms at 2.5
// streams per lane) and 8 lanes per warp (40.2). Those alternatives were removed.
static void schedule_lean(Batch* b) {
  if (b->streams_lean.empty() || b->lean_ctas) return;
  auto len_of = [&](const StreamDev& sd) { return b->sections[b->frames[sd.frame].section_base + sd.group].len; };
  std::stable_sort(b->streams_lean.begin(), b->streams_lean.end(), [&](const StreamDev& x, const StreamDev& y) {
    return x.frame != y.frame ? x.frame < y.frame : len_of(x) > len_of(y);
  });
  const size_t nf = b->frames.size();
  for (auto& F : b->frames) F.lean_first = F.lean_count = F.lean_cta_first = F.lean_ctas = F.lean_lanes = 0;
  for (size_t i = 0; i < b->streams_lean.size();) {
    const uint32_t f = b->streams_lean[i].frame;
    size_t j = i;
    while (j < b->streams_lean.size() && b->streams_lean[j].frame == f) j++;
    b->frames[f].lean_first = uint32_t(i);
    b->frames[f].lean_count = uint32_t(j - i);
    i = j;
  }
  // The kernel keeps 6 CTAs per SM resident (register bound); a grid beyond one resident wave would start its last
  // CTAs only when the first ones end, so the packing is made denser until the grid fits.
  const uint32_t max_ctas = 148 * 6;
  // 4 lanes per warp are the fastest schedule for a batch that has the device to itself; 8 lanes halve the kernel's
  // warp-instructions, which is what counts once several batches share the SMs (64 x 4K: alone 57.2 against 52.3 ms, three
  // resident batches 37.1 against 40.5 ms per batch, five 35.1 against 38.0; 16 and 32 lanes lose again:
  // profiles/r02k_entropy_lanes.log). Three or more live contexts on the device are taken as "batches share the SMs".
  uint32_t S = 4;
  if (g_live_contexts[b->ctx->device & 63].load() >= 3 && b->streams_lean.size() >= 2048) S = 8;
  float per_lane = 1.0f;  // streams per lane (initial stream + queued ones): 1 = every stream starts at once
  std::vector<uint2> warps;
  for (int attempt = 0; attempt < 12; attempt++) {
    warps.clear();
    uint32_t ctas = 0;
    for (size_t f = 0; f < nf; f++) {
      FrameDev& F = b->frames[f];
      F.lean_cta_first = ctas;
      F.lean_ctas = F.lean_lanes = 0;
      if (!F.lean_count) continue;
      uint32_t lanes = uint32_t(std::ceil(float(F.lean_count) / per_lane));
      lanes = std::min(F.lean_count, (lanes + S - 1) / S * S);
      const size_t w0 = warps.size();
      for (uint32_t pos = 0; pos < lanes; pos += S) warps.push_back(make_uint2(pos, std::min(S, lanes - pos)));
      while ((warps.size() - w0) % 4) warps.push_back(make_uint2(F.lean_count, 0));  // idle warps of the frame's last CTA
      F.lean_lanes = lanes;
      F.lean_ctas = uint32_t(warps.size() - w0) / 4;
      ctas += F.lean_ctas;
    }
    b->lean_ctas = ctas;
    if (ctas <= max_ctas) break;
    // denser: first 8 lanes per warp, then more streams per lane
    if (S < 8) S = 8;
    else per_lane *= 1.3f;
  }
  b->lean_S = S;
  b->lean_warps = std::move(warps);
  b->lean_cta_first.assign(nf, 0);
  for (size_t f = 0; f < nf; f++) b->lean_cta_first[f] = b->frames[f].lean_cta_first;
}

static BatchDev make_batch_dev(Batch* b) {
  BatchDev B;
  memset(&B, 0, sizeof(B));
  B.blob = static_cast<const uint8_t*>(b->d_blob.p);
  auto tab = [&](uint64_t off) { return static_cast<const uint8_t*>(b->d_blob.p) + off; };
  B.frames = reinterpret_cast<const FrameDev*>(tab(b->tab.frames));
  B.sections = reinterpret_cast<const SectionDev*>(tab(b->tab.sections));
  B.streams = reinterpret_cast<const StreamDev*>(tab(b->tab.streams));
  B.num_frames = uint32_t(b->frames.size());
  B.num_streams = uint32_t(b->streams.size());
  B.streams_lean = reinterpret_cast<const StreamDev*>(tab(b->tab.streams_lean));
  B.num_lean = uint32_t(b->streams_lean.size());
  B.streams_fast = reinterpret_cast<const StreamDev*>(tab(b->tab.streams_fast));
  B.streams_slow = reinterpret_cast<const StreamDev*>(tab(b->tab.streams_slow));
  B.num_fast = uint32_t(b->streams_fast.size());
  B.num_slow = uint32_t(b->streams_slow.size());
  B.nzlist = static_cast<uint32_t*>(b->d_coeffs.p);  // the pool that held the dense coefficients now holds the lists
  B.block_off = static_cast<uint32_t*>(b->d_block_off.p);
  B.lzwin = static_cast<uint32_t*>(b->ctx->d_lzwin.p);
  B.nz = static_cast<uint8_t*>(b->d_nz.p);
  B.nz_base = reinterpret_cast<uint64_t*>(const_cast<uint8_t*>(tab(b->tab.nz_base)));
  B.planes_a = static_cast<float*>(b->d_planes_a.p);
  B.status = static_cast<int32_t*>(b->d_status.p);
  B.queue = reinterpret_cast<uint32_t*>(B.status + b->streams.size());
  B.lean_cta_first = reinterpret_cast<const uint32_t*>(tab(b->tab.lean_cta));
  B.lean_warp = reinterpret_cast<const uint2*>(tab(b->tab.lean_warp));
  B.desc = static_cast<uint4*>(b->ctx->d_lean_desc.p);
  B.nblk = static_cast<uint32_t*>(b->ctx->d_lean_nblk.p);
  B.dequant_default = static_cast<const float*>(b->ctx->dequant_default.p);
  B.dequant_default_off = static_cast<const uint32_t*>(b->ctx->dequant_default_off.p);
  B.natural_orders = static_cast<const uint32_t*>(b->ctx->natural_orders.p);
  B.natural_order_off = static_cast<const uint32_t*>(b->ctx->natural_order_off.p);
  return B;
}

// Enqueues one run of the batch on `s`. With copy_to_host, the host outputs go back on the device's D2H stream: each of
// up to kMaxRanges frame ranges is copied as soon as its filter launch ends, while the next range is being filtered.
static int launch(Batch* b, cudaStream_t s, bool copy_to_host) {
  const BatchDev B = make_batch_dev(b);
  cudaEvent_t* ev = b->profile ? b->stage_ev : nullptr;
  b->launches = uint64_t(launch_pipeline(B, s, b->debug_stop, ev, b->lean_all_420, b->lean_S, b->lean_ctas, b->lean_ctx_smem));
  if (b->debug_stop == 0) {
    // Fused filter + colour + store, launched per range of frames.
    Context* cx = b->ctx;
    const uint32_t nf = uint32_t(b->frames.size());
    const uint32_t nr = copy_to_host ? std::min<uint32_t>(Context::kMaxRanges, nf) : 1;
    const uint32_t* fp = reinterpret_cast<const uint32_t*>(static_cast<const uint8_t*>(b->d_blob.p) + b->tab.ftiles);
    if (ev) {
      for (int i = 4; i <= 6; i++) cudaEventRecord(ev[i], s);
    }
    for (uint32_t r = 0; r < nr; r++) {
      const uint32_t f0 = uint32_t(uint64_t(nf) * r / nr), f1 = uint32_t(uint64_t(nf) * (r + 1) / nr);
      const uint32_t t0 = b->fused_prefix[f0], t1 = b->fused_prefix[f1];
      b->launches += uint64_t(launch_filter_range(B, fp, t0, t1 - t0, b->filter_cfg_mask, s));
      for (uint32_t f = f0; f < f1; f++) {  // orientation post-pass (rare): staging image -> final place
        const FrameOut& fo = b->outs[f];
        if (fo.orientation == 1) continue;
        void* dst = fo.is_device ? fo.user_ptr : static_cast<void*>(static_cast<uint8_t*>(b->d_out.p) + fo.dev_off);
        launch_orient(static_cast<uint8_t*>(cx->d_orient.p) + fo.stage_off, fo.stage_stride, dst, fo.row_stride, fo.coded_w,
                      fo.coded_h, fo.bpp, fo.orientation, s);
        b->launches++;
      }
      if (copy_to_host) {
        CUDA_TRY(cudaEventRecord(cx->range_done[r], s));
        CUDA_TRY(cudaStreamWaitEvent(cx->d2h_stream, cx->range_done[r], 0));
        for (uint32_t f = f0; f < f1; f++) {
          const FrameOut& fo = b->outs[f];
          if (fo.is_device) continue;
          CUDA_TRY(cudaMemcpyAsync(fo.user_ptr, static_cast<uint8_t*>(b->d_out.p) + fo.dev_off, fo.copy_bytes, cudaMemcpyDeviceToHost,
                                   cx->d2h_stream));
          b->d2h += fo.copy_bytes;
        }
      }
    }
    if (ev) {
      cudaEventRecord(ev[7], s);
      cudaEventRecord(ev[8], s);
    }
  }
  CUDA_TRY(cudaGetLastError());
  return 0;
}

static int copy_status(Batch* b, cudaStream_t s) {
  CUDA_TRY(cudaMemcpyAsync(b->status_host, b->d_status.p, b->status_n * 4, cudaMemcpyDeviceToHost, s));
  return 0;
}

// JXG_TRACE_RUN=1: host-side phase times of jxg_batch_run on stderr (which call blocks, and for how long).
struct RunTrace {
  bool on = getenv("JXG_TRACE_RUN") != nullptr;
  std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now(), last = t0;
  std::string line;
  void mark(const char* what) {
    if (!on) return;
    const auto now = std::chrono::steady_clock::now();
    char buf[64];
    snprintf(buf, sizeof(buf), " %s %.1f", what, std::chrono::duration<double, std::milli>(now - last).count());
    line += buf;
    last = now;
  }
  ~RunTrace() {
    if (on) fprintf(stderr, "[jxg_batch_run]%s | total %.1f ms\n", line.c_str(),
                    std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
  }
};

int jxg_batch_run(void* bp, void* cuda_stream) {
  Batch* b = static_cast<Batch*>(bp);
  if (!b || b->frames.empty()) return JXG_ERR_ARGUMENT;
  RunTrace trace;
  CUDA_TRY(cudaSetDevice(b->ctx->device));
  cudaStream_t s = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : b->ctx->stream;
  b->last_stream = s;
  b->h2d = b->d2h = 0;
  schedule_lean(b);
  // device allocations
  // one coefficient list per HF section (pass x group), worst-case capacity (every coefficient non-zero)
  if (int r = b->d_coeffs.ensure(b->sections.size() * size_t(kListStride) * 4)) return r;
  if (int r = b->d_block_off.ensure(b->total_blocks * 4)) return r;
  if (int r = b->ctx->d_lzwin.ensure(std::max<size_t>(size_t(b->lz_windows) * kLzWindow * 4, 16))) return r;
  if (int r = b->d_nz.ensure(b->nz_bytes)) return r;
  if (int r = b->d_planes_a.ensure(b->total_plane_floats * 4)) return r;
  if (int r = b->d_status.ensure((b->streams.size() + b->frames.size() + 4) * 4)) return r;
  if (int r = b->d_out.ensure(std::max<size_t>(b->out_bytes, 16))) return r;
  if (int r = b->ctx->d_lean_desc.ensure(std::max<size_t>(b->streams.size() * 1024 * 16, 16))) return r;
  if (int r = b->ctx->d_lean_nblk.ensure(std::max<size_t>(b->streams.size() * 4, 16))) return r;
  if (int r = b->ctx->d_orient.ensure(std::max<size_t>(b->orient_bytes, 16))) return r;
  for (size_t f = 0; f < b->frames.size(); f++) {
    const FrameOut& fo = b->outs[f];
    if (fo.orientation != 1) b->frames[f].out_ptr = static_cast<uint8_t*>(b->ctx->d_orient.p) + fo.stage_off;
    else b->frames[f].out_ptr = fo.is_device ? fo.user_ptr : static_cast<uint8_t*>(b->d_out.p) + fo.dev_off;
  }
  b->status_n = b->streams.size();
  if (b->status_n > b->ctx->status_cap) {
    if (b->ctx->status_host) cudaFreeHost(b->ctx->status_host);
    size_t cap = std::max<size_t>(b->status_n * 2, 1 << 16);
    CUDA_TRY(cudaHostAlloc(reinterpret_cast<void**>(&b->ctx->status_host), cap * 4, cudaHostAllocDefault));
    b->ctx->status_cap = cap;
  }
  b->status_host = b->ctx->status_host;
  memset(b->status_host, 0, b->status_n * 4);
  {  // batch tables behind the frames' data in the pinned blob: they travel with the one H2D copy below
    auto put = [&](const void* p, size_t bytes, uint64_t& off) {
      const int64_t o = b->blob.append(bytes ? p : nullptr, bytes, 16, 16);
      if (o < 0) return false;
      off = uint64_t(o);
      return true;
    };
    bool ok = put(b->frames.data(), b->frames.size() * sizeof(FrameDev), b->tab.frames) &&
              put(b->sections.data(), b->sections.size() * sizeof(SectionDev), b->tab.sections) &&
              put(b->streams.data(), b->streams.size() * sizeof(StreamDev), b->tab.streams) &&
              put(b->lean_cta_first.data(), b->lean_cta_first.size() * 4, b->tab.lean_cta) &&
              put(b->lean_warps.data(), b->lean_warps.size() * sizeof(uint2), b->tab.lean_warp) &&
              put(b->streams_lean.data(), b->streams_lean.size() * sizeof(StreamDev), b->tab.streams_lean) &&
              put(b->streams_fast.data(), b->streams_fast.size() * sizeof(StreamDev), b->tab.streams_fast) &&
              put(b->streams_slow.data(), b->streams_slow.size() * sizeof(StreamDev), b->tab.streams_slow) &&
              put(b->nz_base.data(), b->nz_base.size() * 8, b->tab.nz_base) &&
              put(b->fused_prefix.data(), b->fused_prefix.size() * 4, b->tab.ftiles);
    if (!ok) return set_error(JXG_ERR_CUDA, "pinned staging allocation failed");
  }
  if (int r = b->d_blob.ensure(b->blob.size + 64)) return r;
  trace.mark("alloc");
  b->blob.flush();
  trace.mark("flush");
  CUDA_TRY(cudaEventRecord(b->ev0, s));
  CUDA_TRY(cudaMemcpyAsync(b->d_blob.p, b->blob.p, b->blob.size, cudaMemcpyHostToDevice, s));
  trace.mark("blob_h2d");
  b->h2d += b->blob.size;
  b->uploaded = true;
  trace.mark("uploads");
  if (int r = launch(b, s, true)) return r;
  trace.mark("launch");
  if (int r = copy_status(b, s)) return r;
  // ev1 = everything of this batch done. The D2H stream joins the launching stream and carries ev1 when it holds the
  // output copies: the launching stream itself must not wait for them.
  if (b->debug_stop == 0) {
    Context* cx = b->ctx;
    CUDA_TRY(cudaEventRecord(cx->copy_done, s));
    CUDA_TRY(cudaStreamWaitEvent(cx->d2h_stream, cx->copy_done, 0));
    CUDA_TRY(cudaEventRecord(b->ev1, cx->d2h_stream));
  } else {
    CUDA_TRY(cudaEventRecord(b->ev1, s));
  }
  trace.mark("status");
  return JXG_OK;
}

int jxg_batch_rerun_device(void* bp, void* cuda_stream) {
  Batch* b = static_cast<Batch*>(bp);
  if (!b || !b->uploaded) return set_error(JXG_ERR_ARGUMENT, "batch was never submitted");
  CUDA_TRY(cudaSetDevice(b->ctx->device));
  cudaStream_t s = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : b->ctx->stream;
  b->last_stream = s;
  CUDA_TRY(cudaStreamWaitEvent(s, b->ev1, 0));  // the previous run of this batch still owns its device buffers
  CUDA_TRY(cudaEventRecord(b->ev0, s));
  if (int r = launch(b, s, false)) return r;
  CUDA_TRY(cudaMemcpyAsync(b->status_host, b->d_status.p, b->status_n * 4, cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaEventRecord(b->ev1, s));
  return JXG_OK;
}

int jxg_batch_wait(void* bp, uint32_t* first_bad_frame, uint32_t* first_bad_group) {
  Batch* b = static_cast<Batch*>(bp);
  if (!b) return JXG_ERR_ARGUMENT;
  CUDA_TRY(cudaSetDevice(b->ctx->device));
  {
    static const bool traced = getenv("JXG_TRACE_RUN") && atoi(getenv("JXG_TRACE_RUN")) != 0;
    const auto t0 = std::chrono::steady_clock::now();
    const bool was_done = traced && cudaEventQuery(b->ev1) == cudaSuccess;
    CUDA_TRY(cudaEventSynchronize(b->ev1));  // recorded behind the status words and the D2H copies; no stream-wide wait:
                                             // the D2H stream carries later batches too
    if (traced)
      fprintf(stderr, "[jxg_batch_wait] done on entry %d, event wait %.1f ms\n", int(was_done),
              std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
  }
  CUDA_TRY(cudaGetLastError());
  cudaEventElapsedTime(&b->last_ms, b->ev0, b->ev1);
  for (size_t i = 0; i < b->status_n; i++)
    if (b->status_host[i] != 0) {
      if (first_bad_frame) *first_bad_frame = b->streams[i].frame;
      if (first_bad_group) *first_bad_group = b->streams[i].group;
      return set_error(b->status_host[i], "entropy decode failed in frame " + std::to_string(b->streams[i].frame) +
                                              " group " + std::to_string(b->streams[i].group));
    }
  return JXG_OK;
}

int jxg_batch_stats(void* bp, uint64_t* kernel_launches, uint64_t* h2d_bytes, uint64_t* d2h_bytes, float* last_device_ms) {
  Batch* b = static_cast<Batch*>(bp);
  if (!b) return JXG_ERR_ARGUMENT;
  if (kernel_launches) *kernel_launches = b->launches;
  if (h2d_bytes) *h2d_bytes = b->h2d;
  if (d2h_bytes) *d2h_bytes = b->d2h;
  if (last_device_ms) *last_device_ms = b->last_ms;
  return JXG_OK;
}

int jxg_batch_read_coeffs(void* bp, uint32_t f, int32_t* out, size_t out_len) {
  Batch* b = static_cast<Batch*>(bp);
  if (!b || f >= b->frames.size() || !b->uploaded) return JXG_ERR_ARGUMENT;
  const FrameDev& F = b->frames[f];
  size_t n = size_t(F.num_groups) * 3 * kGroupCoeffs;
  if (out_len < n) return JXG_ERR_ARGUMENT;
  CUDA_TRY(cudaSetDevice(b->ctx->device));
  cudaStream_t s = b->last_stream ? b->last_stream : b->ctx->stream;
  CUDA_TRY(cudaStreamSynchronize(s));
  // The device holds lists of non-zero coefficients; the tap expands them into the reference's dense layout.
  DevBuf dense;
  if (int r = dense.ensure(n * 4)) return r;
  CUDA_TRY(cudaMemsetAsync(dense.p, 0, n * 4, s));
  launch_expand_coeffs(make_batch_dev(b), f, F.num_groups, static_cast<int32_t*>(dense.p), s);
  CUDA_TRY(cudaMemcpyAsync(out, dense.p, n * 4, cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaStreamSynchronize(s));
  return JXG_OK;
}

int jxg_batch_read_xyb(void* bp, uint32_t f, int stage, float* out, size_t out_len) {
  Batch* b = static_cast<Batch*>(bp);
  if (!b || f >= b->frames.size() || !b->uploaded || stage != 0) return JXG_ERR_ARGUMENT;
  const FrameDev& F = b->frames[f];
  size_t n = 3 * F.plane_size;
  if (out_len < n) return JXG_ERR_ARGUMENT;
  CUDA_TRY(cudaSetDevice(b->ctx->device));
  CUDA_TRY(cudaStreamSynchronize(b->ctx->stream));
  CUDA_TRY(cudaMemcpy(out, static_cast<const float*>(b->d_planes_a.p) + F.plane_base, n * 4, cudaMemcpyDeviceToHost));
  return JXG_OK;
}

// ---------------- host front-end convenience ----------------

int jxg_parse_file(const uint8_t* data, size_t size, void** parsed, JxgImageInfo* info) {
  return jxg_parse_file_mt(data, size, 1, parsed, info);
}

int jxg_parse_file_mt(const uint8_t* data, size_t size, int threads, void** parsed, JxgImageInfo* info) {
  if (!data || !parsed) return JXG_ERR_ARGUMENT;
  try {
    std::unique_ptr<jxg::FrameState> fs = jxg::parse_vardct_file(data, size, threads);
    if (info) {
      info->coded_width = fs->header.xsize();
      info->coded_height = fs->header.ysize();
      info->orientation = fs->file.orientation;
      info->width = fs->file.orientation >= 5 ? info->coded_height : info->coded_width;
      info->height = fs->file.orientation >= 5 ? info->coded_width : info->coded_height;
      info->num_groups = fs->header.num_groups();
      info->num_passes = fs->header.passes.num_passes;
      info->encoding = 0;
      info->hf_bytes = 0;
      for (uint32_t l : fs->hf_len) info->hf_bytes += l;
    }
    *parsed = fs.release();
    return JXG_OK;
  } catch (jxg::Error& e) {
    return set_error(e.code, e.what());
  } catch (std::exception& e) {
    return set_error(JXG_ERR_BITSTREAM, e.what());
  }
}

void jxg_parsed_free(void* parsed) { jxg::recycle_frame_state(static_cast<jxg::FrameState*>(parsed)); }

int jxg_parsed_desc(void* parsed, uint32_t output_format, JxgFrameDesc* desc, const uint8_t** hf_bytes,
                    const uint64_t** sec_off, const uint32_t** sec_len, uint32_t* n_sections) {
  jxg::FrameState* fs = static_cast<jxg::FrameState*>(parsed);
  if (!fs || !desc) return JXG_ERR_ARGUMENT;
  fs->fill_desc(desc, output_format);
  if (hf_bytes) *hf_bytes = fs->codestream.data();
  if (sec_off) *sec_off = fs->hf_off.data();
  if (sec_len) *sec_len = fs->hf_len.data();
  if (n_sections) *n_sections = uint32_t(fs->hf_off.size());
  return JXG_OK;
}

int jxg_batch_add_parsed(void* batch, void* parsed, uint32_t output_format, void* out, size_t out_row_stride,
                         int out_is_device) {
  jxg::FrameState* fs = static_cast<jxg::FrameState*>(parsed);
  if (!fs) return JXG_ERR_ARGUMENT;
  JxgFrameDesc d;
  fs->fill_desc(&d, output_format);
  return add_frame_impl(batch, &d, fs->codestream.data(), fs->hf_off.data(), fs->hf_len.data(), uint32_t(fs->hf_off.size()), out,
                        out_row_stride, out_is_device, /*trusted=*/true);
}

}  // extern "C"
