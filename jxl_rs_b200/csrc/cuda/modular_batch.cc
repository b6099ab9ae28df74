// C ABI of the Modular-frame path (jxg_modular_*, include/jxg.h): batches of Modular frames whose ModularHF
// sections are decoded on the GPU (modular_kernels.cu). Host work: the front end (modular_frame.cc) and the staging
// of tables, sections and the host-decoded small channels into one pinned blob.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <tuple>
#include <utility>
#include <vector>

#include "../../../include/jxg.h"
#include "../host/modular_frame.h"
#include "batch_common.h"
#include "modular_device.h"

using namespace jxgpu;
using namespace jxgpu::detail;

namespace {

struct MFrame {
  jxg::ModularFrameState* ms;
  void* out;
  size_t out_stride;
  bool out_is_device;
  uint64_t arena_base = 0;         // element offset of this frame's planes
  std::vector<uint64_t> buf_off;   // per plan buffer, element offset in the arena
  uint64_t host_planes_blob = 0;   // blob offset of the packed host-decoded planes
  uint64_t host_planes_elems = 0;
  size_t dev_out_off = 0;
  uint32_t first_stream = 0, num_streams = 0;
};

struct ModularBatch {
  Context* ctx;
  std::vector<MFrame> frames;
  std::vector<MStreamDev> streams;
  std::vector<uint32_t> order, rct_streams;
  std::vector<MRectDev> rects;
  std::vector<MCodeDev> codes;
  std::vector<MRctDev> rcts;
  std::vector<uint32_t> refs;
  std::vector<std::vector<MJobDev>> levels;  // jobs grouped by plan step index
  std::vector<int> level_kind;
  std::vector<MJobDev> store_jobs;
  uint64_t arena_elems = 0, wp_bytes = 0, out_bytes = 0;
  std::vector<uint32_t> stream_frame_group;  // for error reports
  bool uploaded = false;
  uint64_t launches = 0, h2d = 0, d2h = 0;
  uint32_t lanes_per_warp = 1;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_decode = nullptr;
  int32_t* status_host = nullptr;
  // device pools (context-owned buffers are reused where the meaning matches)
  DevBuf d_streams, d_order, d_rct_streams, d_rects, d_codes, d_rcts, d_refs, d_jobs, d_wp;
};

uint64_t blob_append(ModularBatch* b, const void* p, size_t bytes, size_t align = 16, size_t tail = 0) {
  int64_t o = b->ctx->blob.append(p, bytes, align, tail);
  if (o < 0) throw jxg::Error(JXG_ERR_CUDA, "pinned staging allocation failed");
  return uint64_t(o);
}

uint32_t add_code(ModularBatch* b, const jxg::EntropyCode& c) {
  if (c.lz77_enabled) throw jxg::Error(JXG_ERR_UNSUPPORTED, "LZ77 in Modular group streams is not implemented on the device path");
  MCodeDev d;
  memset(&d, 0, sizeof(d));
  d.use_prefix = c.use_prefix;
  d.log_alpha = c.log_alpha_size;
  d.num_clusters = c.num_clusters;
  d.cmap_off = blob_append(b, c.context_map.data(), c.context_map.size());
  std::vector<uint32_t> cfg;
  for (const auto& u : c.uint_configs) cfg.push_back(u.packed());
  d.cfg_off = blob_append(b, cfg.data(), cfg.size() * 4);
  if (c.use_prefix) {
    d.huff_off = blob_append(b, c.huff_entries.data(), c.huff_entries.size() * 4);
    d.huff_offset_off = blob_append(b, c.huff_offset.data(), c.huff_offset.size() * 4);
  } else {
    d.ans_off = blob_append(b, c.ans_buckets.data(), c.ans_buckets.size() * 8);
  }
  b->codes.push_back(d);
  return uint32_t(b->codes.size() - 1);
}

uint64_t add_tree(ModularBatch* b, const jxg::ModularTree& t) {
  std::vector<int32_t> nodes(t.nodes.size() * 4);
  for (size_t i = 0; i < t.nodes.size(); i++) {
    const jxg::TreeNode& n = t.nodes[i];
    nodes[i * 4 + 0] = n.property;
    nodes[i * 4 + 1] = n.val;
    if (n.property >= 0) {
      nodes[i * 4 + 2] = int32_t(n.left);
      nodes[i * 4 + 3] = 0;
    } else {
      if (n.ctx >= (1u << 27)) throw jxg::Error(JXG_ERR_UNSUPPORTED, "MA tree too large for the device encoding");
      nodes[i * 4 + 2] = int32_t(n.left | (n.ctx << 4));  // predictor | ctx << 4
      nodes[i * 4 + 3] = int32_t(n.right);                // multiplier
    }
  }
  return blob_append(b, nodes.data(), nodes.size() * 4, 16);
}

// Table form of a channel's tree walk (see modular_device.h). Returns false when the channel needs the generic walk.
// `root`: first node whose decision is not on the channel index / stream id. Keys of the cache: (tree, root).
struct WalkKey {
  uint64_t tree_off;
  uint32_t root, ci;
  uint64_t stream_id;
  bool operator<(const WalkKey& o) const {
    return std::tie(tree_off, root, ci, stream_id) < std::tie(o.tree_off, o.root, o.ci, o.stream_id);
  }
};

// Does the tree decide on the channel index / stream id (properties 0 / 1) below a split on another property?
bool has_inner_static(const jxg::ModularTree& t) {
  std::vector<std::pair<uint32_t, bool>> stack{{0u, false}};
  while (!stack.empty()) {
    auto [n, below] = stack.back();
    stack.pop_back();
    const jxg::TreeNode& nd = t.nodes[n];
    if (nd.property < 0) continue;
    const bool is_static = nd.property == 0 || nd.property == 1;
    if (is_static && below) return true;
    stack.push_back({nd.left, below || !is_static});
    stack.push_back({nd.right, below || !is_static});
  }
  return false;
}
struct WalkInfo {
  uint32_t walk;
  uint64_t lut_off;
};

uint32_t static_root(const jxg::ModularTree& t, uint32_t ci, uint64_t stream_id) {
  uint32_t n = 0;
  while (t.nodes[n].property == 0 || t.nodes[n].property == 1) {
    const int64_t v = t.nodes[n].property == 0 ? int64_t(ci) : int64_t(int32_t(uint32_t(stream_id)));
    n = v > int64_t(t.nodes[n].val) ? t.nodes[n].left : t.nodes[n].right;
  }
  return n;
}

bool build_walk_table(const jxg::ModularTree& t, uint32_t root, uint32_t ci, uint64_t stream_id, std::vector<uint32_t>& lut,
                      uint32_t& prop, uint32_t& single) {
  struct Item {
    int32_t lo, hi;  // [lo, hi)
    uint32_t node;
  };
  auto entry = [&](uint32_t node, uint32_t& e) {
    const jxg::TreeNode& n = t.nodes[node];
    if (node >= (1u << 16) || n.ctx >= t.code.context_map.size()) return false;
    const uint32_t cluster = t.code.context_map[n.ctx];
    const bool plain = n.val == 0 && n.right == 1;
    e = (n.left & 15u) | (cluster << 4) | (plain ? 1u << 12 : 0u) | (node << 16);
    return true;
  };
  prop = kLutNoProperty;
  lut.assign(kLutSize, 0);
  std::vector<Item> stack{Item{kLutMin, kLutMin + kLutSize, root}};
  bool any_split = false;
  while (!stack.empty()) {
    Item it = stack.back();
    stack.pop_back();
    uint32_t node = it.node;
    // decisions on the channel / stream below other splits are still constant
    while (t.nodes[node].property == 0 || t.nodes[node].property == 1) {
      const int64_t v = t.nodes[node].property == 0 ? int64_t(ci) : int64_t(int32_t(uint32_t(stream_id)));
      node = v > int64_t(t.nodes[node].val) ? t.nodes[node].left : t.nodes[node].right;
    }
    const jxg::TreeNode& n = t.nodes[node];
    if (n.property < 0) {
      uint32_t e;
      if (!entry(node, e)) return false;
      for (int32_t v = it.lo; v < it.hi; v++) lut[size_t(v - kLutMin)] = e;
      single = e;
      continue;
    }
    if (n.property < 2 || n.property > 15) return false;  // properties of previous channels: generic walk
    if (prop == kLutNoProperty) prop = uint32_t(n.property);
    else if (prop != uint32_t(n.property)) return false;
    // values beyond the table are clamped to its ends: the decision must not change there
    if (n.val < kLutMin || n.val > kLutMin + kLutSize - 2) return false;
    any_split = true;
    const int32_t first_left = n.val + 1;  // v > val -> left child
    if (first_left < it.hi) stack.push_back(Item{std::max(first_left, it.lo), it.hi, n.left});
    if (first_left > it.lo) stack.push_back(Item{it.lo, std::min(first_left, it.hi), n.right});
  }
  if (!any_split) prop = kLutNoProperty;
  return true;
}

void add_frame(ModularBatch* b, jxg::ModularFrameState* ms, void* out, size_t stride, bool is_device) {
  if (!ms->device_plan_ok)
    throw jxg::Error(JXG_ERR_UNSUPPORTED, "palette transforms with delta entries or a predictor are not implemented on the device path");
  if (ms->toc.offsets.size() == 1 && !ms->hf[0].empty)
    throw jxg::Error(JXG_ERR_UNSUPPORTED, "single-section Modular frames with a coded group are not on the device path");
  MFrame f;
  f.ms = ms;
  f.out = out;
  f.out_stride = stride;
  f.out_is_device = is_device;
  const uint32_t W = ms->header.xsize(), H = ms->header.ysize();
  const uint32_t orient = ms->file.orientation;  // applied by the store kernel (render/save.rs)
  if (stride < size_t(orient >= 5 ? H : W) * 3) throw jxg::Error(JXG_ERR_INVALID_OUTPUT, "output row stride too small");
  // ---- plane arena: host-decoded coded channels first (one contiguous upload), then the rest ----
  f.arena_base = b->arena_elems;
  f.buf_off.assign(ms->bufs.size(), 0);
  uint64_t cursor = f.arena_base;
  std::vector<int32_t> packed;
  for (size_t c = 0; c < ms->coded.size(); c++)
    if (ms->host_decoded[c]) {
      f.buf_off[c] = cursor;
      cursor += uint64_t(ms->bufs[c].w) * ms->bufs[c].h;
    }
  f.host_planes_elems = cursor - f.arena_base;
  for (size_t i = 0; i < ms->bufs.size(); i++)
    if (i >= ms->coded.size() || !ms->host_decoded[i]) {
      cursor = (cursor + 3) & ~uint64_t(3);
      f.buf_off[i] = cursor;
      cursor += uint64_t(ms->bufs[i].w) * ms->bufs[i].h;
    }
  b->arena_elems = (cursor + 63) & ~uint64_t(63);
  if (f.host_planes_elems) {
    f.host_planes_blob = uint64_t(b->ctx->blob.append(nullptr, 0, 16, 0));
    for (size_t c = 0; c < ms->coded.size(); c++)
      if (ms->host_decoded[c] && !ms->coded[c].data.empty()) blob_append(b, ms->coded[c].data.data(), ms->coded[c].data.size() * 4, 4);
  }
  // ---- codes / trees ----
  uint32_t global_code = 0;
  uint64_t global_tree = 0;
  bool have_global = false;
  std::map<WalkKey, WalkInfo> walk_cache;
  std::map<uint64_t, bool> inner_static;
  f.first_stream = uint32_t(b->streams.size());
  for (const jxg::ModularGroupStream& st : ms->hf) {
    if (st.empty) continue;
    const jxg::ModularTree* tree = st.local_tree ? st.local_tree.get() : &ms->global_tree;
    MStreamDev d;
    memset(&d, 0, sizeof(d));
    if (st.local_tree) {
      d.code = add_code(b, tree->code);
      d.tree_off = add_tree(b, *tree);
    } else {
      if (!have_global) {
        global_code = add_code(b, tree->code);
        global_tree = add_tree(b, *tree);
        have_global = true;
      }
      d.code = global_code;
      d.tree_off = global_tree;
    }
    d.frame = uint32_t(b->frames.size());
    d.group = st.group;
    d.sec_off = blob_append(b, ms->codestream.data() + st.sec_off, st.sec_len, 8, 24);
    d.sec_len = st.sec_len;
    d.data_bitpos = uint32_t(st.data_bitpos);
    d.stream_id = uint32_t(st.stream_id);
    d.uses_wp = tree->uses_wp;
    const jxg::WeightedHeader& wp = st.header.wp;
    const uint32_t wpp[11] = {wp.p1c, wp.p2c, wp.p3ca, wp.p3cb, wp.p3cc, wp.p3cd, wp.p3ce, wp.w[0], wp.w[1], wp.w[2], wp.w[3]};
    memcpy(d.wp_params, wpp, sizeof(wpp));
    d.first_rect = uint32_t(b->rects.size());
    d.num_rects = uint32_t(st.rects.size());
    uint32_t max_w = 0;
    for (size_t ri = 0; ri < st.rects.size(); ri++) {
      const jxg::ModularRect& r = st.rects[ri];
      MRectDev rd;
      rd.stride = ms->coded[r.chan].w;
      rd.base = f.buf_off[r.chan] + uint64_t(r.y0) * rd.stride + r.x0;
      rd.w = r.w;
      rd.h = r.h;
      rd.walk = kWalkGeneric;
      rd.lut_off = 0;
      if (r.w && r.h) {
        const uint32_t root = static_root(*tree, uint32_t(ri), st.stream_id);
        // channel / stream decisions below another split make the table specific to this channel of this stream
        auto is_it = inner_static.find(d.tree_off);
        if (is_it == inner_static.end()) is_it = inner_static.emplace(d.tree_off, has_inner_static(*tree)).first;
        const WalkKey key{d.tree_off, root, is_it->second ? uint32_t(ri) : ~0u, is_it->second ? st.stream_id : ~uint64_t(0)};
        auto it = walk_cache.find(key);
        if (it == walk_cache.end()) {
          std::vector<uint32_t> lut;
          uint32_t prop = kLutNoProperty, single = 0;
          WalkInfo wi{kWalkGeneric, 0};
          if (build_walk_table(*tree, root, uint32_t(ri), st.stream_id, lut, prop, single)) {
            wi.walk = kWalkLut | (prop << 8);
            wi.lut_off = prop == kLutNoProperty ? uint64_t(single) : blob_append(b, lut.data(), lut.size() * 4, 16);
          }
          it = walk_cache.emplace(key, wi).first;
        }
        rd.walk = it->second.walk;
        rd.lut_off = it->second.lut_off;
      }
      // reference channels: earlier channels of the stream with the same shape, nearest first (common.rs:52-60)
      rd.ref_first = uint32_t(b->refs.size());
      if (tree->num_properties > 16)
        for (size_t k = ri; k-- > 0;) {
          const jxg::ModularRect& q = st.rects[k];
          if (q.w == r.w && q.h == r.h && ms->coded[q.chan].hshift == ms->coded[r.chan].hshift &&
              ms->coded[q.chan].vshift == ms->coded[r.chan].vshift)
            b->refs.push_back(d.first_rect + uint32_t(k));
        }
      rd.ref_count = uint32_t(b->refs.size()) - rd.ref_first;
      b->rects.push_back(rd);
      max_w = std::max(max_w, r.w);
    }
    if (d.uses_wp) {
      d.wp_scratch_off = b->wp_bytes;
      b->wp_bytes += (size_t(max_w + 1) * (8 + 2) * 4 + 63) & ~size_t(63);
    }
    d.first_rct = uint32_t(b->rcts.size());
    for (const jxg::ModularTransform& t : st.header.transforms) {
      if (t.id != 0) throw jxg::Error(JXG_ERR_UNSUPPORTED, "only RCT is implemented as a group-local transform on the device path");
      if (t.begin_channel + 3 > st.rects.size()) throw jxg::Error(jxg::kErrBitstream, "RCT channel range");
      const jxg::ModularRect &r0 = st.rects[t.begin_channel], &r1 = st.rects[t.begin_channel + 1], &r2 = st.rects[t.begin_channel + 2];
      if (r0.w != r1.w || r0.w != r2.w || r0.h != r1.h || r0.h != r2.h) throw jxg::Error(jxg::kErrBitstream, "RCT on channels of different size");
      b->rcts.push_back(MRctDev{t.begin_channel, t.rct_type});
    }
    d.num_rct = uint32_t(b->rcts.size()) - d.first_rct;
    if (d.num_rct) b->rct_streams.push_back(uint32_t(b->streams.size()));
    b->streams.push_back(d);
  }
  f.num_streams = uint32_t(b->streams.size()) - f.first_stream;
  // ---- global inverse plan -> jobs per level ----
  for (size_t si = 0; si < ms->steps.size(); si++) {
    const jxg::ModularStep& s = ms->steps[si];
    if (b->levels.size() <= si) {
      b->levels.emplace_back();
      b->level_kind.push_back(int(s.kind));
    }
    if (b->level_kind[si] != int(s.kind))
      throw jxg::Error(JXG_ERR_UNSUPPORTED, "frames of one Modular batch must share the global transform structure");
    MJobDev j;
    memset(&j, 0, sizeof(j));
    j.a = f.buf_off[s.a];
    j.b = f.buf_off[s.b];
    j.c = f.buf_off[s.c];
    j.w = ms->bufs[s.a].w;
    j.h = ms->bufs[s.a].h;
    j.rw = s.kind == 1 ? ms->bufs[s.b].w : (s.kind == 2 ? ms->bufs[s.b].h : 0);
    j.op = s.rct_op;
    if (s.kind == 3) {  // one job per colour channel: a index plane, b palette plane (row c = component c), c output
      if (ms->bufs[s.b].h < s.n || ms->bufs[s.b].w < s.num_colors) throw jxg::Error(jxg::kErrBitstream, "palette channel smaller than its header says");
      for (uint32_t c = 0; c < s.n; c++) {
        j.c = f.buf_off[s.c + c];
        j.rw = s.num_colors;
        j.op = c;
        j.out_stride = ms->bufs[s.b].w;  // palette row stride
        b->levels[si].push_back(j);
      }
      continue;
    }
    b->levels[si].push_back(j);
  }
  if (ms->steps.size() < b->levels.size() && !b->frames.empty())
    throw jxg::Error(JXG_ERR_UNSUPPORTED, "frames of one Modular batch must share the global transform structure");
  MJobDev sj;
  memset(&sj, 0, sizeof(sj));
  const uint32_t nc = ms->num_color_channels;
  sj.a = f.buf_off[ms->out_buf[0]];
  sj.b = f.buf_off[ms->out_buf[nc > 1 ? 1 : 0]];
  sj.c = f.buf_off[ms->out_buf[nc > 2 ? 2 : 0]];
  sj.w = W;
  sj.h = H;
  sj.op = orient;
  for (uint32_t c = 0; c < nc; c++)
    if (ms->bufs[ms->out_buf[c]].w != W || ms->bufs[ms->out_buf[c]].h != H)
      throw jxg::Error(jxg::kErrBitstream, "unexpected output channel size");
  if (!is_device) {
    f.dev_out_off = b->out_bytes;
    b->out_bytes += (size_t(W) * H * 3 + 255) & ~size_t(255);
  }
  b->store_jobs.push_back(sj);
  b->frames.push_back(std::move(f));
}

int launch_all(ModularBatch* b, cudaStream_t s, bool copy_to_host) {
  Context* cx = b->ctx;
  MBatchDev B;
  memset(&B, 0, sizeof(B));
  B.blob = static_cast<const uint8_t*>(cx->d_blob.p);
  B.streams = static_cast<const MStreamDev*>(b->d_streams.p);
  B.order = static_cast<const uint32_t*>(b->d_order.p);
  B.rct_streams = static_cast<const uint32_t*>(b->d_rct_streams.p);
  B.rects = static_cast<const MRectDev*>(b->d_rects.p);
  B.codes = static_cast<const MCodeDev*>(b->d_codes.p);
  B.rcts = static_cast<const MRctDev*>(b->d_rcts.p);
  B.refs = static_cast<const uint32_t*>(b->d_refs.p);
  B.planes = static_cast<int32_t*>(cx->d_planes_a.p);
  B.wp_scratch = static_cast<uint8_t*>(b->d_wp.p);
  B.status = static_cast<int32_t*>(cx->d_status.p);
  B.queue = reinterpret_cast<uint32_t*>(B.status + b->streams.size());
  B.num_streams = uint32_t(b->streams.size());
  // host-decoded planes: blob -> arena (device to device)
  for (const MFrame& f : b->frames)
    if (f.host_planes_elems)
      CUDA_TRY(cudaMemcpyAsync(B.planes + f.arena_base, B.blob + f.host_planes_blob, f.host_planes_elems * 4,
                               cudaMemcpyDeviceToDevice, s));
  uint64_t launches = uint64_t(launch_modular_decode(B, b->lanes_per_warp, uint32_t(b->rct_streams.size()), s));
  if (b->ev_decode) CUDA_TRY(cudaEventRecord(b->ev_decode, s));
  const MJobDev* jobs = static_cast<const MJobDev*>(b->d_jobs.p);
  size_t job_cursor = 0;
  for (size_t l = 0; l < b->levels.size(); l++) {
    uint32_t mw = 0, mh = 0;
    for (const MJobDev& j : b->levels[l]) {
      mw = std::max(mw, j.w);
      mh = std::max(mh, j.h);
    }
    launch_modular_jobs(b->level_kind[l] == 3 ? 4 : b->level_kind[l], jobs + job_cursor, uint32_t(b->levels[l].size()), mw, mh, B.planes, s);
    job_cursor += b->levels[l].size();
    launches++;
  }
  {
    uint32_t mw = 0, mh = 0;
    for (const MJobDev& j : b->store_jobs) {
      mw = std::max(mw, j.w);
      mh = std::max(mh, j.h);
    }
    launch_modular_jobs(3, jobs + job_cursor, uint32_t(b->store_jobs.size()), mw, mh, B.planes, s);
    launches++;
  }
  b->launches = launches;
  if (copy_to_host) {
    for (const MFrame& f : b->frames)
      if (!f.out_is_device) {
        const bool tr = f.ms->file.orientation >= 5;  // display size
        const uint32_t W = tr ? f.ms->header.ysize() : f.ms->header.xsize(), H = tr ? f.ms->header.xsize() : f.ms->header.ysize();
        CUDA_TRY(cudaMemcpy2DAsync(f.out, f.out_stride, static_cast<uint8_t*>(cx->d_out.p) + f.dev_out_off, size_t(W) * 3,
                                   size_t(W) * 3, H, cudaMemcpyDeviceToHost, s));
        b->d2h += size_t(W) * 3 * H;
      }
  }
  CUDA_TRY(cudaMemcpyAsync(b->status_host, cx->d_status.p, b->streams.size() * 4, cudaMemcpyDeviceToHost, s));
  CUDA_TRY(cudaGetLastError());
  return 0;
}

}  // namespace

extern "C" {

int jxg_modular_parse_file(const uint8_t* data, size_t size, void** parsed, JxgImageInfo* info) {
  if (!data || !parsed) return JXG_ERR_ARGUMENT;
  try {
    auto ms = jxg::parse_modular_file(data, size);
    if (info) {
      memset(info, 0, sizeof(*info));
      info->coded_width = ms->header.xsize();
      info->coded_height = ms->header.ysize();
      info->orientation = ms->file.orientation;
      info->width = ms->file.orientation >= 5 ? info->coded_height : info->coded_width;
      info->height = ms->file.orientation >= 5 ? info->coded_width : info->coded_height;
      info->num_groups = ms->header.num_groups();
      info->num_passes = 1;
      info->encoding = 1;
      uint64_t hf = 0;
      for (const auto& st : ms->hf) hf += st.sec_len;
      info->hf_bytes = hf;
    }
    *parsed = ms.release();
    return JXG_OK;
  } catch (jxg::Error& e) {
    return set_error(e.code, e.what());
  }
}

void jxg_modular_parsed_free(void* parsed) { delete static_cast<jxg::ModularFrameState*>(parsed); }

int jxg_modular_batch_begin(void* c, void** out_batch) {
  if (!c || !out_batch) return JXG_ERR_ARGUMENT;
  Context* cx = static_cast<Context*>(c);
  if (cx->batch_live) return set_error(JXG_ERR_ARGUMENT, "one live batch per context: end the previous batch first");
  CUDA_TRY(cudaSetDevice(cx->device));
  auto b = std::make_unique<ModularBatch>();
  b->ctx = cx;
  cx->blob.size = 0;
  cx->blob.pending.clear();
  cx->blob.deferred_threads = 0;
  cx->batch_live = true;
  CUDA_TRY(cudaEventCreate(&b->ev0));
  CUDA_TRY(cudaEventCreate(&b->ev1));
  CUDA_TRY(cudaEventCreate(&b->ev_decode));
  *out_batch = b.release();
  return JXG_OK;
}

int jxg_modular_batch_add(void* bp, void* parsed, void* out, size_t out_row_stride, int out_is_device) {
  ModularBatch* b = static_cast<ModularBatch*>(bp);
  if (!b || !parsed || !out) return JXG_ERR_ARGUMENT;
  if (b->uploaded) return set_error(JXG_ERR_ARGUMENT, "batch already submitted");
  try {
    add_frame(b, static_cast<jxg::ModularFrameState*>(parsed), out, out_row_stride, out_is_device != 0);
    return JXG_OK;
  } catch (jxg::Error& e) {
    return set_error(e.code, e.what());
  }
}

int jxg_modular_batch_set_lanes(void* bp, int lanes_per_warp) {
  ModularBatch* b = static_cast<ModularBatch*>(bp);
  if (!b || lanes_per_warp < 1) return JXG_ERR_ARGUMENT;
  b->lanes_per_warp = uint32_t(lanes_per_warp);
  return JXG_OK;
}

int jxg_modular_batch_run(void* bp, void* cuda_stream) {
  ModularBatch* b = static_cast<ModularBatch*>(bp);
  if (!b || b->frames.empty()) return JXG_ERR_ARGUMENT;
  Context* cx = b->ctx;
  CUDA_TRY(cudaSetDevice(cx->device));
  cudaStream_t s = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : cx->stream;
  b->h2d = b->d2h = 0;
  // longest section first (the decode kernel's queue is a longest-processing-time schedule)
  b->order.resize(b->streams.size());
  for (uint32_t i = 0; i < b->order.size(); i++) b->order[i] = i;
  std::stable_sort(b->order.begin(), b->order.end(), [&](uint32_t x, uint32_t y) { return b->streams[x].sec_len > b->streams[y].sec_len; });
  if (int r = cx->d_blob.ensure(cx->blob.size + 64)) return r;
  if (int r = cx->d_planes_a.ensure(std::max<size_t>(b->arena_elems * 4, 16))) return r;
  if (int r = cx->d_status.ensure((b->streams.size() + 8) * 4)) return r;
  if (int r = cx->d_out.ensure(std::max<size_t>(b->out_bytes, 16))) return r;
  if (int r = b->d_wp.ensure(std::max<size_t>(b->wp_bytes, 16))) return r;
  for (size_t i = 0; i < b->frames.size(); i++) {
    MFrame& f = b->frames[i];
    b->store_jobs[i].out = f.out_is_device ? f.out : static_cast<uint8_t*>(cx->d_out.p) + f.dev_out_off;
    b->store_jobs[i].out_stride =
        f.out_is_device ? f.out_stride : size_t(f.ms->file.orientation >= 5 ? f.ms->header.ysize() : f.ms->header.xsize()) * 3;
  }
  if (b->streams.size() > cx->status_cap) {
    if (cx->status_host) cudaFreeHost(cx->status_host);
    size_t cap = std::max<size_t>(b->streams.size() * 2, 1 << 16);
    CUDA_TRY(cudaHostAlloc(reinterpret_cast<void**>(&cx->status_host), cap * 4, cudaHostAllocDefault));
    cx->status_cap = cap;
  }
  b->status_host = cx->status_host;
  memset(b->status_host, 0, b->streams.size() * 4);
  std::vector<MJobDev> all_jobs;
  for (auto& l : b->levels) all_jobs.insert(all_jobs.end(), l.begin(), l.end());
  all_jobs.insert(all_jobs.end(), b->store_jobs.begin(), b->store_jobs.end());
  CUDA_TRY(cudaEventRecord(b->ev0, s));
  CUDA_TRY(cudaMemcpyAsync(cx->d_blob.p, cx->blob.p, cx->blob.size, cudaMemcpyHostToDevice, s));
  b->h2d += cx->blob.size;
  if (int r = upload(b->d_streams, b->streams, s, &b->h2d)) return r;
  if (int r = upload(b->d_order, b->order, s, &b->h2d)) return r;
  if (int r = upload(b->d_rct_streams, b->rct_streams, s, &b->h2d)) return r;
  if (int r = upload(b->d_rects, b->rects, s, &b->h2d)) return r;
  if (int r = upload(b->d_codes, b->codes, s, &b->h2d)) return r;
  if (int r = upload(b->d_rcts, b->rcts, s, &b->h2d)) return r;
  if (int r = upload(b->d_refs, b->refs, s, &b->h2d)) return r;
  if (int r = upload(b->d_jobs, all_jobs, s, &b->h2d)) return r;
  b->uploaded = true;
  if (int r = launch_all(b, s, true)) return r;
  CUDA_TRY(cudaEventRecord(b->ev1, s));
  return JXG_OK;
}

int jxg_modular_batch_rerun_device(void* bp, void* cuda_stream) {
  ModularBatch* b = static_cast<ModularBatch*>(bp);
  if (!b || !b->uploaded) return set_error(JXG_ERR_ARGUMENT, "batch was never submitted");
  CUDA_TRY(cudaSetDevice(b->ctx->device));
  cudaStream_t s = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : b->ctx->stream;
  CUDA_TRY(cudaEventRecord(b->ev0, s));
  if (int r = launch_all(b, s, false)) return r;
  CUDA_TRY(cudaEventRecord(b->ev1, s));
  return JXG_OK;
}

int jxg_modular_batch_wait(void* bp, uint32_t* bad_frame, uint32_t* bad_group) {
  ModularBatch* b = static_cast<ModularBatch*>(bp);
  if (!b || !b->uploaded) return JXG_ERR_ARGUMENT;
  CUDA_TRY(cudaSetDevice(b->ctx->device));
  CUDA_TRY(cudaEventSynchronize(b->ev1));
  for (size_t i = 0; i < b->streams.size(); i++)
    if (b->status_host[i] != 0) {
      if (bad_frame) *bad_frame = b->streams[i].frame;
      if (bad_group) *bad_group = b->streams[i].group;
      return set_error(b->status_host[i], "Modular group stream failed: frame " + std::to_string(b->streams[i].frame) + " group " +
                                              std::to_string(b->streams[i].group));
    }
  return JXG_OK;
}

// Parity tap: the final colour planes (3 x H x W i32, before the u8 conversion) of frame f.
int jxg_modular_batch_read_planes(void* bp, uint32_t f, int32_t* out, size_t out_len) {
  ModularBatch* b = static_cast<ModularBatch*>(bp);
  if (!b || !b->uploaded || f >= b->frames.size() || !out) return JXG_ERR_ARGUMENT;
  CUDA_TRY(cudaSetDevice(b->ctx->device));
  CUDA_TRY(cudaStreamSynchronize(b->ctx->stream));
  const MJobDev& j = b->store_jobs[f];
  const size_t n = size_t(j.w) * j.h;
  if (out_len < 3 * n) return set_error(JXG_ERR_ARGUMENT, "plane buffer too small");
  const int32_t* planes = static_cast<const int32_t*>(b->ctx->d_planes_a.p);
  CUDA_TRY(cudaMemcpy(out, planes + j.a, n * 4, cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemcpy(out + n, planes + j.b, n * 4, cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemcpy(out + 2 * n, planes + j.c, n * 4, cudaMemcpyDeviceToHost));
  return JXG_OK;
}

// ms[0] = whole batch on the device, ms[1] = the group-stream decode kernel (+ local RCTs) alone.
int jxg_modular_batch_stats(void* bp, uint64_t* h2d, uint64_t* d2h, uint64_t* launches, float* ms) {
  ModularBatch* b = static_cast<ModularBatch*>(bp);
  if (!b || !b->uploaded) return JXG_ERR_ARGUMENT;
  CUDA_TRY(cudaSetDevice(b->ctx->device));
  CUDA_TRY(cudaEventSynchronize(b->ev1));
  if (h2d) *h2d = b->h2d;
  if (d2h) *d2h = b->d2h;
  if (launches) *launches = b->launches;
  if (ms) {
    ms[0] = ms[1] = 0;
    cudaEventElapsedTime(&ms[0], b->ev0, b->ev1);
    cudaEventElapsedTime(&ms[1], b->ev0, b->ev_decode);
    cudaGetLastError();
  }
  return JXG_OK;
}

int jxg_modular_walk_table(const int32_t* nodes, uint32_t n_nodes, const uint8_t* context_map, uint32_t n_contexts,
                           uint32_t channel, uint32_t stream_id, uint32_t* lut_out, uint32_t* property) {
  if (!nodes || !n_nodes || !context_map || !lut_out || !property) return JXG_ERR_ARGUMENT;
  jxg::ModularTree t;
  t.nodes.resize(n_nodes);
  for (uint32_t i = 0; i < n_nodes; i++) {
    jxg::TreeNode& n = t.nodes[i];
    n.property = nodes[i * 5];
    n.val = nodes[i * 5 + 1];
    n.left = uint32_t(nodes[i * 5 + 2]);
    n.right = uint32_t(nodes[i * 5 + 3]);
    n.ctx = uint32_t(nodes[i * 5 + 4]);
    // children must lie behind their parent (no cycles) and inside the array
    if (n.property >= 0 && (n.left <= i || n.right <= i || n.left >= n_nodes || n.right >= n_nodes)) return JXG_ERR_ARGUMENT;
    if (n.property < 0 && n.ctx >= n_contexts) return JXG_ERR_ARGUMENT;
  }
  t.code.context_map.assign(context_map, context_map + n_contexts);
  std::vector<uint32_t> lut;
  uint32_t prop = kLutNoProperty, single = 0;
  const uint32_t root = static_root(t, channel, stream_id);
  if (!build_walk_table(t, root, channel, stream_id, lut, prop, single)) return 0;
  *property = prop;
  for (int i = 0; i < kLutSize; i++) lut_out[i] = prop == kLutNoProperty ? single : lut[size_t(i)];
  return 1;
}

void jxg_modular_batch_end(void* bp) {
  ModularBatch* b = static_cast<ModularBatch*>(bp);
  if (!b) return;
  cudaSetDevice(b->ctx->device);
  cudaStreamSynchronize(b->ctx->stream);
  for (cudaEvent_t e : {b->ev0, b->ev1, b->ev_decode})
    if (e) cudaEventDestroy(e);
  b->ctx->batch_live = false;
  delete b;
}

}  // extern "C"
