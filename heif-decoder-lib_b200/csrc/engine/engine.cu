// engine.cu — device engine behind include/heifcuda.h ("device engine" section): places parsed
// pictures in HBM, launches K1..K5 on a CUDA stream and reads results back.
//
// HBM layout of one batch (all offsets 256-byte aligned):
//   record arena   : [hc_pic[]][hc_ctu[]][hc_blk[]][hc_tb[]][hc_coeff[]][edge_map][qp_map][scaling]
//                    [tb index lists by size][K2 row tasks]        -- ONE pinned->device copy
//   residual buffer: int16, one contiguous nT*nT tile per coded transform block (K1 -> K2)
//   plane pool     : per picture the reconstruction planes (K2 writes, K3 filters in place, K4 reads),
//                    per canvas the final Y/Cb/Cr(/A) planes (K4 writes, K5 reads)
//   rgb buffer     : interleaved output of K5, rows padded to 256 bytes, or the packed planes K8 writes (HC_OUT_YCBCR)
// Device blocks come from a per-engine free list so that the plugin's one-decoder-per-tile call
// pattern (context.cc:1799-1835) does not pay a cudaMalloc per tile.
#include <cuda_runtime.h>
#include <algorithm>
#include <atomic>
#include <thread>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>
#include "../capi/capi_internal.h"
#include "../kernels/launch.h"
#include "../host/k0_host.h"

namespace {

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

bool cuda_ok(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return true;
  hc::set_last_error(std::string(what) + ": " + cudaGetErrorString(e));
  return false;
}

struct Block {
  void* p = nullptr;
  size_t cap = 0;
};

}  // namespace

struct hc_engine {
  int device = 0;
  std::mutex mu;
  std::vector<Block> free_dev, free_pin;
  std::vector<Block> free_out_pin;   // pinned output buffers of hc_heic_decode_stream (gigabytes each: pinning one takes a second)
  std::vector<cudaStream_t> free_streams;      // batch streams (highest priority: K1..K5, copies)
  std::vector<cudaStream_t> free_k0_streams;   // K0 streams (lowest priority), see hc_batch_reconstruct_async
  int prio_lo = 0, prio_hi = 0;
  std::vector<cudaEvent_t> free_events;     // events are recycled: a batch needs 14 and the plugin creates one batch per tile
  hc::k0::Tables* d_k0_tables = nullptr;   // read-only tables of the device parser
  int device_parse = 1;                    // hc_heic_job: let K0 parse every picture it accepts
  int sm_count = 148;
  int k0_max_critical = 160;               // hc_heic_job: pictures whose parse critical path exceeds this many CTBs stay with the host parser
  int premultiply_alpha = 0;               // hc_heic_job: RGBA output multiplied by alpha in K5
  int chroma_upsampling = 0;               // HC_UPSAMPLE_*: colour conversion of hc_heic_job / hc_heic_decode_stream
  int stream_depth = 0;                    // hc_heic_decode_stream: batches in flight; 0 = automatic (3 or 6 by the measured read-back time), 2..6 fixed
  int stream_depth_learned = 0;            // what the last automatic call ended with: the next call starts there
  cudaEvent_t origin = nullptr;            // HEIFCUDA_TRACE: time zero of hc_batch_timeline_ms
  int host_share_pct = -1;                 // hc_heic_job with device_parse: percentage of the coded items the host threads parse meanwhile
  int scale_max_side = 0;                  // hc_heic_job / stream: images larger than this on their longer side are delivered scaled (0: off)

  Block take(std::vector<Block>& list, size_t size, bool pinned) {
    std::lock_guard<std::mutex> lk(mu);
    int best = -1;
    for (int i = 0; i < (int)list.size(); i++)
      if (list[i].cap >= size && (best < 0 || list[i].cap < list[best].cap)) best = i;
    if (best >= 0) {
      Block b = list[best];
      list.erase(list.begin() + best);
      return b;
    }
    Block b;
    size_t cap = align_up(size + size / 4, 1 << 20);
    cudaError_t e = pinned ? cudaMallocHost(&b.p, cap) : cudaMalloc(&b.p, cap);
    if (e != cudaSuccess) {
      // try the exact size before giving up
      cap = align_up(size, 4096);
      e = pinned ? cudaMallocHost(&b.p, cap) : cudaMalloc(&b.p, cap);
    }
    if (e != cudaSuccess) {
      cuda_ok(e, pinned ? "cudaMallocHost" : "cudaMalloc");
      b.p = nullptr;
      cap = 0;
    }
    b.cap = cap;
    return b;
  }
  cudaEvent_t take_event() {
    {
      std::lock_guard<std::mutex> lk(mu);
      if (!free_events.empty()) { cudaEvent_t ev = free_events.back(); free_events.pop_back(); return ev; }
    }
    cudaEvent_t ev = nullptr;
    if (cudaEventCreate(&ev) != cudaSuccess) return nullptr;
    return ev;
  }
  void give_event(cudaEvent_t ev) {
    if (!ev) return;
    std::lock_guard<std::mutex> lk(mu);
    free_events.push_back(ev);
  }
  void give(std::vector<Block>& list, Block b) {
    if (!b.p) return;
    std::lock_guard<std::mutex> lk(mu);
    list.push_back(b);
  }
};

namespace {

// Y, Cb, Cr and alpha planes in the plane pool; w == 0: no such plane
struct Planes {
  size_t off[4] = {0, 0, 0, 0};     // byte offsets in the plane pool
  int stride[4] = {0, 0, 0, 0};     // samples
  int w[4] = {0, 0, 0, 0}, h[4] = {0, 0, 0, 0};
  // plane k at the end of the pool: rows of at least w + 4 samples of ps bytes padded to 128 bytes, the plane 256-byte aligned
  void place(int k, int pw, int ph, int ps, size_t& pool) {
    w[k] = pw; h[k] = ph;
    stride[k] = (int)(align_up((size_t)(pw + 4) * ps, 128) / ps);
    off[k] = pool;
    pool += align_up((size_t)stride[k] * ph * ps, 256);
  }
};

struct Canvas {
  int w = 0, h = 0, chroma = 1, bit_depth = 8;
  bool alpha = false;
  Planes planes;                    // K4 writes them
  // geometric passes between K4 and K5 (irot / imir / clap of the reference, in the order they are given); the output
  // view below is what K5 and the read-backs use; without passes it is the canvas itself
  struct Pass {
    int kind;                        // 0: dihedral map (a = swap, b = flip_x, c = flip_y), 1: crop (a..d = left, top, right, bottom)
    int a, b, c, d;
    // filled at upload: the image size after the pass and the planes this pass writes
    int w = 0, h = 0;
    Planes planes;
  };
  std::vector<Pass> passes;
  bool transformed() const { return !passes.empty(); }
  int ow = 0, oh = 0;               // output image size
  // delivered image size (hc_batch_set_canvas_output_size; 0 = not set): K5 / K7 sample the output view by nearest neighbour.
  // dw x dh is what the conversion writes and the read-backs copy; filled at upload (ow x oh when no size is set).
  int req_w = 0, req_h = 0;
  int dw = 0, dh = 0;
  bool scaled() const { return dw != ow || dh != oh; }
  Planes view;                      // output view: the planes of the last pass, or the canvas' own (filled at upload)
  // 'iovl' derived image (hc_batch_add_overlay_canvas): no planes of its own; K7 composes the child canvases into its RGB output
  bool overlay = false;
  int bkg[3] = {0, 0, 0};
  struct OverlayChild { int canvas, dx, dy; hc_csc_params p; };
  std::vector<OverlayChild> children;
  // K5 writes here instead of the batch's RGB buffer when set (hc_batch_set_rgb_target: a band of a shared image on this or
  // on a peer GPU)
  uint8_t* ext_rgb = nullptr;
  size_t ext_stride = 0;
  // rgb output of the last convert
  size_t rgb_off = 0;
  size_t rgb_stride = 0;
  int rgb_bpp = 0;
  bool converted = false;
  // the last convert was to HC_OUT_YCBCR: K8 packed the output view at rgb_off (poff: plane offsets, packed: total bytes;
  // rgb_bpp: bytes per sample, rgb_stride: the Y row)
  bool planar = false;
  size_t poff[4] = {0, 0, 0, 0};
  size_t packed = 0;
};

struct Placement {
  const hc::PictureRecords* rec;     // host-parsed picture, or
  int canvas, x, y, role, rescale;
  const hc::K0HostPicture* k0 = nullptr;   // picture whose slice data K0 parses on the device
};

}  // namespace

struct hc_batch {
  hc_engine* eng = nullptr;
  cudaStream_t stream = nullptr;
  cudaStream_t k0_stream = nullptr;   // taken on the first K0 launch
  cudaEvent_t ev_fork = nullptr;
  std::vector<Canvas> canvases;
  std::vector<std::pair<int, int>> alpha_links;   // (canvas, alpha canvas): hc_batch_link_alpha
  std::vector<Placement> pics;
  std::vector<hc_pic> hpics;  // host copy with bases / placement filled
  Block d_arena, h_arena, d_resid, d_planes, d_rgb, d_progress;
  size_t arena_bytes = 0, resid_elems = 0, planes_bytes = 0, rgb_bytes = 0;
  hc::BatchView view{};
  const uint32_t* d_tb_index[4] = {nullptr, nullptr, nullptr, nullptr};
  int tb_counts[4] = {0, 0, 0, 0};
  const hc::RowTask* d_tasks = nullptr;
  const hc::WarpWork* d_work = nullptr;   // K2 task lists: 3 per CTA
  int k2_ctas = 0;
  int ntasks = 0;
  int k2_smem = 0;   // dynamic shared memory per K2 CTA
  // K0 (device CABAC parse) of the pictures added as bitstreams
  int nk0 = 0, nchains = 0;
  bool k0_done = false;
  const hc::k0::Pic* d_k0_pics = nullptr;
  const hc::k0::Sub* d_k0_subs = nullptr;
  const hc::k0::Chain* d_k0_chains = nullptr;
  size_t k0_zero_off = 0, k0_zero_bytes = 0;      // device-only zone: cleared to 0 before K0 (edge maps, progress, errors, counters)
  size_t k0_ones_off = 0, k0_ones_bytes = 0;      // cleared to 1 (intra mode maps: DC)
  size_t k0_ctu_off = 0, k0_ctu_bytes = 0;         // CTU records of the K0 pictures (cleared to 0 before K0)
  size_t k0_status_off = 0;                        // [int error per K0 picture][4 list counters]
  const uint32_t* d_k0_tb_index[4] = {nullptr, nullptr, nullptr, nullptr};
  int k0_tb_counts[4] = {0, 0, 0, 0};
  long long k0_list_cap[4] = {0, 0, 0, 0};
  long long k0_max_ctbs = 0;
  bool k0_status_pending = false;                  // K0 ran; its status words were copied to h_status but not looked at yet
  std::vector<int> k0_pic_of;                      // K0 picture -> batch picture index
  Block h_status;
  cudaEvent_t ev_k0[2] = {};
  cudaEvent_t ev_d2h[2] = {};
  size_t k0_input_bytes = 0;
  long long max_dbk_units = 0, max_sao_quads = 0;
  int max_planes = 1;
  bool uploaded = false;
  cudaEvent_t ev[8] = {};
  cudaEvent_t timer[2] = {};
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> csc_events;
  int launches = 0;
  float last_d2h_ms = 0.f;
  std::vector<int> failed_pics;   // pictures whose device parse failed (k0_check_status)
  int pack_threads = 0;     // host threads hc_batch_upload may use to pack the pinned arena (0: hardware concurrency)
};

namespace {

using hc::plane_w;
using hc::plane_h;

// bytes of a canvas' block in the batch's output buffer for interleaved rows of bpp bytes per pixel
size_t interleaved_block_bytes(const Canvas& c, int bpp) {
  return align_up(align_up((size_t)((c.dw + 7) & ~7) * bpp, 256) * c.dh, 256);
}

// HC_OUT_YCBCR: lays the canvas' output view out as hc_image_plane_layout does for its desc. False when the planes differ in
// size from that layout: HeifPixelImage::crop scales a crop window to each plane by integer division, so a window at an odd
// position can leave a chroma plane one sample larger than (w + 1) / 2.
bool planar_layout(const Canvas& c, size_t poff[4], size_t* packed) {
  hc_image_desc d{};
  d.width = c.ow; d.height = c.oh; d.chroma_format = c.chroma; d.bit_depth = c.bit_depth; d.has_alpha = c.alpha;
  d.out_format = HC_OUT_YCBCR;
  int32_t w[4], h[4];
  *packed = hc_image_plane_layout(&d, poff, nullptr, w, h);
  for (int k = 0; k < 4; k++)
    if (w[k] != c.view.w[k] || (w[k] && h[k] != c.view.h[k])) return false;
  return *packed > 0;
}

// the planes of one canvas into a K8 launch (flushing it first when they do not fit)
void add_pack_planes(hc_batch* b, hc::PackBatch& pb, const Canvas& c, const uint8_t* P, uint8_t* out) {
  if (pb.n + 4 > hc::PACK_BATCH_MAX) {
    hc::launch_k8_batch(pb, b->stream);
    b->launches += 1;
    pb.n = 0;
  }
  const int ps = c.bit_depth == 8 ? 1 : 2;
  for (int k = 0; k < 4; k++) {
    if (c.view.w[k] == 0) continue;
    hc::PackPlane& q = pb.p[pb.n++];
    q.src = P + c.view.off[k];
    q.dst = out + c.poff[k];
    q.src_pitch = (unsigned)c.view.stride[k] * ps;
    q.row_bytes = (unsigned)c.view.w[k] * ps;
    q.rows = (unsigned)c.view.h[k];
    q.pad = 0;
  }
}

const int kBppOf[6] = {3, 4, 6, 8, 6, 8};   // bytes per pixel of the interleaved HC_OUT_* formats

// Can `p` convert canvas `c`? Changes nothing, so that a call over several canvases leaves them all as they were when one fails.
int check_convert(const Canvas& c, const hc_csc_params& p) {
  if (p.out_format < 0 || p.out_format > HC_OUT_YCBCR) { hc::set_last_error("bad output format"); return HC_ERR_ARGUMENT; }
  if (!c.overlay && p.in_depth != c.bit_depth) { hc::set_last_error("conversion parameters were selected for another bit depth"); return HC_ERR_ARGUMENT; }
  if (p.out_format != HC_OUT_YCBCR) {
    if (c.ext_rgb && c.ext_stride < (size_t)((c.dw + 7) & ~7) * kBppOf[p.out_format]) { hc::set_last_error("external RGB target: rows too short for this format"); return HC_ERR_ARGUMENT; }
    return HC_OK;
  }
  if (c.overlay) { hc::set_last_error("overlay canvases are composed in RGB: HC_OUT_YCBCR is not available for them"); return HC_ERR_UNSUPPORTED; }
  if (c.ext_rgb) { hc::set_last_error("a canvas with an external RGB target cannot be converted to HC_OUT_YCBCR"); return HC_ERR_UNSUPPORTED; }
  if (c.scaled()) { hc::set_last_error("a scaled canvas cannot be converted to HC_OUT_YCBCR"); return HC_ERR_UNSUPPORTED; }
  size_t poff[4], packed = 0;
  if (!planar_layout(c, poff, &packed)) { hc::set_last_error("HC_OUT_YCBCR: the crop window leaves chroma planes of another size than the packed layout"); return HC_ERR_UNSUPPORTED; }
  return HC_OK;
}

// the output format of the canvas' next convert (after check_convert): interleaved rows, or the packed planes of K8
void apply_format(Canvas& c, const hc_csc_params& p) {
  c.planar = p.out_format == HC_OUT_YCBCR;
  if (c.planar) {
    planar_layout(c, c.poff, &c.packed);
    c.rgb_bpp = c.bit_depth == 8 ? 1 : 2;
    c.rgb_stride = (size_t)c.ow * c.rgb_bpp;
  } else {
    c.rgb_bpp = kBppOf[p.out_format];
    c.rgb_stride = align_up((size_t)((c.dw + 7) & ~7) * c.rgb_bpp, 256);
  }
}

// Where every canvas' output lies after a convert of canvases[0..n) with params[0..n) (after check_convert), decided without
// changing anything: one block per canvas in canvas order, in the new format for the canvases the call names and as it is for
// the others (8 bytes per pixel for a canvas never converted). A converted canvas the call does not name keeps its offset and
// its bytes, so the call fails when the layout would move one, or would make the buffer grow while one exists.
int plan_output(const hc_batch* b, int n, const int* canvases, const hc_csc_params* params, std::vector<size_t>& off, size_t& total) {
  std::vector<const hc_csc_params*> named(b->canvases.size(), nullptr);
  for (int i = 0; i < n; i++) named[canvases[i]] = &params[i];
  off.resize(b->canvases.size());
  total = 0;
  bool kept = false;
  for (size_t k = 0; k < b->canvases.size(); k++) {
    const Canvas& c = b->canvases[k];
    const hc_csc_params* p = named[k];
    if (!p && c.converted) {
      if (c.rgb_off != total) {
        hc::set_last_error("convert: the output of a converted canvas the call does not name would move; convert it in the same call");
        return HC_ERR_ARGUMENT;
      }
      kept = true;
    }
    off[k] = total;
    const bool planar = p ? p->out_format == HC_OUT_YCBCR : c.planar;
    size_t poff[4], packed = c.packed;
    if (p && planar) planar_layout(c, poff, &packed);
    total += planar ? align_up(packed, 256) : interleaved_block_bytes(c, p ? kBppOf[p->out_format] : (c.rgb_bpp ? c.rgb_bpp : 8));
  }
  if (kept && total > b->d_rgb.cap) {
    hc::set_last_error("convert: the output buffer would have to grow under a converted canvas the call does not name; convert it in the same call");
    return HC_ERR_ARGUMENT;
  }
  return HC_OK;
}

// K5's arguments for canvas c: its output view into its block of the output buffer, or into its external target
hc::CscArgs csc_args(const hc_batch* b, const Canvas& c, const hc_csc_params& p) {
  const uint8_t* P = (const uint8_t*)b->d_planes.p;
  hc::CscArgs a;
  a.y = P + c.view.off[0];
  a.cb = c.chroma ? P + c.view.off[1] : nullptr;
  a.cr = c.chroma ? P + c.view.off[2] : nullptr;
  a.a = c.alpha ? P + c.view.off[3] : nullptr;
  a.y_stride = c.view.stride[0]; a.c_stride = c.view.stride[1]; a.a_stride = c.view.stride[3];
  a.width = c.dw; a.height = c.dh; a.chroma_format = c.chroma;
  a.src_w = c.ow; a.src_h = c.oh; a.gather = c.scaled();
  a.out = c.ext_rgb ? c.ext_rgb : (uint8_t*)b->d_rgb.p + c.rgb_off;
  a.out_stride = (long long)(c.ext_rgb ? c.ext_stride : c.rgb_stride);
  a.p = p;
  return a;
}

// Enqueues the copy of a converted canvas' output to dst: the packed planes in one 1-D copy (HC_OUT_YCBCR: dst_stride must be
// the Y row), else dh rows of dw interleaved pixels. `timed`: between the events ev_d2h.
int enqueue_output_copy(hc_batch* b, const char* fn, int canvas, void* dst, size_t dst_stride, cudaMemcpyKind kind, bool timed) {
  if (!b || !dst || canvas < 0 || canvas >= (int)b->canvases.size()) { hc::set_last_error(std::string(fn) + ": bad argument"); return HC_ERR_ARGUMENT; }
  const Canvas& c = b->canvases[canvas];
  if (!c.converted) { hc::set_last_error("canvas was not converted"); return HC_ERR_ARGUMENT; }
  if (c.ext_rgb) { hc::set_last_error("this image is written to an external RGB target (hc_batch_set_rgb_target): read it there"); return HC_ERR_ARGUMENT; }
  if (c.planar && dst_stride != c.rgb_stride) { hc::set_last_error("HC_OUT_YCBCR: the packed planes are read with the stride of the Y row"); return HC_ERR_ARGUMENT; }
  const uint8_t* src = (const uint8_t*)b->d_rgb.p + c.rgb_off;
  if (timed) cudaEventRecord(b->ev_d2h[0], b->stream);
  const cudaError_t e = c.planar ? cudaMemcpyAsync(dst, src, c.packed, kind, b->stream)
                                 : cudaMemcpy2DAsync(dst, dst_stride, src, c.rgb_stride, (size_t)c.dw * c.rgb_bpp, c.dh, kind, b->stream);
  if (timed) cudaEventRecord(b->ev_d2h[1], b->stream);
  return cuda_ok(e, c.planar ? "cudaMemcpyAsync(packed planes)" : "cudaMemcpy2DAsync(rgb)") ? HC_OK : HC_ERR_CUDA;
}

// plane k of a canvas' output view, which the plane read-backs copy
int check_view_plane(const Canvas& c, int k) {
  if (c.view.w[k] != 0) return HC_OK;
  hc::set_last_error("canvas has no such plane");
  return HC_ERR_ARGUMENT;
}

void release_blocks(hc_batch* b) {
  hc_engine* e = b->eng;
  e->give(e->free_dev, b->d_arena);
  e->give(e->free_pin, b->h_arena);
  e->give(e->free_dev, b->d_resid);
  e->give(e->free_dev, b->d_planes);
  e->give(e->free_dev, b->d_rgb);
  e->give(e->free_dev, b->d_progress);
  e->give(e->free_pin, b->h_status);
  b->d_arena = b->h_arena = b->d_resid = b->d_planes = b->d_rgb = b->d_progress = b->h_status = Block();
}

}  // namespace

extern "C" {

int hc_has_cuda_engine(void) { return 1; }

hc_engine* hc_engine_create(int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    hc::set_last_error(std::string("no CUDA device available (") + (e != cudaSuccess ? cudaGetErrorString(e) : "0 devices") +
                       "); this engine has no CPU fallback");
    return nullptr;
  }
  if (device < 0 || device >= n) {
    hc::set_last_error("hc_engine_create: device ordinal out of range");
    return nullptr;
  }
  if (!cuda_ok(cudaSetDevice(device), "cudaSetDevice")) return nullptr;
  hc_engine* eng = new (std::nothrow) hc_engine;
  if (!eng) return nullptr;
  eng->device = device;
  cudaDeviceGetAttribute(&eng->sm_count, cudaDevAttrMultiProcessorCount, device);
  cudaDeviceGetStreamPriorityRange(&eng->prio_lo, &eng->prio_hi);   // (least, greatest): greatest is numerically lowest
  if (const char* m = getenv("HEIFCUDA_PARSER")) eng->device_parse = strcmp(m, "host") != 0;
  if (const char* m = getenv("HEIFCUDA_HOST_SHARE")) eng->host_share_pct = std::max(-1, std::min(100, atoi(m)));
  if (!cuda_ok(cudaMalloc(&eng->d_k0_tables, sizeof(hc::k0::Tables)), "cudaMalloc(K0 tables)") ||
      !cuda_ok(cudaMemcpy(eng->d_k0_tables, &hc::k0_tables(), sizeof(hc::k0::Tables), cudaMemcpyHostToDevice), "cudaMemcpy(K0 tables)")) {
    delete eng;
    return nullptr;
  }
  return eng;
}

void hc_engine_destroy(hc_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  for (auto& b : e->free_dev) cudaFree(b.p);
  for (auto& b : e->free_pin) cudaFreeHost(b.p);
  for (auto& b : e->free_out_pin) cudaFreeHost(b.p);
  for (auto s : e->free_streams) cudaStreamDestroy(s);
  for (auto s : e->free_k0_streams) cudaStreamDestroy(s);
  for (auto ev : e->free_events) cudaEventDestroy(ev);
  if (e->d_k0_tables) cudaFree(e->d_k0_tables);
  delete e;
}

int hc_engine_set_option(hc_engine* e, const char* name, int value) {
  if (!e || !name) return HC_ERR_ARGUMENT;
  if (!strcmp(name, "device_parse")) { e->device_parse = value; return HC_OK; }
  if (!strcmp(name, "k0_max_critical_ctbs")) { e->k0_max_critical = value < 1 ? 1 : value; return HC_OK; }
  if (!strcmp(name, "stream_depth")) { e->stream_depth = value <= 0 ? 0 : (value < 2 ? 2 : (value > 6 ? 6 : value)); return HC_OK; }
  if (!strcmp(name, "stream_depth_learned")) { e->stream_depth_learned = value; return HC_OK; }
  if (!strcmp(name, "host_share_pct")) { e->host_share_pct = value < 0 ? -1 : (value > 100 ? 100 : value); return HC_OK; }
  if (!strcmp(name, "premultiply_alpha")) { e->premultiply_alpha = value != 0; return HC_OK; }
  if (!strcmp(name, "scale_max_side")) {
    if (value < 0) { hc::set_last_error("scale_max_side: 0 (off) or the longest side in pixels"); return HC_ERR_ARGUMENT; }
    e->scale_max_side = value;
    return HC_OK;
  }
  if (!strcmp(name, "chroma_upsampling")) {
    if (value != HC_UPSAMPLE_NEAREST && value != HC_UPSAMPLE_BILINEAR) { hc::set_last_error("chroma_upsampling: HC_UPSAMPLE_NEAREST or HC_UPSAMPLE_BILINEAR"); return HC_ERR_ARGUMENT; }
    e->chroma_upsampling = value;
    return HC_OK;
  }
  hc::set_last_error(std::string("unknown engine option ") + name);
  return HC_ERR_ARGUMENT;
}
int hc_engine_get_option(const hc_engine* e, const char* name) {
  if (!e || !name) return 0;
  if (!strcmp(name, "device_parse")) return e->device_parse;
  if (!strcmp(name, "stream_depth")) return e->stream_depth;
  if (!strcmp(name, "stream_depth_learned")) return e->stream_depth_learned;
  if (!strcmp(name, "host_share_pct")) return e->host_share_pct;
  if (!strcmp(name, "chroma_upsampling")) return e->chroma_upsampling;
  if (!strcmp(name, "premultiply_alpha")) return e->premultiply_alpha;
  if (!strcmp(name, "scale_max_side")) return e->scale_max_side;
  if (!strcmp(name, "k0_max_critical_ctbs")) return e->k0_max_critical;
  return 0;
}

hc_batch* hc_batch_create(hc_engine* e) {
  if (!e) { hc::set_last_error("hc_batch_create: null engine"); return nullptr; }
  if (!cuda_ok(cudaSetDevice(e->device), "cudaSetDevice")) return nullptr;
  hc_batch* b = new (std::nothrow) hc_batch;
  if (!b) return nullptr;
  b->eng = e;
  {
    std::lock_guard<std::mutex> lk(e->mu);
    if (!e->free_streams.empty()) { b->stream = e->free_streams.back(); e->free_streams.pop_back(); }
  }
  if (!b->stream && !cuda_ok(cudaStreamCreateWithPriority(&b->stream, cudaStreamNonBlocking, e->prio_hi), "cudaStreamCreate")) {
    delete b;
    return nullptr;
  }
  bool ok = true;
  for (auto& ev : b->ev) ok &= (ev = e->take_event()) != nullptr;
  for (auto& ev : b->timer) ok &= (ev = e->take_event()) != nullptr;
  for (auto& ev : b->ev_k0) ok &= (ev = e->take_event()) != nullptr;
  ok &= (b->ev_fork = e->take_event()) != nullptr;
  for (auto& ev : b->ev_d2h) ok &= (ev = e->take_event()) != nullptr;
  if (!ok) { hc::set_last_error("cudaEventCreate failed"); hc_batch_destroy(b); return nullptr; }
  return b;
}

void hc_batch_destroy(hc_batch* b) {
  if (!b) return;
  cudaSetDevice(b->eng->device);
  cudaStreamSynchronize(b->stream);
  if (b->k0_stream) cudaStreamSynchronize(b->k0_stream);
  release_blocks(b);
  for (auto& ev : b->ev) b->eng->give_event(ev);
  for (auto& ev : b->timer) b->eng->give_event(ev);
  for (auto& ev : b->ev_k0) b->eng->give_event(ev);
  b->eng->give_event(b->ev_fork);
  for (auto& ev : b->ev_d2h) b->eng->give_event(ev);
  for (auto& p : b->csc_events) { b->eng->give_event(p.first); b->eng->give_event(p.second); }
  {
    std::lock_guard<std::mutex> lk(b->eng->mu);
    b->eng->free_streams.push_back(b->stream);
    if (b->k0_stream) b->eng->free_k0_streams.push_back(b->k0_stream);
  }
  delete b;
}

int hc_batch_add_canvas(hc_batch* b, int width, int height, int chroma_format, int bit_depth, int with_alpha) {
  if (!b || width <= 0 || height <= 0 || chroma_format < 0 || chroma_format > 3 || bit_depth < 8 || bit_depth > 16) {
    hc::set_last_error("hc_batch_add_canvas: bad argument");
    return HC_ERR_ARGUMENT;
  }
  Canvas c;
  c.w = width; c.h = height; c.chroma = chroma_format; c.bit_depth = bit_depth; c.alpha = with_alpha != 0;
  b->canvases.push_back(c);
  return (int)b->canvases.size() - 1;
}

int hc_batch_set_canvas_transform(hc_batch* b, int canvas, int swap, int flip_x, int flip_y) {
  if (!b || canvas < 0 || canvas >= (int)b->canvases.size()) { hc::set_last_error("hc_batch_set_canvas_transform: bad argument"); return HC_ERR_ARGUMENT; }
  Canvas& c = b->canvases[canvas];
  c.passes.clear();
  b->uploaded = false;
  if (swap || flip_x || flip_y) return hc_batch_add_canvas_pass(b, canvas, HC_PASS_DIHEDRAL, swap != 0, flip_x != 0, flip_y != 0, 0);
  return HC_OK;
}

int hc_batch_add_canvas_pass(hc_batch* b, int canvas, int kind, int a0, int a1, int a2, int a3) {
  if (!b || canvas < 0 || canvas >= (int)b->canvases.size() || (kind != HC_PASS_DIHEDRAL && kind != HC_PASS_CROP)) {
    hc::set_last_error("hc_batch_add_canvas_pass: bad argument");
    return HC_ERR_ARGUMENT;
  }
  Canvas& c = b->canvases[canvas];
  if (kind == HC_PASS_CROP && (a0 < 0 || a1 < 0 || a2 < a0 || a3 < a1)) { hc::set_last_error("hc_batch_add_canvas_pass: bad crop window"); return HC_ERR_ARGUMENT; }
  Canvas::Pass p;
  p.kind = kind; p.a = a0; p.b = a1; p.c = a2; p.d = a3;
  c.passes.push_back(p);
  b->uploaded = false;
  return HC_OK;
}

int hc_batch_set_canvas_output_size(hc_batch* b, int canvas, int width, int height) {
  if (!b || canvas < 0 || canvas >= (int)b->canvases.size() || width < 1 || height < 1) {
    hc::set_last_error("hc_batch_set_canvas_output_size: bad argument");
    return HC_ERR_ARGUMENT;
  }
  Canvas& c = b->canvases[canvas];
  if (c.ext_rgb) { hc::set_last_error("hc_batch_set_canvas_output_size: the canvas has an external RGB target"); return HC_ERR_UNSUPPORTED; }
  c.req_w = width; c.req_h = height;
  b->uploaded = false;
  return HC_OK;
}

int hc_batch_link_alpha(hc_batch* b, int canvas, int alpha_canvas) {
  if (!b || canvas < 0 || canvas >= (int)b->canvases.size() || alpha_canvas < 0 || alpha_canvas >= (int)b->canvases.size() || canvas == alpha_canvas) {
    hc::set_last_error("hc_batch_link_alpha: bad argument");
    return HC_ERR_ARGUMENT;
  }
  const Canvas& c = b->canvases[canvas];
  const Canvas& a = b->canvases[alpha_canvas];
  if (!c.alpha) { hc::set_last_error("canvas has no alpha plane"); return HC_ERR_ARGUMENT; }
  if ((a.bit_depth == 8) != (c.bit_depth == 8)) { hc::set_last_error("alpha image sample size differs from the colour image"); return HC_ERR_UNSUPPORTED; }
  b->alpha_links.push_back({canvas, alpha_canvas});
  b->uploaded = false;
  return HC_OK;
}

static int add_picture(hc_batch* b, const hc::PictureRecords* rec, const hc::K0HostPicture* k0, int canvas, int x, int y, int role,
                       int rescale_limited) {
  if (!b || (!rec && !k0) || canvas < 0 || canvas >= (int)b->canvases.size() || x < 0 || y < 0) {
    hc::set_last_error("hc_batch_add_picture: bad argument");
    return HC_ERR_ARGUMENT;
  }
  const Canvas& c = b->canvases[canvas];
  const hc_pic& p = rec ? rec->pic : k0->hpic;
  if (b->pics.size() >= 65535) { hc::set_last_error("too many pictures in one batch"); return HC_ERR_ARGUMENT; }
  if (role == HC_ROLE_COLOUR) {
    if (p.chroma_format != c.chroma) { hc::set_last_error("picture has a different chroma format than its canvas"); return HC_ERR_BITSTREAM; }
    if (p.bit_depth_y != c.bit_depth || (p.chroma_format && p.bit_depth_c != c.bit_depth)) {
      hc::set_last_error("picture has a different bit depth than its canvas");
      return HC_ERR_BITSTREAM;
    }
  } else if (role == HC_ROLE_LUMA) {
    if (c.chroma != 0 || c.alpha) { hc::set_last_error("a luma-only picture needs a monochrome canvas"); return HC_ERR_ARGUMENT; }
    if (p.bit_depth_y != c.bit_depth) { hc::set_last_error("picture has a different bit depth than its canvas"); return HC_ERR_BITSTREAM; }
  } else if (role == HC_ROLE_ALPHA) {
    if (!c.alpha) { hc::set_last_error("canvas has no alpha plane"); return HC_ERR_ARGUMENT; }
    if ((p.bit_depth_y == 8) != (c.bit_depth == 8)) { hc::set_last_error("alpha image sample size differs from the colour image"); return HC_ERR_UNSUPPORTED; }
  } else {
    hc::set_last_error("hc_batch_add_picture: unknown role");
    return HC_ERR_ARGUMENT;
  }
  if (x >= c.w || y >= c.h) { hc::set_last_error("picture placed outside its canvas"); return HC_ERR_BITSTREAM; }
  b->pics.push_back({rec, canvas, x, y, role, rescale_limited, k0});
  b->uploaded = false;
  return (int)b->pics.size() - 1;
}

int hc_batch_add_picture(hc_batch* b, const hc_records* rec, int canvas, int x, int y, int role, int rescale_limited) {
  return add_picture(b, rec ? rec->rec.get() : nullptr, nullptr, canvas, x, y, role, rescale_limited);
}

int hc_batch_add_k0_picture(hc_batch* b, const hc_k0_picture* k, int canvas, int x, int y, int role, int rescale_limited) {
  if (k && !k->hp.eligible) { hc::set_last_error("picture is not eligible for the device parser: " + k->hp.why_not); return HC_ERR_UNSUPPORTED; }
  return add_picture(b, nullptr, k ? &k->hp : nullptr, canvas, x, y, role, rescale_limited);
}

int hc_batch_upload(hc_batch* b) {
  if (!b) return HC_ERR_ARGUMENT;
  if (!cuda_ok(cudaSetDevice(b->eng->device), "cudaSetDevice")) return HC_ERR_CUDA;
  const int np = (int)b->pics.size();
  if (np == 0) { hc::set_last_error("hc_batch_upload: empty batch"); return HC_ERR_ARGUMENT; }

  // ---- plane pool layout ----
  size_t pool = 0;
  b->hpics.resize(np);
  for (auto& c : b->canvases) {
    const int ps = c.bit_depth == 8 ? 1 : 2;
    c.planes = Planes();
    for (int k = 0; k < (c.alpha ? 4 : 3); k++)
      if (!c.overlay && plane_w(c.w, c.chroma, k)) c.planes.place(k, plane_w(c.w, c.chroma, k), plane_h(c.h, c.chroma, k), ps, pool);
    c.converted = false;
    // pass outputs: every pass writes its own set of planes (passes are rare; the chain stays simple and exact)
    int iw = c.w, ih = c.h;
    const Planes* in = &c.planes;
    for (Canvas::Pass& pass : c.passes) {
      int nw, nh;
      if (pass.kind == HC_PASS_DIHEDRAL) { nw = pass.a ? ih : iw; nh = pass.a ? iw : ih; }
      else {
        if (pass.c >= iw || pass.d >= ih) { hc::set_last_error("crop window outside the image"); return HC_ERR_ARGUMENT; }
        nw = pass.c - pass.a + 1; nh = pass.d - pass.b + 1;
      }
      pass.planes = Planes();
      for (int k = 0; k < 4; k++) {
        const int w = in->w[k], h = in->h[k];
        if (w == 0) continue;
        if (pass.kind == HC_PASS_DIHEDRAL) pass.planes.place(k, pass.a ? h : w, pass.a ? w : h, ps, pool);
        else {
          // HeifPixelImage::crop (pixelimage.cc:820-823): the window is scaled to every plane by integer division
          const int pl = pass.a * w / iw, pr = pass.c * w / iw, pt = pass.b * h / ih, pb = pass.d * h / ih;
          pass.planes.place(k, pr - pl + 1, pb - pt + 1, ps, pool);
        }
      }
      pass.w = iw = nw; pass.h = ih = nh;
      in = &pass.planes;
    }
    c.ow = iw; c.oh = ih;
    c.dw = c.req_w ? c.req_w : iw; c.dh = c.req_h ? c.req_h : ih;
    c.view = c.passes.empty() ? c.planes : c.passes.back().planes;
  }
  // ---- record bases ----
  size_t n_ctu = 0, n_blk = 0, n_tb = 0, n_coeff = 0, n_edge = 0, n_qp = 0, n_scal = 0;
  uint64_t n_resid = 0;
  int counts[4] = {0, 0, 0, 0};
  std::vector<int> idx_base((size_t)np * 4);   // first slot of picture i in the size-l launch list
  int max_rows = 0;
  size_t n_tasks = 0;
  b->max_dbk_units = b->max_sao_quads = 0;
  b->max_planes = 1;
  b->nk0 = 0;
  b->k0_pic_of.clear();
  for (int i = 0; i < np; i++) {
    hc_pic& p = b->hpics[i];
    if (const hc::K0HostPicture* k = b->pics[i].k0) {
      // device-parsed picture: its record regions live in the device-only zone behind the uploaded arena (bases below)
      p = k->hpic;
      const uint64_t nctb = (uint64_t)k->pic.ctbs_w * k->pic.ctbs_h;
      p.scaling_base = (uint32_t)n_scal; n_scal += k->scaling.size();
      p.resid_count = nctb * k->pic.resid_cap_ctb;
      p.resid_base = n_resid;         n_resid += align_up(p.resid_count, 8);
      b->k0_pic_of.push_back(i);
      b->k0_max_ctbs = b->nk0 ? std::max<long long>(b->k0_max_ctbs, (long long)nctb) : (long long)nctb;
      b->nk0++;
    } else {
      const hc::PictureRecords& r = *b->pics[i].rec;
      p = r.pic;
      p.ctu_base = (uint32_t)n_ctu;   n_ctu += r.ctus.size();
      p.blk_base = (uint32_t)n_blk;   n_blk += r.blks.size();
      p.tb_base = (uint32_t)n_tb;     n_tb += r.tbs.size();
      p.coeff_base = (uint32_t)n_coeff; n_coeff += r.coeffs.size();
      p.edge_base = (uint32_t)n_edge; n_edge += r.edge_map.size();
      p.qp_base = (uint32_t)n_qp;     n_qp += r.qp_map.size();
      p.scaling_base = (uint32_t)n_scal; n_scal += r.scaling.size();
      p.resid_base = n_resid;         n_resid += align_up(r.resid_count, 8);
      if (n_blk > 0xFFFFFFFFull || n_coeff > 0xFFFFFFFFull) { hc::set_last_error("batch too large"); return HC_ERR_ARGUMENT; }
      for (int l = 0; l < 4; l++) { idx_base[(size_t)i * 4 + l] = counts[l]; counts[l] += (int)r.tbs_by_size[l]; }
    }
    const int ncomp = p.chroma_format ? 3 : 1;
    max_rows = std::max(max_rows, (int)p.ctbs_h);
    n_tasks += (size_t)ncomp * p.ctbs_h;
    b->max_planes = std::max(b->max_planes, ncomp);
    b->max_dbk_units = std::max(b->max_dbk_units, (long long)(p.width >> 3) * (p.height >> 2));
    b->max_sao_quads = std::max(b->max_sao_quads, (long long)p.ctbs_w * p.ctbs_h);   // CTBs: K4 runs one warp per CTB
    // reconstruction planes
    const int ps = (p.bit_depth_y == 8 && p.bit_depth_c == 8) ? 1 : 2;
    const int SubW = (p.chroma_format == 1 || p.chroma_format == 2) ? 2 : 1, SubH = p.chroma_format == 1 ? 2 : 1;
    for (int c = 0; c < ncomp; c++) {
      const int w = c ? p.width / SubW : p.width, h = c ? p.height / SubH : p.height;
      p.rec_stride[c] = (uint32_t)(align_up((size_t)w * ps, 128) / ps);
      p.rec_off[c] = pool;
      pool += align_up((size_t)p.rec_stride[c] * h * ps, 256);
    }
    // destination
    const Canvas& cv = b->canvases[b->pics[i].canvas];
    p.dst_x = b->pics[i].x; p.dst_y = b->pics[i].y; p.dst_w = cv.w; p.dst_h = cv.h;
    p.dst_flags = 0;
    if (b->pics[i].rescale) p.dst_flags |= HC_DST_RESCALE_LIMITED;
    if (b->pics[i].role == HC_ROLE_ALPHA) {
      p.dst_off[0] = cv.planes.off[3]; p.dst_stride[0] = (uint32_t)cv.planes.stride[3];
      p.dst_flags |= HC_DST_SKIP_CB | HC_DST_SKIP_CR;
    } else if (b->pics[i].role == HC_ROLE_LUMA) {
      p.dst_off[0] = cv.planes.off[0]; p.dst_stride[0] = (uint32_t)cv.planes.stride[0];
      p.dst_flags |= HC_DST_SKIP_CB | HC_DST_SKIP_CR;
    } else {
      for (int c = 0; c < ncomp; c++) { p.dst_off[c] = cv.planes.off[c]; p.dst_stride[c] = (uint32_t)cv.planes.stride[c]; }
    }
  }

  // ---- arena layout ----
  size_t o = 0;
  auto place = [&](size_t bytes) { size_t at = o; o += align_up(bytes ? bytes : 1, 256); return at; };
  const size_t o_pics = place(sizeof(hc_pic) * np), o_ctus = place(sizeof(hc_ctu) * n_ctu), o_blks = place(sizeof(hc_blk) * n_blk);
  const size_t o_tbs = place(sizeof(hc_tb) * n_tb), o_coeffs = place(sizeof(hc_coeff) * n_coeff);
  const size_t o_edge = place(n_edge), o_qp = place(n_qp), o_scal = place(n_scal);
  size_t o_idx[4];
  for (int l = 0; l < 4; l++) o_idx[l] = place(sizeof(uint32_t) * counts[l]);
  const size_t o_tasks = place(sizeof(hc::RowTask) * n_tasks);
  const size_t o_work = place(sizeof(hc::WarpWork) * 3 * n_tasks);   // K2 task lists: at most one CTA per task
  // K0 inputs (uploaded): picture descriptors, slices, per-CTB tables, substreams, chains, RBSP bytes
  const int nk0 = b->nk0;
  size_t k_slices = 0, k_ctbs = 0, k_subs = 0, k_chains = 0, k_bytes = 0;
  for (int q = 0; q < nk0; q++) {
    const hc::K0HostPicture& k = *b->pics[b->k0_pic_of[q]].k0;
    k_slices += k.slices.size(); k_ctbs += k.ctb_slice.size(); k_subs += k.subs.size(); k_chains += k.chains.size();
    k_bytes += align_up(k.bytes.size(), 16);
  }
  const size_t o_kpics = place(sizeof(hc::k0::Pic) * nk0), o_kslices = place(sizeof(hc::k0::Slice) * k_slices);
  const size_t o_kctbslice = place(4 * k_ctbs), o_kstatic = place(4 * k_ctbs), o_ksubs = place(sizeof(hc::k0::Sub) * k_subs);
  const size_t o_kchains = place(sizeof(hc::k0::Chain) * k_chains), o_kbytes = place(k_bytes + 64);
  b->arena_bytes = o;
  b->k0_input_bytes = nk0 ? o - o_kpics : 0;
  b->nchains = (int)k_chains;

  // device-only zone behind the uploaded arena: the fixed-capacity record regions K0 fills, its scratch maps,
  // status words and K1 launch lists. Laid out by category so that each clear is one memset.
  size_t z = align_up(o, 256);
  auto zplace = [&](size_t bytes, size_t align) { z = align_up(z, align); size_t at = z; z += bytes; return at; };
  struct K0Off { size_t ctus, blks, tbs, coeffs, edge, qp, ct_depth, ipm, ipm_c, wpp, progress; };
  std::vector<K0Off> koff(nk0);
  size_t z_lists[4] = {0, 0, 0, 0}, list_cap[4] = {0, 0, 0, 0};
  if (nk0) {
    for (int q = 0; q < nk0; q++) {   // ctu regions must sit at a multiple of sizeof(hc_ctu) from the ctu array base
      const hc::k0::Pic& kp = b->pics[b->k0_pic_of[q]].k0->pic;
      z = o_ctus + align_up(z - o_ctus, sizeof(hc_ctu));
      koff[q].ctus = z; z += sizeof(hc_ctu) * (size_t)kp.ctbs_w * kp.ctbs_h;
    }
    // the CTU records of all K0 pictures form one contiguous run; it is cleared before K0 so that a CTB a failing chain
    // never reached has no blocks and no SAO (K2..K4 run on the batch without waiting for K0's verdict)
    b->k0_ctu_off = koff[0].ctus;
    b->k0_ctu_bytes = z - koff[0].ctus;
    // the byte-addressed maps first: their bases are 32-bit BYTE offsets from the uploaded arrays (hc_pic::edge_base / qp_base),
    // so they must not sit behind the record regions (13 GB for 96 twelve-megapixel files); the record bases are element
    // indices and reach 16 GB (coefficients) / 64 GB (blocks, transform blocks)
    for (int q = 0; q < nk0; q++) { const hc::k0::Pic& kp = b->pics[b->k0_pic_of[q]].k0->pic; koff[q].qp = zplace((size_t)kp.w8 * kp.h8, 1); }
    for (int q = 0; q < nk0; q++) { const hc::k0::Pic& kp = b->pics[b->k0_pic_of[q]].k0->pic; koff[q].ct_depth = zplace((size_t)kp.w8 * kp.h8, 1); }
    for (int q = 0; q < nk0; q++) { const hc::k0::Pic& kp = b->pics[b->k0_pic_of[q]].k0->pic; koff[q].wpp = zplace((size_t)kp.ctbs_h * hc::k0::CTX_BYTES, 16); }
    // cleared to 1: intra prediction mode maps (DC)
    b->k0_ones_off = zplace(0, 256);
    for (int q = 0; q < nk0; q++) { const hc::k0::Pic& kp = b->pics[b->k0_pic_of[q]].k0->pic; koff[q].ipm = zplace((size_t)kp.w4 * kp.h4, 1); koff[q].ipm_c = zplace((size_t)kp.w4 * kp.h4, 1); }
    b->k0_ones_bytes = z - b->k0_ones_off;
    // cleared to 0: edge maps, row progress, status
    b->k0_zero_off = zplace(0, 256);
    for (int q = 0; q < nk0; q++) { const hc::k0::Pic& kp = b->pics[b->k0_pic_of[q]].k0->pic; koff[q].edge = zplace((size_t)kp.w4 * kp.h4, 1); }
    for (int q = 0; q < nk0; q++) { const hc::k0::Pic& kp = b->pics[b->k0_pic_of[q]].k0->pic; koff[q].progress = zplace(4 * (size_t)kp.ctbs_h, 4); }
    b->k0_status_off = zplace(4 * ((size_t)nk0 + 4), 16);
    b->k0_zero_bytes = z - b->k0_zero_off;
    for (int q = 0; q < nk0; q++) { const hc::k0::Pic& kp = b->pics[b->k0_pic_of[q]].k0->pic; koff[q].blks = zplace(sizeof(hc_blk) * (size_t)kp.ctbs_w * kp.ctbs_h * kp.blk_cap_ctb, 16); }
    for (int q = 0; q < nk0; q++) { const hc::k0::Pic& kp = b->pics[b->k0_pic_of[q]].k0->pic; koff[q].tbs = zplace(sizeof(hc_tb) * (size_t)kp.ctbs_w * kp.ctbs_h * kp.tb_cap_ctb, 16); }
    for (int q = 0; q < nk0; q++) { const hc::k0::Pic& kp = b->pics[b->k0_pic_of[q]].k0->pic; koff[q].coeffs = zplace(sizeof(hc_coeff) * (size_t)kp.ctbs_w * kp.ctbs_h * kp.coeff_cap_ctb, 16); }
    for (int l = 0; l < 4; l++) {
      for (int q = 0; q < nk0; q++) { const hc::k0::Pic& kp = b->pics[b->k0_pic_of[q]].k0->pic; list_cap[l] += ((size_t)kp.ctbs_w * kp.ctbs_h * kp.tb_cap_ctb >> (2 * l)) + 64; }
      z_lists[l] = zplace(4 * list_cap[l], 16);
    }
  }
  const size_t arena_total = align_up(z, 256);

  release_blocks(b);
  b->h_arena = b->eng->take(b->eng->free_pin, o, true);
  b->d_arena = b->eng->take(b->eng->free_dev, arena_total, false);
  if (nk0) b->h_status = b->eng->take(b->eng->free_pin, 4 * ((size_t)nk0 + 4), true);
  b->d_resid = b->eng->take(b->eng->free_dev, std::max<size_t>(n_resid * 2, 256), false);
  b->d_planes = b->eng->take(b->eng->free_dev, std::max<size_t>(pool, 256), false);
  b->d_progress = b->eng->take(b->eng->free_dev, std::max<size_t>(n_tasks * sizeof(int), 256), false);
  if (!b->h_arena.p || !b->d_arena.p || !b->d_resid.p || !b->d_planes.p || !b->d_progress.p) return HC_ERR_MEMORY;
  b->resid_elems = n_resid;
  b->planes_bytes = pool;

  if (nk0 && !b->h_status.p) return HC_ERR_MEMORY;
  uint8_t* H = (uint8_t*)b->h_arena.p;
  uint8_t* Dk = (uint8_t*)b->d_arena.p;
  // the RBSP bytes of the device-parsed pictures (the bulk of such a batch's upload) are copied by the packing threads below
  struct K0Copy { uint8_t* dst; const uint8_t* src; size_t n; };
  std::vector<K0Copy> k0_copies;
  // ---- K0 pictures: record bases (element offsets from the uploaded array bases into the device-only zone) + inputs ----
  if (nk0) {
    hc::k0::Pic* kp_out = (hc::k0::Pic*)(H + o_kpics);
    hc::k0::Slice* ks_out = (hc::k0::Slice*)(H + o_kslices);
    int32_t* kc_out = (int32_t*)(H + o_kctbslice);
    uint8_t* kst_out = H + o_kstatic;
    hc::k0::Sub* ksub_out = (hc::k0::Sub*)(H + o_ksubs);
    size_t is = 0, ic = 0, isub = 0, ib = 0;
    struct ChainKey { int row; uint64_t bytes; hc::k0::Chain chain; };   // row of the first substream, slice data bytes
    std::vector<ChainKey> chains;
    for (int q = 0; q < nk0; q++) {
      const int i = b->k0_pic_of[q];
      const hc::K0HostPicture& k = *b->pics[i].k0;
      hc_pic& p = b->hpics[i];
      p.ctu_base = (uint32_t)((koff[q].ctus - o_ctus) / sizeof(hc_ctu));
      p.blk_base = (uint32_t)((koff[q].blks - o_blks) / sizeof(hc_blk));
      p.tb_base = (uint32_t)((koff[q].tbs - o_tbs) / sizeof(hc_tb));
      p.coeff_base = (uint32_t)((koff[q].coeffs - o_coeffs) / sizeof(hc_coeff));
      p.edge_base = (uint32_t)(koff[q].edge - o_edge);
      p.qp_base = (uint32_t)(koff[q].qp - o_qp);
      if ((koff[q].blks - o_blks) / sizeof(hc_blk) > 0xFFFFFFFFull || (koff[q].coeffs - o_coeffs) / sizeof(hc_coeff) > 0xFFFFFFFFull ||
          koff[q].edge - o_edge > 0xFFFFFFFFull) { hc::set_last_error("batch too large for the device parser"); return HC_ERR_ARGUMENT; }
      hc::k0::Pic kp = k.pic;
      kp.pic_index = (uint32_t)i;
      kp.tb_global_base = p.tb_base;
      kp.bytes = Dk + o_kbytes + ib;
      kp.slices = (const hc::k0::Slice*)(Dk + o_kslices) + is;
      kp.ctb_slice = (const int32_t*)(Dk + o_kctbslice) + ic;
      kp.ctu_static = Dk + o_kstatic + 4 * ic;
      kp.ct_depth = Dk + koff[q].ct_depth; kp.ipm = Dk + koff[q].ipm; kp.ipm_c = Dk + koff[q].ipm_c; kp.wpp_ctx = Dk + koff[q].wpp;
      kp.progress = (int*)(Dk + koff[q].progress);
      kp.error = (int*)(Dk + b->k0_status_off) + q;
      kp.qp_map = (int8_t*)(Dk + koff[q].qp); kp.edge_map = Dk + koff[q].edge;
      kp.ctus = (hc_ctu*)(Dk + koff[q].ctus); kp.blks = (hc_blk*)(Dk + koff[q].blks); kp.tbs = (hc_tb*)(Dk + koff[q].tbs);
      kp.coeffs = (hc_coeff*)(Dk + koff[q].coeffs);
      for (int l = 0; l < 4; l++) kp.tb_lists[l] = (uint32_t*)(Dk + z_lists[l]);
      kp.tb_counts = (unsigned int*)(Dk + b->k0_status_off) + nk0;
      kp_out[q] = kp;
      memcpy(ks_out + is, k.slices.data(), sizeof(hc::k0::Slice) * k.slices.size());
      memcpy(kc_out + ic, k.ctb_slice.data(), 4 * k.ctb_slice.size());
      memcpy(kst_out + 4 * ic, k.ctu_static.data(), k.ctu_static.size());
      k0_copies.push_back({H + o_kbytes + ib, k.bytes.data(), k.bytes.size()});
      for (size_t t = 0; t < k.subs.size(); t++) { ksub_out[isub + t] = k.subs[t]; ksub_out[isub + t].pic = (uint32_t)q; }
      for (const hc::k0::Chain& c : k.chains) {
        // a substream ends at the next one's entry point or at the end of its slice segment's data
        uint64_t bytes = 0;
        for (uint32_t t = c.first_sub; t < c.first_sub + c.nsubs; t++) {
          const hc::k0::Sub& sub = k.subs[t];
          const bool entry_next = t + 1 < k.subs.size() && k.subs[t + 1].slice == sub.slice;
          const uint32_t end = entry_next ? k.subs[t + 1].byte_begin : k.slices[sub.slice].data_end;
          bytes += end > sub.byte_begin ? end - sub.byte_begin : 0;
        }
        chains.push_back({k.subs[c.first_sub].first_ctb / k.pic.ctbs_w, bytes, {(uint32_t)(isub + c.first_sub), c.nsubs}});
      }
      is += k.slices.size(); ic += k.ctb_slice.size(); isub += k.subs.size(); ib += align_up(k.bytes.size(), 16);
    }
    memset(H + o_kbytes + ib, 0, 64);
    // rows of all pictures interleaved: a chain only ever waits for a chain with a smaller index. Within a row the chain
    // with the most slice data comes first: the four chains of a K0 CTA, which holds its slot until the slowest one
    // ends, then take about the same time, and the longest chains do not start last. The key (row, -bytes, position) is
    // total, so the order is deterministic.
    std::stable_sort(chains.begin(), chains.end(), [](const ChainKey& a, const ChainKey& c) { return a.row != c.row ? a.row < c.row : a.bytes > c.bytes; });
    hc::k0::Chain* kch_out = (hc::k0::Chain*)(H + o_kchains);
    for (size_t t = 0; t < chains.size(); t++) kch_out[t] = chains[t].chain;
    b->d_k0_pics = (const hc::k0::Pic*)(Dk + o_kpics);
    b->d_k0_subs = (const hc::k0::Sub*)(Dk + o_ksubs);
    b->d_k0_chains = (const hc::k0::Chain*)(Dk + o_kchains);
    for (int l = 0; l < 4; l++) { b->d_k0_tb_index[l] = (const uint32_t*)(Dk + z_lists[l]); b->k0_list_cap[l] = (long long)list_cap[l]; }
  }
  b->k0_done = false;
  b->k0_status_pending = false;

  // ---- pack: every picture's records go to disjoint slices of the pinned arena, in parallel ----
  memcpy(H + o_pics, b->hpics.data(), sizeof(hc_pic) * np);
  uint32_t* idx[4];
  for (int l = 0; l < 4; l++) idx[l] = (uint32_t*)(H + o_idx[l]);
  auto pack_picture = [&](int i) {
    const hc_pic& p = b->hpics[i];
    if (const hc::K0HostPicture* k = b->pics[i].k0) {
      if (!k->scaling.empty()) memcpy(H + o_scal + p.scaling_base, k->scaling.data(), k->scaling.size());
      return;
    }
    const hc::PictureRecords& r = *b->pics[i].rec;
    memcpy(H + o_ctus + sizeof(hc_ctu) * p.ctu_base, r.ctus.data(), sizeof(hc_ctu) * r.ctus.size());
    memcpy(H + o_blks + sizeof(hc_blk) * p.blk_base, r.blks.data(), sizeof(hc_blk) * r.blks.size());
    hc_tb* tb = (hc_tb*)(H + o_tbs) + p.tb_base;
    int fill[4];
    for (int l = 0; l < 4; l++) fill[l] = idx_base[(size_t)i * 4 + l];
    for (size_t k = 0; k < r.tbs.size(); k++) {
      tb[k] = r.tbs[k];
      tb[k].pic = (uint16_t)i;
      const int l = tb[k].log2 - 2;
      idx[l][fill[l]++] = (uint32_t)(p.tb_base + k);
    }
    memcpy(H + o_coeffs + sizeof(hc_coeff) * p.coeff_base, r.coeffs.data(), sizeof(hc_coeff) * r.coeffs.size());
    memcpy(H + o_edge + p.edge_base, r.edge_map.data(), r.edge_map.size());
    memcpy(H + o_qp + p.qp_base, r.qp_map.data(), r.qp_map.size());
    if (!r.scaling.empty()) memcpy(H + o_scal + p.scaling_base, r.scaling.data(), r.scaling.size());
  };
  {
    // `pack_threads` comes from the job (its host thread count): several ranks share one box, and a rank that took every
    // hardware thread for a few milliseconds of memcpy made all of them slower
    int nthreads = b->pack_threads > 0 ? b->pack_threads : (int)std::thread::hardware_concurrency();
    const int nwork = np + (int)k0_copies.size();
    nthreads = std::max(1, std::min(nthreads, std::min(nwork, (int)(o >> 22) + 1)));   // ~4 MB per thread at least
    auto work = [&](int i) {
      if (i < np) pack_picture(i);
      else { const K0Copy& c = k0_copies[i - np]; memcpy(c.dst, c.src, c.n); }
    };
    if (nthreads == 1) {
      for (int i = 0; i < nwork; i++) work(i);
    } else {
      std::atomic<int> next{0};
      std::vector<std::thread> pool;
      for (int t = 0; t < nthreads; t++)
        pool.emplace_back([&]() { for (int i; (i = next.fetch_add(1)) < nwork;) work(i); });
      for (auto& t : pool) t.join();
    }
  }
  // K2 tasks: row-major across all pictures so that every wavefront advances together and a task
  // only depends on a task with a smaller index
  {
    hc::RowTask* tasks = (hc::RowTask*)(H + o_tasks);
    std::vector<int> first_of_row((size_t)np * 3, -1), prev((size_t)np * 3, -1);
    int t = 0;
    for (int row = 0; row < max_rows; row++)
      for (int i = 0; i < np; i++) {
        const hc_pic& p = b->hpics[i];
        if (row >= p.ctbs_h) continue;
        const int ncomp = p.chroma_format ? 3 : 1;
        for (int c = 0; c < ncomp; c++) {
          hc::RowTask& k = tasks[t];
          k.pic = (uint32_t)i; k.row = (uint16_t)row; k.comp = (uint8_t)c; k.pad = 0;
          k.dep = prev[(size_t)i * 3 + c];
          prev[(size_t)i * 3 + c] = t;
          t++;
        }
      }
    b->ntasks = t;
    // Per-warp task lists of the K2 CTAs (kernels/k2_intra.cu: k2_intra_lists_kernel) and each task's slice of its CTA's
    // shared memory. A CTA is three warps: a luma-class row (luma, or chroma that is not subsampled) takes a warp of its
    // own, subsampled chroma rows share the third warp up to four units (4:2:0 row = 1, 4:2:2 row = 2; a 4:2:0 chroma row
    // takes about a quarter of a luma row), so that all warps of a CTA run for about the same time. The chroma rows of a
    // CTA run one after the other and share one region of shared memory.
    hc::WarpWork* work = (hc::WarpWork*)(H + o_work);
    auto task_bytes = [&](int idx, int& units) {
      const hc_pic& p = b->hpics[tasks[idx].pic];
      const int ps = (p.bit_depth_y == 8 && p.bit_depth_c == 8) ? 1 : 2;
      const int c = tasks[idx].comp;
      const int sw = (c && (p.chroma_format == 1 || p.chroma_format == 2)) ? 1 : 0, sh = (c && p.chroma_format == 1) ? 1 : 0;
      units = (sw + sh == 2) ? 1 : (sw + sh == 1 ? 2 : 0);   // 0: luma class
      return hc::k2_task_smem_bytes((1 << p.log2_ctb) >> sw, (1 << p.log2_ctb) >> sh, ps);
    };
    int ncta = 0;
    b->k2_smem = 0;
    int luma[2], nl = 0, chroma[4], nc = 0, cunits = 0;
    auto flush = [&]() {
      if (nl == 0 && nc == 0) return;
      hc::WarpWork* w = work + 3 * (size_t)ncta;
      memset(w, 0, 3 * sizeof(hc::WarpWork));
      int off = 0, u;
      for (int k = 0; k < nl; k++) { w[k].task[0] = (uint32_t)luma[k]; w[k].n = 1; tasks[luma[k]].smem_off = (uint32_t)off; off += task_bytes(luma[k], u); }
      int cmax = 0;
      for (int k = 0; k < nc; k++) { w[2].task[k] = (uint32_t)chroma[k]; tasks[chroma[k]].smem_off = (uint32_t)off; cmax = std::max(cmax, task_bytes(chroma[k], u)); }
      w[2].n = (uint32_t)nc;
      b->k2_smem = std::max(b->k2_smem, off + cmax);
      ncta++;
      nl = nc = cunits = 0;
    };
    for (int idx = 0; idx < t; idx++) {
      int units;
      task_bytes(idx, units);
      if (units == 0) {
        if (nl == 2) flush();
        luma[nl++] = idx;
      } else {
        if (cunits + units > 4 || nc == 4) flush();
        chroma[nc++] = idx;
        cunits += units;
      }
    }
    flush();
    b->k2_ctas = ncta;
  }

  // ---- device view ----
  uint8_t* D = (uint8_t*)b->d_arena.p;
  b->view.pics = (const hc_pic*)(D + o_pics);
  b->view.ctus = (const hc_ctu*)(D + o_ctus);
  b->view.blks = (const hc_blk*)(D + o_blks);
  b->view.tbs = (const hc_tb*)(D + o_tbs);
  b->view.coeffs = (const hc_coeff*)(D + o_coeffs);
  b->view.edge_map = D + o_edge;
  b->view.qp_map = (const int8_t*)(D + o_qp);
  b->view.scaling = D + o_scal;
  b->view.resid = (int16_t*)b->d_resid.p;
  b->view.planes = (uint8_t*)b->d_planes.p;
  b->view.npics = np;
  for (int l = 0; l < 4; l++) { b->d_tb_index[l] = (const uint32_t*)(D + o_idx[l]); b->tb_counts[l] = counts[l]; }
  b->d_tasks = (const hc::RowTask*)(D + o_tasks);
  b->d_work = (const hc::WarpWork*)(D + o_work);

  cudaEventRecord(b->ev[0], b->stream);
  if (!cuda_ok(cudaMemcpyAsync(D, H, o, cudaMemcpyHostToDevice, b->stream), "cudaMemcpyAsync(H2D records)")) return HC_ERR_CUDA;
  cudaEventRecord(b->ev[1], b->stream);
  b->uploaded = true;
  return HC_OK;
}

// Looks at the status words K0 left in pinned memory. The stream must have been synchronised.
static int k0_check_status(hc_batch* b) {
  if (!b->k0_status_pending) return HC_OK;
  b->k0_status_pending = false;
  const int* status = (const int*)b->h_status.p;
  for (int l = 0; l < 4; l++) { b->k0_tb_counts[l] = status[b->nk0 + l]; b->launches += b->k0_tb_counts[l] > 0; }
  // every failing picture is remembered (hc_batch_failed_pictures: the stream API isolates the files they belong to — a
  // failing chain never touches another picture's regions); the first one names the error
  b->failed_pics.clear();
  for (int q = 0; q < b->nk0; q++)
    if (status[q]) {
      if (b->failed_pics.empty())
        hc::set_last_error("picture " + std::to_string(b->k0_pic_of[q]) + (status[q] == hc::k0::ERR_CAPACITY ? ": device parser capacity exceeded"
                                                                                                             : ": malformed slice data (device parser)"));
      b->failed_pics.push_back(b->k0_pic_of[q]);
    }
  return b->failed_pics.empty() ? HC_OK : HC_ERR_BITSTREAM;
}

// Synchronises the stream and reports a K0 parse error of the batch, if any.
static int batch_sync_checked(hc_batch* b, const char* what) {
  if (!cuda_ok(cudaStreamSynchronize(b->stream), what)) return HC_ERR_CUDA;
  return k0_check_status(b);
}

// Enqueues K0 (first run only) and K1..K4 without waiting for anything: the K1 launch lists K0 builds are consumed
// through their device-side counters. A K0 parse error surfaces at the next synchronising call.
int hc_batch_reconstruct_async(hc_batch* b, int stages) {
  if (!b || !b->uploaded) { hc::set_last_error("hc_batch_reconstruct: batch not uploaded"); return HC_ERR_ARGUMENT; }
  if (!cuda_ok(cudaSetDevice(b->eng->device), "cudaSetDevice")) return HC_ERR_CUDA;
  cudaStream_t s = b->stream;
  b->launches = 0;
  for (auto& p : b->csc_events) { b->eng->give_event(p.first); b->eng->give_event(p.second); }
  b->csc_events.clear();
  cudaMemsetAsync(b->d_progress.p, 0, std::max<size_t>((size_t)b->ntasks * sizeof(int), 4), s);
  uint8_t* D = (uint8_t*)b->d_arena.p;
  if (b->nk0 && !b->k0_done) {
    // K0: the slice data of the pictures added as bitstreams is parsed on the device, straight into their record
    // regions; afterwards the records stay resident (a second hc_batch_reconstruct re-uses them)
    // K0 runs on a stream of the LOWEST priority, K1..K5 and the copies on the batch stream (highest): K0's chains live for
    // tens of milliseconds and fill the register file, so when the K0 kernels of consecutive batches overlap (the tail of
    // one wavefront leaves most chain slots idle, the next batch's chains take them) the short streaming kernels of the
    // finished batch get every CTA slot that frees up first instead of queueing behind the next parse.
    if (!b->k0_stream) {
      {
        std::lock_guard<std::mutex> lk(b->eng->mu);
        if (!b->eng->free_k0_streams.empty()) { b->k0_stream = b->eng->free_k0_streams.back(); b->eng->free_k0_streams.pop_back(); }
      }
      if (!b->k0_stream && !cuda_ok(cudaStreamCreateWithPriority(&b->k0_stream, cudaStreamNonBlocking, b->eng->prio_lo), "cudaStreamCreate(K0)"))
        return HC_ERR_CUDA;
    }
    cudaStream_t ks = b->k0_stream;
    cudaEventRecord(b->ev_fork, s);          // upload + progress reset
    cudaStreamWaitEvent(ks, b->ev_fork, 0);
    cudaEventRecord(b->ev_k0[0], ks);
    cudaMemsetAsync(D + b->k0_ones_off, 1, b->k0_ones_bytes, ks);
    cudaMemsetAsync(D + b->k0_zero_off, 0, b->k0_zero_bytes, ks);
    cudaMemsetAsync(D + b->k0_ctu_off, 0, b->k0_ctu_bytes, ks);
    hc::launch_k0(b->eng->d_k0_tables, b->d_k0_pics, b->d_k0_subs, b->d_k0_chains, b->nchains, ks);
    hc::launch_k0_finish(b->d_k0_pics, b->nk0, (int)b->k0_max_ctbs, ks);
    cudaEventRecord(b->ev_k0[1], ks);
    cudaStreamWaitEvent(s, b->ev_k0[1], 0);
    const size_t status_bytes = 4 * ((size_t)b->nk0 + 4);
    if (!cuda_ok(cudaMemcpyAsync(b->h_status.p, D + b->k0_status_off, status_bytes, cudaMemcpyDeviceToHost, s), "cudaMemcpyAsync(K0 status)"))
      return HC_ERR_CUDA;
    b->k0_status_pending = true;
    b->k0_done = true;
    b->launches += 2;
  }
  cudaEventRecord(b->ev[2], s);
  hc::launch_k1(b->view, b->d_tb_index, b->tb_counts, s);
  for (int l = 0; l < 4; l++) b->launches += b->tb_counts[l] > 0;
  if (b->nk0 && !b->k0_status_pending)
    for (int l = 0; l < 4; l++) b->launches += b->k0_tb_counts[l] > 0;   // counted by k0_check_status on the first run
  if (b->nk0)
    hc::launch_k1_indirect(b->view, b->d_k0_tb_index, b->k0_list_cap, (const unsigned*)(D + b->k0_status_off) + b->nk0, b->eng->sm_count, s);
  cudaEventRecord(b->ev[3], s);
  hc::launch_k2(b->view, b->d_tasks, b->d_work, b->k2_ctas, b->k2_smem, (int*)b->d_progress.p, s);
  b->launches += 1;
  cudaEventRecord(b->ev[4], s);
  // K4 always runs: it is also the crop + paste pass; SAO parameters are ignored when disabled
  hc::BatchView v = b->view;
  v.flags = (stages & HC_STAGE_SAO) ? 0 : hc::HC_VIEW_NO_SAO;
  if (stages & HC_STAGE_DEBLOCK) {
    hc::launch_k3(b->view, b->max_dbk_units, b->max_planes, s);
    b->launches += 2;
  }
  cudaEventRecord(b->ev[5], s);
  hc::launch_k4(v, b->max_sao_quads, b->max_planes, s);
  b->launches += 1;
  // K6: irot / imir / clap passes of the canvases that carry any, plane by plane (rare; timed with K4)
  for (const Canvas& c : b->canvases) {
    if (!c.transformed()) continue;
    const int ps = c.bit_depth == 8 ? 1 : 2;
    int iw = c.w, ih = c.h;
    const Planes* in = &c.planes;
    for (const Canvas::Pass& p : c.passes) {
      const Planes& out = p.planes;
      for (int k = 0; k < 4; k++) {
        if (out.w[k] == 0) continue;
        const uint8_t* src = (const uint8_t*)b->d_planes.p + in->off[k];
        uint8_t* dst = (uint8_t*)b->d_planes.p + out.off[k];
        if (p.kind == HC_PASS_DIHEDRAL) {
          hc::XformArgs a;
          a.src = src; a.dst = dst;
          a.w = in->w[k]; a.h = in->h[k]; a.src_stride = in->stride[k]; a.dst_stride = out.stride[k];
          a.swap = p.a; a.flip_x = p.b; a.flip_y = p.c;
          hc::launch_k6(a, c.bit_depth != 8, s);
        } else {
          const int pl = p.a * in->w[k] / iw, pt = p.b * in->h[k] / ih;
          cudaMemcpy2DAsync(dst, (size_t)out.stride[k] * ps, src + ((size_t)pt * in->stride[k] + pl) * ps, (size_t)in->stride[k] * ps,
                            (size_t)out.w[k] * ps, out.h[k], cudaMemcpyDeviceToDevice, s);
        }
        b->launches += 1;
      }
      iw = p.w; ih = p.h; in = &out;
    }
  }
  // alpha planes that come from an alpha image of another size (hc_batch_link_alpha): nearest-neighbour rescale of the
  // alpha canvas' output view into the alpha plane of the colour canvas' output view
  for (const auto& l : b->alpha_links) {
    const Canvas& c = b->canvases[l.first];
    const Planes& a = b->canvases[l.second].view;
    hc::launch_k6_scale((const uint8_t*)b->d_planes.p + a.off[0], a.w[0], a.h[0], a.stride[0], (uint8_t*)b->d_planes.p + c.view.off[3],
                        c.view.w[3], c.view.h[3], c.view.stride[3], c.bit_depth != 8, s);
    b->launches += 1;
  }
  cudaEventRecord(b->ev[6], s);
  if (!cuda_ok(cudaGetLastError(), "kernel launch")) return HC_ERR_CUDA;
  return HC_OK;
}

// Same, but a batch with device-parsed pictures waits for K0's verdict, so that malformed slice data is reported here.
int hc_batch_reconstruct(hc_batch* b, int stages) {
  const int rc = hc_batch_reconstruct_async(b, stages);
  if (rc != HC_OK) return rc;
  if (b->k0_status_pending) return batch_sync_checked(b, "K0 (device CABAC parse)");
  return HC_OK;
}

int hc_batch_convert(hc_batch* b, int canvas, const hc_csc_params* params) {
  if (!b || !params || canvas < 0 || canvas >= (int)b->canvases.size()) { hc::set_last_error("hc_batch_convert: bad argument"); return HC_ERR_ARGUMENT; }
  return hc_batch_convert_many(b, 1, &canvas, params);
}

// K5 / K7 / K8 for several canvases with as few launches as possible (K5: one per group of up to CSC_BATCH_MAX canvases of
// the same sample size).
int hc_batch_convert_many(hc_batch* b, int n, const int* canvases, const hc_csc_params* params) {
  if (!b || n <= 0 || !canvases || !params || !b->uploaded) { hc::set_last_error("hc_batch_convert_many: bad argument"); return HC_ERR_ARGUMENT; }
  if (!cuda_ok(cudaSetDevice(b->eng->device), "cudaSetDevice")) return HC_ERR_CUDA;
  for (int i = 0; i < n; i++) {   // every canvas is checked before any of them changes
    if (canvases[i] < 0 || canvases[i] >= (int)b->canvases.size()) { hc::set_last_error("hc_batch_convert_many: bad canvas"); return HC_ERR_ARGUMENT; }
    if (int rc = check_convert(b->canvases[canvases[i]], params[i])) return rc;
  }
  std::vector<size_t> off;
  size_t total = 0;
  if (int rc = plan_output(b, n, canvases, params, off, total)) return rc;
  if (b->d_rgb.cap < total) {   // no converted canvas outside the call (plan_output): nothing in the old buffer is kept
    Block grown = b->eng->take(b->eng->free_dev, total, false);
    if (!grown.p) return HC_ERR_MEMORY;
    b->eng->give(b->eng->free_dev, b->d_rgb);
    b->d_rgb = grown;
  }
  for (size_t k = 0; k < b->canvases.size(); k++) b->canvases[k].rgb_off = off[k];
  for (int i = 0; i < n; i++) apply_format(b->canvases[canvases[i]], params[i]);
  const uint8_t* P = (const uint8_t*)b->d_planes.p;
  cudaEvent_t e0 = b->eng->take_event(), e1 = b->eng->take_event();
  cudaEventRecord(e0, b->stream);
  for (int i = 0; i < n; i++) {          // 'iovl' canvases: K7 composes their children (timed with K5)
    Canvas& c = b->canvases[canvases[i]];
    if (!c.overlay) continue;
    hc::OverlayArgs oa;
    memset(&oa, 0, sizeof(oa));
    oa.n = (int)c.children.size();
    for (int k = 0; k < oa.n; k++) {
      const Canvas& ch = b->canvases[c.children[k].canvas];
      hc::OverlayChild& oc = oa.child[k];
      oc.y = P + ch.view.off[0]; oc.cb = P + ch.view.off[1]; oc.cr = P + ch.view.off[2]; oc.a = ch.alpha ? P + ch.view.off[3] : nullptr;
      oc.y_stride = ch.view.stride[0]; oc.c_stride = ch.view.stride[1]; oc.a_stride = ch.view.stride[3];
      oc.w = ch.ow; oc.h = ch.oh; oc.dx = c.children[k].dx; oc.dy = c.children[k].dy;
      const hc_csc_params& cp = c.children[k].p;
      oc.mode = cp.mode; oc.full_range = cp.full_range;
      oc.r_cr = cp.r_cr; oc.g_cb = cp.g_cb; oc.g_cr = cp.g_cr; oc.b_cb = cp.b_cb;
    }
    oa.width = c.dw; oa.height = c.dh;
    oa.src_w = c.ow; oa.src_h = c.oh;
    for (int k = 0; k < 3; k++) oa.bkg[k] = c.bkg[k];
    oa.out_format = params[i].out_format;
    oa.out = c.ext_rgb ? c.ext_rgb : (uint8_t*)b->d_rgb.p + c.rgb_off;
    oa.out_stride = (long long)(c.ext_rgb ? c.ext_stride : c.rgb_stride);
    hc::launch_k7(oa, b->stream);
    b->launches += 1;
    c.converted = true;
  }
  for (int sixteen = 0; sixteen < 2; sixteen++) {
    hc::CscBatch cb;
    cb.n = 0;
    for (int i = 0; i <= n; i++) {
      if (i < n && !b->canvases[canvases[i]].overlay && !b->canvases[canvases[i]].planar &&
          (b->canvases[canvases[i]].bit_depth != 8) == (sixteen != 0)) {
        Canvas& c = b->canvases[canvases[i]];
        cb.a[cb.n++] = csc_args(b, c, params[i]);
        c.converted = true;
      }
      if (cb.n == hc::CSC_BATCH_MAX || (i == n && cb.n > 0)) {
        hc::launch_k5_batch(cb, sixteen != 0, b->stream);
        b->launches += 1;
        cb.n = 0;
      }
    }
  }
  {   // HC_OUT_YCBCR canvases: K8 packs their planes, any sample size in one launch
    hc::PackBatch pb;
    pb.n = 0;
    for (int i = 0; i < n; i++) {
      Canvas& c = b->canvases[canvases[i]];
      if (!c.planar) continue;
      add_pack_planes(b, pb, c, P, (uint8_t*)b->d_rgb.p + c.rgb_off);
      c.converted = true;
    }
    if (pb.n > 0) {
      hc::launch_k8_batch(pb, b->stream);
      b->launches += 1;
    }
  }
  cudaEventRecord(e1, b->stream);
  b->csc_events.push_back({e0, e1});
  if (!cuda_ok(cudaGetLastError(), "kernel launch (K5 / K8)")) return HC_ERR_CUDA;
  return HC_OK;
}

int hc_batch_sync(hc_batch* b) {
  if (!b) return HC_ERR_ARGUMENT;
  return batch_sync_checked(b, "cudaStreamSynchronize");
}

int hc_batch_read_plane(hc_batch* b, int canvas, int plane, void* dst, size_t dst_stride) {
  if (!b || !dst || canvas < 0 || canvas >= (int)b->canvases.size() || plane < 0 || plane > 3) {
    hc::set_last_error("hc_batch_read_plane: bad argument");
    return HC_ERR_ARGUMENT;
  }
  const Canvas& c = b->canvases[canvas];
  if (int rc = check_view_plane(c, plane)) return rc;
  const int ps = c.bit_depth == 8 ? 1 : 2;
  cudaEvent_t e0 = b->ev_d2h[0], e1 = b->ev_d2h[1];
  cudaEventRecord(e0, b->stream);
  cudaError_t e = cudaMemcpy2DAsync(dst, dst_stride, (const uint8_t*)b->d_planes.p + c.view.off[plane], (size_t)c.view.stride[plane] * ps,
                                    (size_t)c.view.w[plane] * ps, c.view.h[plane], cudaMemcpyDeviceToHost, b->stream);
  cudaEventRecord(e1, b->stream);
  if (!cuda_ok(e, "cudaMemcpy2DAsync(D2H plane)")) return HC_ERR_CUDA;
  if (int rc = batch_sync_checked(b, "cudaStreamSynchronize")) return rc;
  cudaEventElapsedTime(&b->last_d2h_ms, e0, e1);
  return HC_OK;
}

// Planes 0..nplanes-1 of a canvas with ONE synchronisation: device -> pinned staging (async) -> caller's rows.
// The plugin returns its planes in libheif's pageable memory; three separate pageable read-backs cost three
// driver-serialised synchronous copies per tile.
int hc_batch_read_planes(hc_batch* b, int canvas, int nplanes, void* const* dst, const size_t* dst_strides) {
  if (!b || !dst || !dst_strides || canvas < 0 || canvas >= (int)b->canvases.size() || nplanes < 1 || nplanes > 4) {
    hc::set_last_error("hc_batch_read_planes: bad argument");
    return HC_ERR_ARGUMENT;
  }
  const Canvas& c = b->canvases[canvas];
  const Planes& v = c.view;
  const int ps = c.bit_depth == 8 ? 1 : 2;
  size_t off[4] = {0, 0, 0, 0}, total = 0;
  for (int k = 0; k < nplanes; k++) {
    if (!dst[k]) { hc::set_last_error("hc_batch_read_planes: bad argument"); return HC_ERR_ARGUMENT; }
    if (int rc = check_view_plane(c, k)) return rc;
    off[k] = total;
    total += align_up((size_t)v.w[k] * ps * v.h[k], 256);
  }
  Block stage = b->eng->take(b->eng->free_pin, total, true);
  if (!stage.p) return HC_ERR_MEMORY;
  cudaEventRecord(b->ev_d2h[0], b->stream);
  cudaError_t e = cudaSuccess;
  for (int k = 0; k < nplanes && e == cudaSuccess; k++)
    e = cudaMemcpy2DAsync((uint8_t*)stage.p + off[k], (size_t)v.w[k] * ps, (const uint8_t*)b->d_planes.p + v.off[k], (size_t)v.stride[k] * ps,
                          (size_t)v.w[k] * ps, v.h[k], cudaMemcpyDeviceToHost, b->stream);
  cudaEventRecord(b->ev_d2h[1], b->stream);
  int rc = cuda_ok(e, "cudaMemcpy2DAsync(D2H planes)") ? batch_sync_checked(b, "cudaStreamSynchronize") : HC_ERR_CUDA;
  if (rc == HC_OK) {
    for (int k = 0; k < nplanes; k++) {
      const size_t row = (size_t)v.w[k] * ps;
      const uint8_t* src = (const uint8_t*)stage.p + off[k];
      for (int y = 0; y < v.h[k]; y++) memcpy((uint8_t*)dst[k] + (size_t)y * dst_strides[k], src + (size_t)y * row, row);
    }
    cudaEventElapsedTime(&b->last_d2h_ms, b->ev_d2h[0], b->ev_d2h[1]);
  }
  b->eng->give(b->eng->free_pin, stage);
  return rc;
}

int hc_batch_read_rgb(hc_batch* b, int canvas, void* dst, size_t dst_stride) {
  if (int rc = enqueue_output_copy(b, "hc_batch_read_rgb", canvas, dst, dst_stride, cudaMemcpyDeviceToHost, true)) return rc;
  if (int rc = batch_sync_checked(b, "cudaStreamSynchronize")) return rc;
  cudaEventElapsedTime(&b->last_d2h_ms, b->ev_d2h[0], b->ev_d2h[1]);
  return HC_OK;
}

int hc_batch_copy_rgb_device(hc_batch* b, int canvas, void* dst, size_t dst_stride) {
  // cudaMemcpyDefault: `dst` may live on a peer device (unified addressing; a peer copy over NVLink then)
  if (int rc = enqueue_output_copy(b, "hc_batch_copy_rgb_device", canvas, dst, dst_stride, cudaMemcpyDefault, false)) return rc;
  return batch_sync_checked(b, "cudaStreamSynchronize");
}

// internal (heic_job.cc): the stream API's pinned output buffers live as long as the engine — a second call, or a pipeline
// that grows deeper, does not pin gigabytes again (1.3 s per 2.6 GB buffer measured)
extern "C" void* hc_engine_take_out_pinned(hc_engine* e, size_t bytes, size_t* cap) {
  if (!e || !cuda_ok(cudaSetDevice(e->device), "cudaSetDevice")) return nullptr;
  Block b = e->take(e->free_out_pin, bytes, true);
  if (cap) *cap = b.cap;
  return b.p;
}
extern "C" void hc_engine_give_out_pinned(hc_engine* e, void* p, size_t cap) {
  if (!e || !p) return;
  Block b; b.p = p; b.cap = cap;
  e->give(e->free_out_pin, b);
}
// internal (heic_job.cc): brackets the asynchronous read-backs of a batch with events; hc_batch_async_d2h_ms (after a sync)
// says how long the copies took on the device's copy engine, queueing behind other batches' copies included
extern "C" void hc_batch_mark_d2h(hc_batch* b, int which) {
  if (b && (which == 0 || which == 1)) cudaEventRecord(b->ev_d2h[which], b->stream);
}
extern "C" float hc_batch_async_d2h_ms(hc_batch* b) {
  float ms = 0.f;
  if (b && cudaEventElapsedTime(&ms, b->ev_d2h[0], b->ev_d2h[1]) != cudaSuccess) { cudaGetLastError(); ms = 0.f; }
  return ms;
}

int hc_batch_read_rgb_async(hc_batch* b, int canvas, void* dst, size_t dst_stride) {
  return enqueue_output_copy(b, "hc_batch_read_rgb_async", canvas, dst, dst_stride, cudaMemcpyDeviceToHost, false);
}

int hc_batch_add_overlay_canvas(hc_batch* b, int width, int height, const uint16_t background[4]) {
  if (!b || width <= 0 || height <= 0 || !background) { hc::set_last_error("hc_batch_add_overlay_canvas: bad argument"); return HC_ERR_ARGUMENT; }
  Canvas c;
  c.w = c.ow = width; c.h = c.oh = height; c.chroma = 3; c.bit_depth = 8; c.alpha = false;
  c.overlay = true;
  for (int k = 0; k < 3; k++) c.bkg[k] = background[k] >> 8;      // fill_RGB_16bit keeps the high byte (pixelimage.cc:983)
  b->canvases.push_back(c);
  b->uploaded = false;
  return (int)b->canvases.size() - 1;
}

int hc_batch_overlay_add_child(hc_batch* b, int overlay_canvas, int child_canvas, int dx, int dy, const hc_csc_params* child_params) {
  if (!b || !child_params || overlay_canvas < 0 || overlay_canvas >= (int)b->canvases.size() || child_canvas < 0 ||
      child_canvas >= (int)b->canvases.size() || !b->canvases[overlay_canvas].overlay || b->canvases[child_canvas].overlay) {
    hc::set_last_error("hc_batch_overlay_add_child: bad argument");
    return HC_ERR_ARGUMENT;
  }
  Canvas& o = b->canvases[overlay_canvas];
  const Canvas& c = b->canvases[child_canvas];
  // the reference converts every child to planar RGB 4:4:4 before overlaying and only finds a pipeline for 4:4:4 input
  // (context.cc:2650-2654 -> "Unsupported color conversion"); its canvas is 8 bit (context.cc:2629-2631)
  if (c.chroma != 3 || c.bit_depth != 8) { hc::set_last_error("Unsupported color conversion: overlay children must be 8-bit 4:4:4 images"); return HC_ERR_UNSUPPORTED; }
  if (dx < 0 || dy < 0) { hc::set_last_error("overlay children with negative offsets are not supported"); return HC_ERR_UNSUPPORTED; }
  if ((int)o.children.size() >= hc::OVERLAY_MAX) { hc::set_last_error("too many overlay children"); return HC_ERR_UNSUPPORTED; }
  o.children.push_back({child_canvas, dx, dy, *child_params});
  return HC_OK;
}

int hc_batch_set_rgb_target(hc_batch* b, int canvas, void* device_dst, size_t stride_bytes) {
  if (!b || canvas < 0 || canvas >= (int)b->canvases.size() || (device_dst && ((reinterpret_cast<uintptr_t>(device_dst) | stride_bytes) & 15))) {
    hc::set_last_error("hc_batch_set_rgb_target: bad argument (the target and its stride must be 16-byte aligned)");
    return HC_ERR_ARGUMENT;
  }
  Canvas& c = b->canvases[canvas];
  if (c.planar) { hc::set_last_error("hc_batch_set_rgb_target: the canvas is converted to HC_OUT_YCBCR"); return HC_ERR_UNSUPPORTED; }
  if (device_dst && c.req_w) { hc::set_last_error("hc_batch_set_rgb_target: the canvas has an output size of its own"); return HC_ERR_UNSUPPORTED; }
  c.ext_rgb = (uint8_t*)device_dst;
  c.ext_stride = device_dst ? stride_bytes : 0;
  c.converted = false;
  return HC_OK;
}

int hc_batch_read_residual(hc_batch* b, int pic, int16_t* dst, size_t count) {
  if (!b || !dst || pic < 0 || pic >= (int)b->hpics.size()) { hc::set_last_error("hc_batch_read_residual: bad argument"); return HC_ERR_ARGUMENT; }
  const hc_pic& p = b->hpics[pic];
  if (count > p.resid_count) count = p.resid_count;
  if (!cuda_ok(cudaMemcpyAsync(dst, (const int16_t*)b->d_resid.p + p.resid_base, count * 2, cudaMemcpyDeviceToHost, b->stream), "D2H residual"))
    return HC_ERR_CUDA;
  return batch_sync_checked(b, "cudaStreamSynchronize");
}

int hc_batch_stage_ms(hc_batch* b, float ms[8]) {
  if (!b || !ms) return HC_ERR_ARGUMENT;
  if (int rc = batch_sync_checked(b, "cudaStreamSynchronize")) return rc;
  for (int i = 0; i < 8; i++) ms[i] = 0.f;
  cudaEventElapsedTime(&ms[0], b->ev[0], b->ev[1]);
  for (int k = 0; k < 4; k++) cudaEventElapsedTime(&ms[1 + k], b->ev[2 + k], b->ev[3 + k]);
  for (auto& p : b->csc_events) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, p.first, p.second) == cudaSuccess) ms[5] += t;
    b->eng->give_event(p.first); b->eng->give_event(p.second);
  }
  b->csc_events.clear();
  ms[6] = b->last_d2h_ms;
  if (b->nk0 && b->k0_done) cudaEventElapsedTime(&ms[7], b->ev_k0[0], b->ev_k0[1]);
  cudaGetLastError();
  return HC_OK;
}

// internal (heic_job.cc, HEIFCUDA_TRACE): where the batch's device phases lie on the engine's clock — milliseconds since the
// engine's origin event for [0] upload start, [1] K0 start, [2] K0 end, [3] K1 start, [4] K4 end (K5 follows)
extern "C" int hc_batch_timeline_ms(hc_batch* b, float t[5]) {
  if (!b || !t) return HC_ERR_ARGUMENT;
  hc_engine* e = b->eng;
  {
    std::lock_guard<std::mutex> lk(e->mu);
    if (!e->origin) { cudaEventCreate(&e->origin); cudaEventRecord(e->origin, b->stream); cudaEventSynchronize(e->origin); }
  }
  for (int i = 0; i < 5; i++) t[i] = 0.f;
  cudaEventElapsedTime(&t[0], e->origin, b->ev[0]);
  if (b->nk0 && b->k0_done) { cudaEventElapsedTime(&t[1], e->origin, b->ev_k0[0]); cudaEventElapsedTime(&t[2], e->origin, b->ev_k0[1]); }
  cudaEventElapsedTime(&t[3], e->origin, b->ev[2]);
  cudaEventElapsedTime(&t[4], e->origin, b->ev[6]);
  cudaGetLastError();
  return HC_OK;
}

void* hc_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (!cuda_ok(cudaMallocHost(&p, bytes ? bytes : 1), "cudaMallocHost")) return nullptr;
  return p;
}
void hc_host_free(void* p) { if (p) cudaFreeHost(p); }

int hc_batch_timer_start(hc_batch* b) {
  if (!b) return HC_ERR_ARGUMENT;
  return cuda_ok(cudaEventRecord(b->timer[0], b->stream), "cudaEventRecord") ? HC_OK : HC_ERR_CUDA;
}
int hc_batch_timer_stop_ms(hc_batch* b, float* ms) {
  if (!b || !ms) return HC_ERR_ARGUMENT;
  if (!cuda_ok(cudaEventRecord(b->timer[1], b->stream), "cudaEventRecord")) return HC_ERR_CUDA;
  if (!cuda_ok(cudaEventSynchronize(b->timer[1]), "cudaEventSynchronize")) return HC_ERR_CUDA;
  return cuda_ok(cudaEventElapsedTime(ms, b->timer[0], b->timer[1]), "cudaEventElapsedTime") ? HC_OK : HC_ERR_CUDA;
}
int hc_batch_launch_count(const hc_batch* b) { return b ? b->launches : 0; }
size_t hc_batch_upload_bytes(const hc_batch* b) { return b ? b->arena_bytes : 0; }
int hc_batch_k0_pictures(const hc_batch* b) { return b ? b->nk0 : 0; }
// internal (heic_job.cc): pictures of the batch whose device parse failed at the last synchronising call
int hc_batch_failed_pictures(const hc_batch* b, const int** pics) {
  if (!b) return 0;
  if (pics) *pics = b->failed_pics.data();
  return (int)b->failed_pics.size();
}
// internal (heic_job.cc): host threads hc_batch_upload may use
void hc_batch_set_pack_threads(hc_batch* b, int n) { if (b) b->pack_threads = n; }


// ---- hc_shared_image: one RGB buffer on the owner GPU that the K5 kernels of other GPUs store into ----------------------
struct hc_shared_image {
  int device = 0;          // device the VIEW belongs to (the engine that created / opened / attached it)
  int owner_device = 0;
  void* ptr = nullptr;
  size_t stride = 0;
  int width = 0, height = 0, bpp = 0;
  int kind = 0;            // 0 owner (cudaMalloc), 1 IPC mapping, 2 same-process peer view
};

static size_t shared_stride(int width, int bpp) { return align_up((size_t)((width + 7) & ~7) * bpp, 256); }

hc_shared_image* hc_shared_image_create(hc_engine* e, int width, int height, int bytes_per_pixel) {
  if (!e || width <= 0 || height <= 0 || bytes_per_pixel < 3 || bytes_per_pixel > 8) { hc::set_last_error("hc_shared_image_create: bad argument"); return nullptr; }
  if (!cuda_ok(cudaSetDevice(e->device), "cudaSetDevice")) return nullptr;
  hc_shared_image* s = new (std::nothrow) hc_shared_image;
  if (!s) return nullptr;
  s->device = s->owner_device = e->device;
  s->width = width; s->height = height; s->bpp = bytes_per_pixel;
  s->stride = shared_stride(width, bytes_per_pixel);
  if (!cuda_ok(cudaMalloc(&s->ptr, s->stride * (size_t)height), "cudaMalloc(shared image)")) { delete s; return nullptr; }
  return s;
}

int hc_shared_image_export(const hc_shared_image* s, uint8_t handle[HC_IPC_HANDLE_BYTES]) {
  static_assert(sizeof(cudaIpcMemHandle_t) == HC_IPC_HANDLE_BYTES, "IPC handle size");
  if (!s || !handle || s->kind != 0) { hc::set_last_error("hc_shared_image_export: only the owner exports"); return HC_ERR_ARGUMENT; }
  if (!cuda_ok(cudaSetDevice(s->device), "cudaSetDevice")) return HC_ERR_CUDA;
  cudaIpcMemHandle_t h;
  if (!cuda_ok(cudaIpcGetMemHandle(&h, s->ptr), "cudaIpcGetMemHandle")) return HC_ERR_CUDA;
  memcpy(handle, &h, sizeof(h));
  return HC_OK;
}

hc_shared_image* hc_shared_image_open(hc_engine* e, const uint8_t handle[HC_IPC_HANDLE_BYTES], int width, int height, int bytes_per_pixel) {
  if (!e || !handle || width <= 0 || height <= 0) { hc::set_last_error("hc_shared_image_open: bad argument"); return nullptr; }
  if (!cuda_ok(cudaSetDevice(e->device), "cudaSetDevice")) return nullptr;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  hc_shared_image* s = new (std::nothrow) hc_shared_image;
  if (!s) return nullptr;
  // the mapping is made in this device's context; stores through it travel over NVLink when the owner is a peer
  if (!cuda_ok(cudaIpcOpenMemHandle(&s->ptr, h, cudaIpcMemLazyEnablePeerAccess), "cudaIpcOpenMemHandle")) { delete s; return nullptr; }
  s->device = e->device; s->owner_device = -1; s->kind = 1;
  s->width = width; s->height = height; s->bpp = bytes_per_pixel;
  s->stride = shared_stride(width, bytes_per_pixel);
  return s;
}

hc_shared_image* hc_shared_image_attach(hc_engine* e, const hc_shared_image* owner) {
  if (!e || !owner || owner->kind != 0) { hc::set_last_error("hc_shared_image_attach: bad argument"); return nullptr; }
  if (!cuda_ok(cudaSetDevice(e->device), "cudaSetDevice")) return nullptr;
  if (e->device != owner->device) {
    int can = 0;
    cudaDeviceCanAccessPeer(&can, e->device, owner->device);
    if (!can) { hc::set_last_error("no peer access between the two devices"); return nullptr; }
    const cudaError_t r = cudaDeviceEnablePeerAccess(owner->device, 0);
    if (r != cudaSuccess && r != cudaErrorPeerAccessAlreadyEnabled) { cuda_ok(r, "cudaDeviceEnablePeerAccess"); return nullptr; }
    cudaGetLastError();   // clear "already enabled"
  }
  hc_shared_image* s = new (std::nothrow) hc_shared_image(*owner);
  if (!s) return nullptr;
  s->device = e->device;
  s->kind = 2;
  return s;
}

void hc_shared_image_destroy(hc_shared_image* s) {
  if (!s) return;
  cudaSetDevice(s->device);
  if (s->kind == 0) cudaFree(s->ptr);
  else if (s->kind == 1) cudaIpcCloseMemHandle(s->ptr);
  delete s;
}

void* hc_shared_image_device_ptr(const hc_shared_image* s) { return s ? s->ptr : nullptr; }
size_t hc_shared_image_stride(const hc_shared_image* s) { return s ? s->stride : 0; }

int hc_shared_image_read(hc_shared_image* s, int first_row, int rows, void* dst, size_t dst_stride) {
  if (!s || !dst || first_row < 0 || rows <= 0 || first_row + rows > s->height || dst_stride < (size_t)s->width * s->bpp) {
    hc::set_last_error("hc_shared_image_read: bad argument");
    return HC_ERR_ARGUMENT;
  }
  if (!cuda_ok(cudaSetDevice(s->device), "cudaSetDevice")) return HC_ERR_CUDA;
  if (!cuda_ok(cudaDeviceSynchronize(), "cudaDeviceSynchronize")) return HC_ERR_CUDA;
  return cuda_ok(cudaMemcpy2D(dst, dst_stride, (const uint8_t*)s->ptr + (size_t)first_row * s->stride, s->stride, (size_t)s->width * s->bpp, rows,
                              cudaMemcpyDeviceToHost), "cudaMemcpy2D(shared image)") ? HC_OK : HC_ERR_CUDA;
}

// used by hc_heic_job_set_rgb_target (heic_job.cc)
int hc_shared_image_geometry(const hc_shared_image* s, int* width, int* height, int* bpp) {
  if (!s) return HC_ERR_ARGUMENT;
  if (width) *width = s->width;
  if (height) *height = s->height;
  if (bpp) *bpp = s->bpp;
  return HC_OK;
}

}  // extern "C"
