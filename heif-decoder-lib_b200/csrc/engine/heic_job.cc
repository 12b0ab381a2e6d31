// heic_job.cc — HEIC files -> interleaved RGB for many files at once (include/heifcuda.h,
// "HEIC batch decode"). Host-side orchestration only: container resolution, threaded CABAC parse,
// batch placement; every pixel is produced by the device engine (no CPU reconstruction exists).
//
// Mirrors, per file, what HeifContext::decode_image_user does in the reference
// (libheif/context.cc:1516-1600): decode_image_planar (:1729) for hvc1 items, decode_full_grid_image
// (:2120-2404) + decode_and_paste_tile_image (:2407-2539) for grids, the alpha auxiliary image
// (:2029-2078), the nclx precedence (:1844-1847) and convert_colorspace (colorconversion.cc:487).
#include <atomic>
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <chrono>
#include <deque>
#include <future>
#include <mutex>
#include <thread>
#include <vector>
#include "../capi/capi_internal.h"

extern "C" void hc_batch_set_pack_threads(hc_batch* b, int n);   // engine.cu (internal)
extern "C" int hc_batch_failed_pictures(const hc_batch* b, const int** pics);
extern "C" int hc_batch_timeline_ms(hc_batch* b, float t[5]);
extern "C" void hc_batch_mark_d2h(hc_batch* b, int which);
extern "C" float hc_batch_async_d2h_ms(hc_batch* b);
extern "C" void* hc_engine_take_out_pinned(hc_engine* e, size_t bytes, size_t* cap);
extern "C" void hc_engine_give_out_pinned(hc_engine* e, void* p, size_t cap);

namespace {

// HEIFCUDA_TRACE=1: per-batch phase times of the job / stream pipeline on stderr
bool trace_on() { static const bool on = getenv("HEIFCUDA_TRACE") != nullptr; return on; }
double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// Rational arithmetic of the reference's clean-aperture evaluation (class Fraction, box.cc:51-147: 32-bit numerator /
// denominator, halved until they fit, truncating division) — the crop window must round exactly like it does.
struct Frac {
  int32_t n = 0, d = 1;
  static Frac from32(int32_t num, int32_t den) {
    Frac f; f.n = num; f.d = den;
    while (f.d > 0x10000 || f.d < -0x10000) { f.n /= 2; f.d /= 2; }
    while (f.d > 1 && (f.n > 0x10000 || f.n < -0x10000)) { f.n /= 2; f.d /= 2; }
    return f;
  }
  static Frac from64(int64_t num, int64_t den) {
    while (num < INT32_MIN || num > INT32_MAX || den < INT32_MIN || den > INT32_MAX) {
      num = (num + (num >= 0 ? 1 : -1)) / 2;
      den = (den + (den >= 0 ? 1 : -1)) / 2;
    }
    Frac f; f.n = (int32_t)num; f.d = (int32_t)den;
    return f;
  }
  Frac plus(const Frac& b) const {
    if (d == b.d) return from64((int64_t)n + b.n, d);
    return from64((int64_t)n * b.d + (int64_t)b.n * d, (int64_t)d * b.d);
  }
  Frac minus(const Frac& b) const {
    if (d == b.d) return from64((int64_t)n - b.n, d);
    return from64((int64_t)n * b.d - (int64_t)b.n * d, (int64_t)d * b.d);
  }
  Frac plus_int(int v) const { return from64(n + v * (int64_t)d, d); }
  Frac minus_int(int v) const { return from64(n - v * (int64_t)d, d); }
  Frac div_int(int v) const { return from64(n, (int64_t)d * v); }
  int32_t round_down() const { return n / d; }
  int32_t round() const { return (int32_t)((n + (int64_t)d / 2) / d); }
  bool valid() const { return d != 0; }
};

// clap -> inclusive crop window of a w x h image (Box_clap::left_rounded .. bottom_rounded, box.cc:3771-3804, and the
// clamping of context.cc:1990-2003). Returns an error text or "".
std::string clap_window(const hc::HeifItem::Clap& cl, int w, int h, int win[4]) {
  if (cl.w_num > (uint32_t)INT32_MAX || cl.w_den > (uint32_t)INT32_MAX || cl.h_num > (uint32_t)INT32_MAX || cl.h_den > (uint32_t)INT32_MAX ||
      cl.hoff_den > (uint32_t)INT32_MAX || cl.voff_den > (uint32_t)INT32_MAX)
    return "clap: exceeded supported value range";
  const Frac caw = Frac::from32((int32_t)cl.w_num, (int32_t)cl.w_den), cah = Frac::from32((int32_t)cl.h_num, (int32_t)cl.h_den);
  const Frac hoff = Frac::from32(cl.hoff_num, (int32_t)cl.hoff_den), voff = Frac::from32(cl.voff_num, (int32_t)cl.voff_den);
  if (!caw.valid() || !cah.valid() || !hoff.valid() || !voff.valid()) return "clap: invalid fractional number";
  const Frac pcx = hoff.plus(Frac::from32(w - 1, 2)), pcy = voff.plus(Frac::from32(h - 1, 2));
  const Frac fl = pcx.minus(caw.minus_int(1).div_int(2)), ft = pcy.minus(cah.minus_int(1).div_int(2));
  if (!fl.valid() || !ft.valid()) return "clap: invalid fractional number";
  int left = fl.round_down();
  int right = caw.minus_int(1).plus_int(left).round();
  int top = ft.round();
  int bottom = cah.minus_int(1).plus_int(top).round();
  if (left < 0) left = 0;
  if (top < 0) top = 0;
  if (right >= w) right = w - 1;
  if (bottom >= h) bottom = h - 1;
  if (left > right || top > bottom) return "invalid clean aperture";
  win[0] = left; win[1] = top; win[2] = right; win[3] = bottom;
  return "";
}

struct CodedItem {
  int file;
  uint32_t item_id;
  std::vector<uint8_t> stream;
  hc_records rec;                          // host-parsed records, or
  std::unique_ptr<hc_k0_picture> k0;       // headers + slice bytes for the device parser (K0)
  std::string error;
  const hc_pic& pic() const { return k0 ? k0->hp.hpic : rec.rec->pic; }
};

struct ImagePlan {
  int file = 0;
  hc_heif_image_info info{};
  std::vector<int> tiles;   // indices into items (1 for a single image)
  int alpha = -1;           // index into items (the first tile when the alpha image is a grid)
  std::vector<int> alpha_tiles;   // grid-coded alpha image: its tiles (indices into items), row-major
  int alpha_cols = 0, alpha_w = 0, alpha_h = 0;
  int band_first_row = 0;   // first tile row of a banded grid decode (multi-GPU, config C5)
  int band_y0 = 0;          // first output row of the band
  int full_height = 0;      // height of the whole image
  int canvas = -1;
  hc_image_desc desc{};
  hc_csc_params csc{};
  // 'iovl' derived image: its children are decoded on canvases of their own (hc_heic_job::children) and composed by K7
  bool overlay = false;
  uint16_t background[4] = {0, 0, 0, 0};
  std::vector<int> child_plans;                          // indices into hc_heic_job::children
  std::vector<std::pair<int32_t, int32_t>> child_offsets;
  bool scaled = false;      // delivered smaller than its full-size output (engine option "scale_max_side")
};

// the fit rule of "scale_max_side" (include/heifcuda.h): the delivered size of a W x H image, S > 0
void fit_within(int W, int H, int S, int* w, int* h) {
  *w = W; *h = H;
  if (std::max(W, H) <= S) return;
  if (W >= H) { *w = S; *h = (int)std::max<int64_t>(1, (int64_t)H * S / W); }
  else { *w = (int)std::max<int64_t>(1, (int64_t)W * S / H); *h = S; }
}

// bytes one delivered image takes: the packed planes of HC_OUT_YCBCR, else tight interleaved rows
size_t image_bytes(const hc_image_desc& d) {
  if (d.out_format == HC_OUT_YCBCR) return hc_image_plane_layout(&d, nullptr, nullptr, nullptr, nullptr);
  return (size_t)d.width * d.bytes_per_pixel * d.height;
}

int add_item(hc_batch* b, std::vector<int>& pic_file, const CodedItem& ci, int canvas, int x, int y, int role, int rescale) {
  const int pic = ci.k0 ? hc_batch_add_k0_picture(b, ci.k0.get(), canvas, x, y, role, rescale) : hc_batch_add_picture(b, &ci.rec, canvas, x, y, role, rescale);
  if (pic >= 0) {
    if ((int)pic_file.size() <= pic) pic_file.resize((size_t)pic + 1, -1);
    pic_file[pic] = ci.file;
  }
  return pic;
}

}  // namespace

struct hc_heic_job {
  hc_engine* eng = nullptr;
  hc_batch* batch = nullptr;
  std::vector<std::unique_ptr<hc::HeifFile>> files;
  std::vector<CodedItem> items;
  std::vector<ImagePlan> images;
  std::vector<ImagePlan> children;      // images that are only decoded as input of an overlay image
  double parse_seconds = 0;
  bool want_alpha = false;
  int forced_format = -1;   // HC_OUT_* for every image, or -1: by bit depth
  std::vector<int> pic_file;   // batch picture -> file it belongs to (error isolation of the stream API)
};

extern "C" {

void hc_heic_job_destroy(hc_heic_job* j) {
  if (!j) return;
  if (j->batch) hc_batch_destroy(j->batch);
  delete j;
}

}  // extern "C"

// band_begin/band_end: tile rows [begin, end) of a grid image to decode (band_end < 0: everything)
// host_share: percentage of the coded items the host threads parse although the device parser is on (hybrid; < 0: the
// engine option, where "auto" means none outside hc_heic_decode_stream)
static hc_heic_job* job_create_impl(hc_engine* e, int nfiles, const uint8_t* const* data, const size_t* sizes,
                                    int want_alpha, int threads, int band_begin, int band_end, int host_share_arg) {
  if (!e || nfiles <= 0 || !data || !sizes) {
    hc::set_last_error("hc_heic_job_create: bad argument");
    return nullptr;
  }
  std::unique_ptr<hc_heic_job> j(new hc_heic_job);
  j->eng = e;
  // `want_alpha` doubles as the output selector: 0 / 1 = automatic (RGB(A) for 8-bit images, RRGGBB(AA)_LE for deeper ones),
  // HC_OUTPUT_FORMAT(fmt) = that interleaved format for every image, whatever its bit depth, or the native planes (HC_OUT_YCBCR)
  j->forced_format = (want_alpha & 0x100) ? (want_alpha & 0xff) : -1;
  if (j->forced_format > HC_OUT_YCBCR) { hc::set_last_error("hc_heic_job_create: unknown output format"); return nullptr; }
  const bool planar = j->forced_format == HC_OUT_YCBCR;
  if (planar && band_end >= 0) { hc::set_last_error("banded decode: HC_OUT_YCBCR is not supported, bands are written as interleaved rows"); return nullptr; }
  const int scale_max = hc_engine_get_option(e, "scale_max_side");
  if (scale_max > 0 && planar) { hc::set_last_error("scale_max_side: HC_OUT_YCBCR images are not delivered scaled"); return nullptr; }
  if (scale_max > 0 && band_end >= 0) { hc::set_last_error("scale_max_side: band jobs are not delivered scaled"); return nullptr; }
  j->want_alpha = j->forced_format >= 0 ? (j->forced_format == HC_OUT_RGBA || j->forced_format == HC_OUT_RRGGBBAA_BE || j->forced_format == HC_OUT_RRGGBBAA_LE)
                                        : want_alpha != 0;
  const auto t0 = std::chrono::steady_clock::now();

  // ---- containers: which coded items does every image need? ----
  j->files.resize(nfiles);
  j->images.resize(nfiles);
  // which coded items does image item `id` of file f need? (a single picture, the tiles of a grid, an alpha image)
  auto plan_image = [&](int f, uint32_t id, ImagePlan& im) -> bool {
    hc::HeifFile& hf = *j->files[f];
    std::string err;
    im.file = f;
    const hc::HeifItem* it = hf.item(id);
    if (!it) { hc::set_last_error("file " + std::to_string(f) + ": no such image item"); return false; }
    im.info.id = id;
    im.info.rows = im.info.cols = 1;
    im.info.width = it->ispe_w;
    im.info.height = it->ispe_h;
    im.info.nclx_present = it->nclx.present;
    im.info.primaries = it->nclx.primaries;
    im.info.transfer = it->nclx.transfer;
    im.info.matrix = it->nclx.matrix;
    im.info.full_range = it->nclx.full_range;
    im.info.alpha_id = hf.alpha_item(id);
    std::vector<uint32_t> ids;
    if (hf.is_grid(id)) {
      hc::HeifGrid g;
      err = hf.grid(id, g);
      if (!err.empty()) { hc::set_last_error("file " + std::to_string(f) + ": " + err); return false; }
      im.info.is_grid = 1;
      im.info.rows = g.rows; im.info.cols = g.cols; im.info.width = g.out_w; im.info.height = g.out_h;
      // the reference's security limit (context.cc:547-560 check_resolution, heif_limits.h:37-38)
      if (g.out_w <= 0 || g.out_h <= 0 || (uint64_t)g.out_w * (uint64_t)g.out_h > (uint64_t)32768 * 32768) {
        hc::set_last_error("file " + std::to_string(f) + ": grid output size exceeds the maximum image size");
        return false;
      }
      ids = g.tiles;
      if (band_end >= 0) {
        if (band_begin < 0 || band_begin >= band_end || band_end > g.rows) { hc::set_last_error("tile row band outside the grid"); return false; }
        ids.assign(g.tiles.begin() + (size_t)band_begin * g.cols, g.tiles.begin() + (size_t)band_end * g.cols);
        im.band_first_row = band_begin;
        im.info.rows = band_end - band_begin;
      }
    } else {
      if (band_end >= 0) { hc::set_last_error("a tile row band needs a grid image"); return false; }
      ids.push_back(id);
    }
    if (band_end >= 0 && im.info.alpha_id) { hc::set_last_error("banded decode of images with an alpha plane is not supported"); return false; }
    for (uint32_t t : ids) {
      im.tiles.push_back((int)j->items.size());
      j->items.emplace_back();
      j->items.back().file = f;
      j->items.back().item_id = t;
    }
    if (im.info.alpha_id && hf.is_grid(im.info.alpha_id)) {
      // the alpha image is decoded like any image item (context.cc:2040-2071 decode_image_planar), so it may be a grid too
      hc::HeifGrid ag;
      err = hf.grid(im.info.alpha_id, ag);
      if (!err.empty()) { hc::set_last_error("file " + std::to_string(f) + ": alpha image: " + err); return false; }
      if (ag.out_w <= 0 || ag.out_h <= 0 || (uint64_t)ag.out_w * (uint64_t)ag.out_h > (uint64_t)32768 * 32768) {
        hc::set_last_error("file " + std::to_string(f) + ": grid output size exceeds the maximum image size");
        return false;
      }
      im.alpha = (int)j->items.size();
      im.alpha_cols = ag.cols; im.alpha_w = ag.out_w; im.alpha_h = ag.out_h;
      for (uint32_t t : ag.tiles) {
        im.alpha_tiles.push_back((int)j->items.size());
        j->items.emplace_back();
        j->items.back().file = f;
        j->items.back().item_id = t;
      }
    } else if (im.info.alpha_id) {
      im.alpha = (int)j->items.size();
      j->items.emplace_back();
      j->items.back().file = f;
      j->items.back().item_id = im.info.alpha_id;
    }
    return true;
  };
  for (int f = 0; f < nfiles; f++) {
    j->files[f].reset(new hc::HeifFile);
    std::string err = j->files[f]->parse(data[f], sizes[f]);
    if (!err.empty()) { hc::set_last_error("file " + std::to_string(f) + ": " + err); return nullptr; }
    hc::HeifFile& hf = *j->files[f];
    ImagePlan& im = j->images[f];
    const uint32_t id = hf.primary_id();
    if (hf.is_overlay(id)) {
      // 'iovl' (context.cc:2579-2675): every referenced image is decoded like a top-level image, then composed
      if (band_end >= 0) { hc::set_last_error("a tile row band needs a grid image"); return nullptr; }
      if (planar) { hc::set_last_error("file " + std::to_string(f) + ": overlay images are composed in RGB: HC_OUT_YCBCR is not supported for them"); return nullptr; }
      hc::HeifOverlay ov;
      err = hf.overlay(id, ov);
      if (!err.empty()) { hc::set_last_error("file " + std::to_string(f) + ": " + err); return nullptr; }
      if (ov.children.size() != ov.offsets.size()) { hc::set_last_error("Number of image offsets does not match the number of image references"); return nullptr; }
      const hc::HeifItem* oit = hf.item(id);
      if (oit && !oit->xforms.empty()) { hc::set_last_error("transformations on overlay images are not supported"); return nullptr; }
      im.file = f;
      im.overlay = true;
      im.info.id = id;
      im.info.rows = im.info.cols = 1;
      im.info.width = ov.canvas_w; im.info.height = ov.canvas_h;
      for (int k = 0; k < 4; k++) im.background[k] = ov.background[k];
      im.child_offsets = ov.offsets;
      for (uint32_t cid : ov.children) {
        ImagePlan child;
        if (hf.is_overlay(cid)) { hc::set_last_error("nested overlay images are not supported"); return nullptr; }
        if (!plan_image(f, cid, child)) return nullptr;
        im.child_plans.push_back((int)j->children.size());
        j->children.push_back(child);
      }
      continue;
    }
    if (!plan_image(f, id, im)) return nullptr;
  }

  const double t_containers = now_s();
  // ---- serial CABAC parse of every coded item, in parallel across items ----
  int nthreads = threads > 0 ? threads : (int)std::thread::hardware_concurrency();
  if (nthreads < 1) nthreads = 1;
  nthreads = std::min<int>(nthreads, (int)j->items.size());
  const bool device_parse = hc_engine_get_option(e, "device_parse") != 0;
  const int k0_max_critical = hc_engine_get_option(e, "k0_max_critical_ctbs");
  bool device_parse_job = device_parse;
  if (device_parse && host_share_arg < 0 && hc_engine_get_option(e, "host_share_pct") < 0) {
    // A single job cannot overlap its host parse with K0 (K0 starts at hc_heic_job_run), so with the automatic setting
    // it takes whichever side is expected to finish first: K0 costs its critical path (~3 ms per CTB of a chain, measured
    // on B200) or its throughput (~1000 CTBs in flight), the host ~0.09 ms per CTB and thread. One 12 MP grid file parses
    // faster on 16 host threads (17 ms vs 66 ms); from a handful of files on, the GPU wins.
    double ctbs = 0, critical = 0;
    for (const CodedItem& ci : j->items) {
      const hc::HeifItem* it = j->files[ci.file]->item(ci.item_id);
      if (!it) continue;
      const double cw = (it->ispe_w + 63) / 64, ch = (it->ispe_h + 63) / 64;
      ctbs += cw * ch;
      critical = std::max(critical, cw + 2 * (ch - 1));
    }
    const double est_host = ctbs * 0.09 / nthreads, est_k0 = std::max(critical * 3.0, ctbs * 3.0 / 1000.0);
    device_parse_job = est_k0 < est_host;
  }
  const int host_share = !device_parse ? 0 : (host_share_arg >= 0 ? host_share_arg : std::max(0, hc_engine_get_option(e, "host_share_pct")));
  std::atomic<size_t> next{0};
  auto parse_item = [&](size_t i) {
      CodedItem& ci = j->items[i];
      std::string err = j->files[ci.file]->coded_stream(ci.item_id, ci.stream);
      if (!err.empty()) { ci.error = err; return; }
      // hybrid: while the GPU parses the previous batch, the host cores parse an evenly spread share of this one
      const bool to_host = host_share > 0 && ((i + 1) * (size_t)host_share) / 100 != (i * (size_t)host_share) / 100;
      if (device_parse_job && !to_host) {
        // K0: only parameter sets and slice headers are read here; the GPU parses the slice data
        std::unique_ptr<hc_k0_picture> k(new hc_k0_picture);
        err = hc::k0_prepare(ci.stream.data(), ci.stream.size(), HC_STREAM_LENGTH_PREFIXED, k->hp);
        if (!err.empty()) { ci.error = err; return; }
        // K0 is serial per substream: a picture is worth parsing on the GPU when its critical path is short — CTB rows of
        // a WPP picture advance two CTBs behind each other, a picture without WPP is ONE chain of all its CTBs (a 1080p
        // picture: 510 CTBs x ~3 ms against ~40 ms on one host core). Long ones stay with the host parser.
        bool short_enough = false;
        if (k->hp.eligible) {
          const hc::k0::Pic& kp = k->hp.pic;
          const bool rows = !k->hp.subs.empty() && (k->hp.subs[0].flags & hc::k0::SUB_ROW_CHAIN);
          const int critical = rows ? kp.ctbs_w + 2 * (kp.ctbs_h - 1) : kp.ctbs_w * kp.ctbs_h;
          short_enough = critical <= k0_max_critical;
        }
        if (k->hp.eligible && short_enough) {
          ci.k0 = std::move(k);
          std::vector<uint8_t>().swap(ci.stream);
          return;
        }
      }
      thread_local hc::HevcIntraParser parser;   // reused: see k0_prepare
      parser.reset();
      parser.set_collect_only(false);
      err = parser.push_length_prefixed(ci.stream.data(), ci.stream.size());
      if (!err.empty()) { ci.error = err; return; }
      ci.rec.rec = parser.take_picture(&err);
      if (!ci.rec.rec) ci.error = err;
      std::vector<uint8_t>().swap(ci.stream);
  };
  // the workers are std::threads: an exception leaving one would terminate the process
  auto worker = [&]() {
    for (;;) {
      const size_t i = next.fetch_add(1);
      if (i >= j->items.size()) return;
      try {
        parse_item(i);
      } catch (const std::bad_alloc&) {
        j->items[i].error = "out of memory while parsing";
      } catch (const std::exception& ex) {
        j->items[i].error = std::string("parser failure: ") + ex.what();
      }
    }
  };
  if (nthreads == 1) worker();
  else {
    std::vector<std::thread> pool;
    for (int t = 0; t < nthreads; t++) pool.emplace_back(worker);
    for (auto& t : pool) t.join();
  }
  for (auto& ci : j->items)
    if (!ci.error.empty()) {
      hc::set_last_error("file " + std::to_string(ci.file) + " item " + std::to_string(ci.item_id) + ": " + ci.error);
      return nullptr;
    }
  j->parse_seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
  const double t_parsed = now_s();

  // ---- batch placement ----
  j->batch = hc_batch_create(e);
  if (!j->batch) return nullptr;
  hc_batch_set_pack_threads(j->batch, threads > 0 ? threads : 0);
  // one image item -> canvas, pictures, transformation passes, colour conversion parameters (`fmt_override` >= 0: the
  // conversion parameters are selected for that output format, used for overlay children)
  auto place_image = [&](ImagePlan& im, int fmt_override) -> bool {
    const hc_pic& p0 = j->items[im.tiles[0]].pic();
    const bool has_alpha = im.alpha >= 0;
    int W = im.info.width, H = im.info.height;
    if (!im.info.is_grid) { W = p0.crop_w; H = p0.crop_h; }   // decoded size, like the reference
    im.full_height = H;
    if (im.info.is_grid && band_end >= 0) {                     // this job owns output rows [y0, y0 + H)
      im.band_y0 = im.band_first_row * p0.crop_h;
      if (im.band_y0 >= H) { hc::set_last_error("tile row band lies below the output image"); return false; }
      H = std::min(H, band_end * p0.crop_h) - im.band_y0;
    }
    im.canvas = hc_batch_add_canvas(j->batch, W, H, p0.chroma_format, p0.bit_depth_y, has_alpha);
    if (im.canvas < 0) return false;
    int matrix, primaries, full;
    // the tiles of one grid item onto one canvas (context.cc:2328-2337, :2407-2539)
    auto place_tiles = [&](const std::vector<int>& tiles, int cols, int canvas, int CW, int CH, int role) -> bool {
      const hc_pic& t0 = j->items[tiles[0]].pic();
      const int tw = t0.crop_w, th = t0.crop_h;
      for (size_t k = 0; k < tiles.size(); k++) {
        CodedItem& ci = j->items[tiles[k]];
        const hc_pic& p = ci.pic();
        const hc::HeifItem* tit = j->files[im.file]->item(ci.item_id);
        if (p.crop_w != tw || p.crop_h != th) { hc::set_last_error("Grid tiles have different sizes"); return false; }
        if (p.chroma_format != t0.chroma_format || p.bit_depth_y != t0.bit_depth_y) { hc::set_last_error("grid tiles differ in chroma format or bit depth"); return false; }
        if (tit && !tit->xforms.empty()) { hc::set_last_error("transformations on grid tile items are not supported"); return false; }
        const int tfull = tit && tit->nclx.present ? tit->nclx.full_range : p.full_range;
        const int tmatrix = tit && tit->nclx.present ? tit->nclx.matrix : p.matrix_coeffs;
        const int x0 = (int)(k % cols) * tw, y0 = (int)(k / cols) * th;
        if (x0 >= CW || y0 >= CH) { hc::set_last_error("grid tile lies outside the output image"); return false; }
        if (add_item(j->batch, j->pic_file, ci, canvas, x0, y0, role, (!tfull && tmatrix != 0) ? 1 : 0) < 0) return false;
      }
      return true;
    };
    if (im.info.is_grid) {
      const int tw = p0.crop_w, th = p0.crop_h;
      for (size_t k = 0; k < im.tiles.size(); k++) {
        CodedItem& ci = j->items[im.tiles[k]];
        const hc_pic& p = ci.pic();
        const hc::HeifItem* tit = j->files[im.file]->item(ci.item_id);
        // context.cc:2328-2337: every tile has the size of the first one ("Grid tiles have different sizes"); tiles of another
        // chroma format or bit depth cannot share a canvas (the reference fails in its paste, context.cc:2452-2465)
        if (p.crop_w != tw || p.crop_h != th) { hc::set_last_error("Grid tiles have different sizes"); return false; }
        if (p.chroma_format != p0.chroma_format || p.bit_depth_y != p0.bit_depth_y) { hc::set_last_error("grid tiles differ in chroma format or bit depth"); return false; }
        // the reference decodes every tile through decode_image_planar, which applies the tile item's own irot / imir / clap
        // (context.cc:1955-2016) before the paste; that combination is not built here
        if (tit && !tit->xforms.empty()) { hc::set_last_error("transformations on grid tile items are not supported"); return false; }
        const int tfull = tit && tit->nclx.present ? tit->nclx.full_range : p.full_range;
        const int tmatrix = tit && tit->nclx.present ? tit->nclx.matrix : p.matrix_coeffs;
        const int x0 = (int)(k % im.info.cols) * tw, y0 = (int)(k / im.info.cols) * th;
        if (x0 >= W || y0 >= H) { hc::set_last_error("grid tile lies outside the output image"); return false; }
        // context.cc:2504: limited-range tiles (matrix != 0) are expanded to full range while pasting
        if (add_item(j->batch, j->pic_file, ci, im.canvas, x0, y0, HC_ROLE_COLOUR, (!tfull && tmatrix != 0) ? 1 : 0) < 0) return false;
      }
      // the canvas only has an nclx if the grid item itself carries one (context.cc:1841-1844)
      matrix = im.info.nclx_present ? im.info.matrix : 2;
      primaries = im.info.nclx_present ? im.info.primaries : 2;
      full = im.info.nclx_present ? im.info.full_range : 1;
    } else {
      if (add_item(j->batch, j->pic_file, j->items[im.tiles[0]], im.canvas, 0, 0, HC_ROLE_COLOUR, 0) < 0) return false;
      matrix = im.info.nclx_present ? im.info.matrix : p0.matrix_coeffs;
      primaries = im.info.nclx_present ? im.info.primaries : p0.colour_primaries;
      full = im.info.nclx_present ? im.info.full_range : p0.full_range;
    }
    // ---- irot / imir / clap of an image item, in ipma order (context.cc:1955-2016). Consecutive rotations and mirrors
    // are composed into one dihedral pass; a clap becomes a crop pass on the image as it is at that point. Returns
    // false on error; `any` reports whether the item carries transformations at all. Cw x Ch follows the size of the chroma
    // planes through the passes (HeifPixelImage::crop scales the window to each plane, pixelimage.cc:820-823, as the
    // engine's crop pass does). ----
    auto apply_xforms = [&](int canvas, const hc::HeifItem* pit, int& Wc, int& Hc, int& Cw, int& Ch, int chroma_format, int bit_depth,
                            bool& any) -> bool {
      int swap = 0, fx = 0, fy = 0;
      any = false;
      size_t next_clap = 0;
      auto flush_dihedral = [&]() -> bool {
        if (!(swap | fx | fy)) return true;
        if (swap && chroma_format == 2) { hc::set_last_error("quarter turns of 4:2:2 images are not supported"); return false; }
        if (hc_batch_add_canvas_pass(j->batch, canvas, HC_PASS_DIHEDRAL, swap, fx, fy, 0) != HC_OK) return false;
        swap = fx = fy = 0;
        return true;
      };
      if (!pit) return true;
      for (uint8_t op : pit->xforms) {
        any = true;
        if (op == HC_XF_CLAP) {
          if (!flush_dihedral()) return false;
          if (next_clap >= pit->claps.size()) { hc::set_last_error("clap property without its box"); return false; }
          int win[4] = {0, 0, 0, 0};
          const std::string e = clap_window(pit->claps[next_clap++], Wc, Hc, win);
          if (!e.empty()) { hc::set_last_error(e); return false; }
          if (hc_batch_add_canvas_pass(j->batch, canvas, HC_PASS_CROP, win[0], win[1], win[2], win[3]) != HC_OK) return false;
          if (Cw > 0) {
            Cw = (int)((int64_t)win[2] * Cw / Wc - (int64_t)win[0] * Cw / Wc) + 1;
            Ch = (int)((int64_t)win[3] * Ch / Hc - (int64_t)win[1] * Ch / Hc) + 1;
          }
          Wc = win[2] - win[0] + 1; Hc = win[3] - win[1] + 1;
          continue;
        }
        const int s2 = (op == HC_XF_ROT90 || op == HC_XF_ROT270) ? 1 : 0;
        const int fx2 = (op == HC_XF_ROT90 || op == HC_XF_ROT180 || op == HC_XF_MIRROR_H) ? 1 : 0;
        const int fy2 = (op == HC_XF_ROT270 || op == HC_XF_ROT180 || op == HC_XF_MIRROR_V) ? 1 : 0;
        if ((op == HC_XF_MIRROR_H || op == HC_XF_MIRROR_V) && bit_depth != 8) {
          hc::set_last_error("Can currently only mirror images with 8 bits per pixel");   // pixelimage.cc:748-752
          return false;
        }
        // out2(x, y) = out1(x1, y1): see hc_batch_set_canvas_transform for the map of one operation
        const int nfx = swap ? (fx ^ fy2) : (fx ^ fx2), nfy = swap ? (fy ^ fx2) : (fy ^ fy2);
        swap ^= s2; fx = nfx; fy = nfy;
        if (s2) { std::swap(Wc, Hc); std::swap(Cw, Ch); }
      }
      return flush_dihedral();
    };
    const hc::HeifItem* pit = j->files[im.file]->item(im.info.id);
    const hc::HeifItem* ait = has_alpha ? j->files[im.file]->item(im.info.alpha_id) : nullptr;
    // Is the alpha image pasted straight into the canvas' alpha plane (same decoded size, same transformations), or
    // decoded on its own canvas, transformed by its own properties and rescaled by nearest neighbour afterwards
    // (context.cc:2040-2071: decode_image_planar of the alpha item, then scale_nearest_neighbor to the colour image's size)?
    bool alpha_separate = false;
    const bool alpha_grid = !im.alpha_tiles.empty();
    if (has_alpha) {
      const hc_pic& pa = j->items[im.alpha].pic();
      // a grid-coded alpha image always gets a canvas of its own (its tiles are pasted there like those of any grid)
      bool same = !alpha_grid && pa.crop_w == W && pa.crop_h == H;
      if (same && pit && !pit->xforms.empty()) {
        same = ait && ait->xforms == pit->xforms && ait->claps.size() == pit->claps.size();
        for (size_t k = 0; same && k < pit->claps.size(); k++) same = memcmp(&ait->claps[k], &pit->claps[k], sizeof(hc::HeifItem::Clap)) == 0;
      } else if (same && ait && !ait->xforms.empty()) {
        same = false;
      }
      alpha_separate = !same;
      if (!alpha_separate && add_item(j->batch, j->pic_file, j->items[im.alpha], im.canvas, 0, 0, HC_ROLE_ALPHA, 0) < 0) return false;
    }
    {
      bool any = false;
      int Cw = hc::plane_w(W, p0.chroma_format, 1), Ch = hc::plane_h(H, p0.chroma_format, 1);
      if (!apply_xforms(im.canvas, pit, W, H, Cw, Ch, p0.chroma_format, p0.bit_depth_y, any)) return false;
      if (any && band_end >= 0) { hc::set_last_error("banded decode of transformed images is not supported"); return false; }
      // the packed layout (hc_image_plane_layout) has (w + 1) / 2 chroma samples per row of 4:2:0 / 4:2:2 and (h + 1) / 2 rows
      // of 4:2:0; a clean aperture at an odd position leaves one more, and the desc cannot describe that
      if (fmt_override < 0 && planar && (Cw != hc::plane_w(W, p0.chroma_format, 1) || Ch != hc::plane_h(H, p0.chroma_format, 1))) {
        hc::set_last_error("file " + std::to_string(im.file) + ": HC_OUT_YCBCR: the clean aperture leaves chroma planes of " + std::to_string(Cw) +
                           " x " + std::to_string(Ch) + " samples, not the packed layout's " + std::to_string(hc::plane_w(W, p0.chroma_format, 1)) + " x " +
                           std::to_string(hc::plane_h(H, p0.chroma_format, 1)));
        return false;
      }
    }
    if (alpha_separate) {
      const hc_pic& pa = j->items[im.alpha].pic();
      int Wa = alpha_grid ? im.alpha_w : pa.crop_w, Ha = alpha_grid ? im.alpha_h : pa.crop_h;
      const int ac = hc_batch_add_canvas(j->batch, Wa, Ha, 0, pa.bit_depth_y, 0);
      if (ac < 0) return false;
      if (alpha_grid) {
        if (!place_tiles(im.alpha_tiles, im.alpha_cols, ac, Wa, Ha, HC_ROLE_LUMA)) return false;
      } else if (add_item(j->batch, j->pic_file, j->items[im.alpha], ac, 0, 0, HC_ROLE_LUMA, 0) < 0) return false;
      bool any = false;
      int Cwa = 0, Cha = 0;   // monochrome: no chroma planes
      if (!apply_xforms(ac, ait, Wa, Ha, Cwa, Cha, 0, pa.bit_depth_y, any)) return false;
      if (hc_batch_link_alpha(j->batch, im.canvas, ac) != HC_OK) return false;
    }
    const bool hdr = p0.bit_depth_y != 8;
    const int fmt = fmt_override >= 0 ? fmt_override : j->forced_format >= 0 ? j->forced_format : (hdr ? (j->want_alpha ? HC_OUT_RRGGBBAA_LE : HC_OUT_RRGGBB_LE) : (j->want_alpha ? HC_OUT_RGBA : HC_OUT_RGB));
    if (hc_csc_select_opt(matrix, primaries, full, p0.chroma_format, p0.bit_depth_y, has_alpha, fmt, hc_engine_get_option(e, "chroma_upsampling"), &im.csc) != HC_OK) return false;
    static const int bpp_of[6] = {3, 4, 6, 8, 6, 8};
    im.desc.width = W; im.desc.height = H; im.desc.chroma_format = p0.chroma_format; im.desc.bit_depth = p0.bit_depth_y;
    im.desc.has_alpha = has_alpha; im.desc.out_format = fmt;
    im.desc.bytes_per_pixel = fmt == HC_OUT_YCBCR ? (p0.bit_depth_y == 8 ? 1 : 2) : bpp_of[fmt];
    im.desc.coded_pictures = (int)im.tiles.size() + (has_alpha ? (alpha_grid ? (int)im.alpha_tiles.size() : 1) : 0);
    // premultiplied alpha: a flag the file sets ('prem' reference, context.cc:1150-1161, :2074-2075) — or the result of
    // heif_image_rgba_premultiply_alpha (heif.cc:1444-1490), which only takes interleaved RGBA that is not premultiplied yet
    im.desc.premultiplied_alpha = has_alpha && j->files[im.file]->premultiplied(im.info.id) ? 1 : 0;
    if (hc_engine_get_option(e, "premultiply_alpha") && fmt == HC_OUT_RGBA && !im.desc.premultiplied_alpha) {
      im.csc.premultiply = 1;
      im.desc.premultiplied_alpha = 1;
    }
    return true;
  };
  for (ImagePlan& im : j->images) {
    if (!im.overlay) {
      if (!place_image(im, -1)) return nullptr;
      continue;
    }
    // 'iovl': children first (each on its own canvas, converted like Op_YCbCr_to_RGB<uint8_t> would), then the overlay canvas
    im.canvas = -1;
    std::vector<int> child_canvases;
    for (int ci : im.child_plans) {
      ImagePlan& ch = j->children[ci];
      if (!place_image(ch, HC_OUT_RGB)) return nullptr;
      if (ch.desc.bit_depth != 8 || ch.desc.chroma_format != 3) {   // context.cc:2650-2654: the only children the reference converts
        hc::set_last_error("Unsupported color conversion: the reference only composes overlays of 8-bit 4:4:4 images");
        return nullptr;
      }
      child_canvases.push_back(ch.canvas);
    }
    im.canvas = hc_batch_add_overlay_canvas(j->batch, im.info.width, im.info.height, im.background);
    if (im.canvas < 0) return nullptr;
    for (size_t k = 0; k < child_canvases.size(); k++) {
      const ImagePlan& ch = j->children[im.child_plans[k]];
      if (hc_batch_overlay_add_child(j->batch, im.canvas, child_canvases[k], im.child_offsets[k].first, im.child_offsets[k].second, &ch.csc) != HC_OK) return nullptr;
    }
    const int fmt = j->forced_format >= 0 ? j->forced_format : (j->want_alpha ? HC_OUT_RGBA : HC_OUT_RGB);
    static const int bpp_of_fmt[6] = {3, 4, 6, 8, 6, 8};
    memset(&im.csc, 0, sizeof(im.csc));
    im.csc.out_format = fmt;
    im.desc.width = im.info.width; im.desc.height = im.info.height; im.desc.chroma_format = 3; im.desc.bit_depth = 8;
    im.desc.has_alpha = 0; im.desc.out_format = fmt; im.desc.bytes_per_pixel = bpp_of_fmt[fmt];
    im.desc.coded_pictures = 0;
    for (int ci : im.child_plans) im.desc.coded_pictures += j->children[ci].desc.coded_pictures;
  }
  if (scale_max > 0) {
    // overlay children stay full size: K7 samples the composed image
    for (ImagePlan& im : j->images) {
      int w, h;
      fit_within(im.desc.width, im.desc.height, scale_max, &w, &h);
      if (w == im.desc.width && h == im.desc.height) continue;
      if (hc_batch_set_canvas_output_size(j->batch, im.canvas, w, h) != HC_OK) return nullptr;
      im.desc.width = w; im.desc.height = h;
      im.scaled = true;
    }
  }
  if (trace_on())
    fprintf(stderr, "[heifcuda] job_create: %d files, %zu items: containers %.2f ms, parse/prepare %.2f ms (%d threads), placement %.2f ms\n", nfiles,
            j->items.size(), (t_containers - std::chrono::duration<double>(t0.time_since_epoch()).count()) * 1e3, (t_parsed - t_containers) * 1e3, nthreads,
            (now_s() - t_parsed) * 1e3);
  return j.release();
}

// No exception may cross the C ABI: a crafted file can make any allocation of the walk above fail.
static hc_heic_job* job_create(hc_engine* e, int nfiles, const uint8_t* const* data, const size_t* sizes,
                               int want_alpha, int threads, int band_begin, int band_end, int host_share_arg = -1) {
  try {
    return job_create_impl(e, nfiles, data, sizes, want_alpha, threads, band_begin, band_end, host_share_arg);
  } catch (const std::bad_alloc&) {
    hc::set_last_error("out of memory while preparing the job");
  } catch (const std::exception& ex) {
    hc::set_last_error(std::string("job preparation failed: ") + ex.what());
  }
  return nullptr;
}

extern "C" {

hc_heic_job* hc_heic_job_create(hc_engine* e, int nfiles, const uint8_t* const* data, const size_t* sizes,
                                int want_alpha, int threads) {
  return job_create(e, nfiles, data, sizes, want_alpha, threads, 0, -1);
}

hc_heic_job* hc_heic_job_create_band(hc_engine* e, const uint8_t* data, size_t size, int want_alpha, int threads,
                                     int tile_row_begin, int tile_row_end, int* first_output_row, int* full_height) {
  if (tile_row_end < 0) { hc::set_last_error("hc_heic_job_create_band: bad band"); return nullptr; }
  hc_heic_job* j = job_create(e, 1, &data, &size, want_alpha, threads, tile_row_begin, tile_row_end);
  if (j && first_output_row) *first_output_row = j->images[0].band_y0;
  if (j && full_height) *full_height = j->images[0].full_height;
  return j;
}

extern "C" int hc_shared_image_geometry(const hc_shared_image* s, int* width, int* height, int* bpp);

int hc_heic_job_set_rgb_target(hc_heic_job* j, int image, hc_shared_image* dst, int first_row) {
  if (!j || image < 0 || image >= (int)j->images.size() || !dst || first_row < 0) { hc::set_last_error("hc_heic_job_set_rgb_target: bad argument"); return HC_ERR_ARGUMENT; }
  const ImagePlan& im = j->images[image];
  if (im.desc.out_format == HC_OUT_YCBCR) { hc::set_last_error("hc_heic_job_set_rgb_target: HC_OUT_YCBCR images are not written to shared images"); return HC_ERR_UNSUPPORTED; }
  if (im.scaled) { hc::set_last_error("hc_heic_job_set_rgb_target: scaled images are not written to shared images"); return HC_ERR_UNSUPPORTED; }
  int w = 0, h = 0, bpp = 0;
  hc_shared_image_geometry(dst, &w, &h, &bpp);
  if (w != im.desc.width || bpp != im.desc.bytes_per_pixel || first_row + im.desc.height > h) {
    hc::set_last_error("hc_heic_job_set_rgb_target: the image does not fit the shared image (width / pixel size / rows)");
    return HC_ERR_ARGUMENT;
  }
  return hc_batch_set_rgb_target(j->batch, im.canvas, (uint8_t*)hc_shared_image_device_ptr(dst) + (size_t)first_row * hc_shared_image_stride(dst), hc_shared_image_stride(dst));
}

int hc_heic_job_copy_rgb_device(hc_heic_job* j, int image, void* device_dst, size_t dst_stride_bytes) {
  if (!j || image < 0 || image >= (int)j->images.size()) { hc::set_last_error("hc_heic_job_copy_rgb_device: bad argument"); return HC_ERR_ARGUMENT; }
  return hc_batch_copy_rgb_device(j->batch, j->images[image].canvas, device_dst, dst_stride_bytes);
}

int hc_heic_job_image_count(const hc_heic_job* j) { return j ? (int)j->images.size() : 0; }

int hc_heic_job_image_desc(const hc_heic_job* j, int image, hc_image_desc* desc) {
  if (!j || !desc || image < 0 || image >= (int)j->images.size()) { hc::set_last_error("hc_heic_job_image_desc: bad argument"); return HC_ERR_ARGUMENT; }
  *desc = j->images[image].desc;
  return HC_OK;
}

int hc_heic_job_upload(hc_heic_job* j) { return j ? hc_batch_upload(j->batch) : HC_ERR_ARGUMENT; }

int hc_heic_job_run(hc_heic_job* j) {
  if (!j) return HC_ERR_ARGUMENT;
  int rc = hc_batch_reconstruct_async(j->batch, HC_STAGE_ALL);   // K0 errors surface in hc_heic_job_sync / read
  if (rc != HC_OK) return rc;
  std::vector<int> canvases;
  std::vector<hc_csc_params> params;
  for (ImagePlan& im : j->images) { canvases.push_back(im.canvas); params.push_back(im.csc); }
  return hc_batch_convert_many(j->batch, (int)canvases.size(), canvases.data(), params.data());
}

int hc_heic_job_sync(hc_heic_job* j) { return j ? hc_batch_sync(j->batch) : HC_ERR_ARGUMENT; }

int hc_heic_job_read_rgb(hc_heic_job* j, int image, void* dst, size_t stride) {
  if (!j || image < 0 || image >= (int)j->images.size()) { hc::set_last_error("hc_heic_job_read_rgb: bad argument"); return HC_ERR_ARGUMENT; }
  return hc_batch_read_rgb(j->batch, j->images[image].canvas, dst, stride);
}

int hc_heic_job_read_plane(hc_heic_job* j, int image, int plane, void* dst, size_t stride) {
  if (!j || image < 0 || image >= (int)j->images.size()) { hc::set_last_error("hc_heic_job_read_plane: bad argument"); return HC_ERR_ARGUMENT; }
  // the planes are full size, the desc (which sizes the caller's destination) is the delivered size
  if (j->images[image].scaled) { hc::set_last_error("hc_heic_job_read_plane: the image is delivered scaled"); return HC_ERR_UNSUPPORTED; }
  return hc_batch_read_plane(j->batch, j->images[image].canvas, plane, dst, stride);
}

int hc_heic_job_stage_ms(hc_heic_job* j, float ms[8]) { return j ? hc_batch_stage_ms(j->batch, ms) : HC_ERR_ARGUMENT; }
int hc_heic_job_timer_start(hc_heic_job* j) { return j ? hc_batch_timer_start(j->batch) : HC_ERR_ARGUMENT; }
int hc_heic_job_timer_stop_ms(hc_heic_job* j, float* ms) { return j ? hc_batch_timer_stop_ms(j->batch, ms) : HC_ERR_ARGUMENT; }
int hc_heic_job_launch_count(const hc_heic_job* j) { return j ? hc_batch_launch_count(j->batch) : 0; }
size_t hc_heic_job_upload_bytes(const hc_heic_job* j) { return j ? hc_batch_upload_bytes(j->batch) : 0; }
double hc_heic_job_parse_seconds(const hc_heic_job* j) { return j ? j->parse_seconds : 0.0; }

int hc_heic_decode_stream(hc_engine* e, int nfiles, const uint8_t* const* data, const size_t* sizes, int want_alpha,
                          int threads, int files_per_batch, hc_image_callback on_image, void* user,
                          hc_stream_stats* stats) {
  return hc_heic_decode_stream_ext(e, nfiles, data, sizes, want_alpha, threads, files_per_batch, nullptr, nullptr, on_image, user, stats);
}

int hc_heic_decode_stream_ext(hc_engine* e, int nfiles, const uint8_t* const* data, const size_t* sizes, int want_alpha,
                              int threads, int files_per_batch_arg, const hc_stream_dest* dests, int* file_status, hc_image_callback on_image,
                              void* user, hc_stream_stats* stats) {
  int files_per_batch = files_per_batch_arg;
  if (e && nfiles > 0 && data && sizes && files_per_batch == 0) {
    // automatic batch size: the device parser wants some 20,000 substream chains in flight and the kernels behind it stream;
    // measured optimum 64 files of 12 MP (3.6 -> 3.9 GP/s against 32) and 384 of 1080p (1.5 -> 3.2 GP/s against 96), i.e.
    // about 800 MP of output per batch — taken from the size of the LARGEST primary image among up to 32 files sampled
    // evenly over the list (a batch of the largest must fit)
    double mp = 0.0;
    const int nsample = std::min(nfiles, 32);
    for (int q = 0; q < nsample; q++) {
      const int k = (int)((long long)q * nfiles / nsample);
      hc::HeifFile hf;
      if (!hf.parse(data[k], sizes[k]).empty()) continue;
      const hc::HeifItem* it = hf.item(hf.primary_id());
      if (it && it->ispe_w > 0 && it->ispe_h > 0) mp = std::max(mp, (double)it->ispe_w * it->ispe_h / 1e6);
    }
    if (mp <= 0.0) mp = 12.0;
    files_per_batch = (int)std::max(1.0, std::min(512.0, 800.0 / std::max(mp, 0.05)));
  }
  if (!e || nfiles <= 0 || !data || !sizes || files_per_batch <= 0) {
    hc::set_last_error("hc_heic_decode_stream: bad argument");
    return HC_ERR_ARGUMENT;
  }
  if ((want_alpha & 0x100) && (want_alpha & 0xff) == HC_OUT_YCBCR && hc_engine_get_option(e, "scale_max_side") > 0) {
    // a property of the call, not of a file: error isolation would otherwise fail every file on its own
    hc::set_last_error("scale_max_side: HC_OUT_YCBCR images are not delivered scaled");
    return HC_ERR_UNSUPPORTED;
  }
  using clock = std::chrono::steady_clock;
  auto secs = [](clock::time_point a, clock::time_point b) { return std::chrono::duration<double>(b - a).count(); };
  hc_stream_stats st{};
  const auto t_begin = clock::now();
  const int nbatches = (nfiles + files_per_batch - 1) / files_per_batch;

  // stage 1 (host threads): container + CABAC parse of one batch; runs one batch ahead of stage 2
  // Hybrid parse: with the device parser on, the host threads that prepare batch b+1 would idle while the GPU works on
  // batch b, so they parse a share of the coded items themselves. "auto" (engine option -1) starts from a static prior
  // and follows the measured costs per item on either side, so that a rank with few host threads ends up at 0.
  const int share_opt = hc_engine_get_option(e, "host_share_pct");
  // static prior (per coded 512 x 512 item, measured on B200 + this box's cores): device 0.069 ms in the steady state of
  // the pipeline (K0-bound: 97 ms + 9 ms of K1..K5 per 1536 items); one host thread 4 ms for the slice data of an item
  // it parses itself and 0.08 ms for the container / header work every item needs. The host must finish
  // n * c_hdr + share * n * c_host within 0.9 of the device's (1 - share) * n * c_dev, hence balanced_share() — which is 0
  // for a rank with two host threads (8 ranks on a 16-core box): there the headers alone take most of a period.
  const int pool_threads = threads > 0 ? threads : std::max(1, (int)std::thread::hardware_concurrency());
  const double c_dev0 = 0.069e-3, c_host0 = 4.0e-3 / pool_threads, c_hdr0 = 0.08e-3 / pool_threads;
  auto balanced_share = [](double c_dev, double c_host, double c_hdr) {
    const double s = (0.9 * c_dev - c_hdr) / (c_host + 0.9 * c_dev);
    return std::max(0, std::min(90, (int)(100.0 * s + 0.5)));
  };
  std::atomic<int> share{share_opt >= 0 ? share_opt : balanced_share(c_dev0, c_host0, c_hdr0)};
  double c_host = c_host0, c_dev = c_dev0, c_hdr = c_hdr0;
  std::mutex parse_mu;
  // `map`: image of the job -> file of the batch (identity unless files were dropped by the error isolation)
  struct Parsed { hc_heic_job* job = nullptr; std::string error; double seconds = 0; int share = 0; std::vector<int> map; };
  if (file_status) std::fill(file_status, file_status + nfiles, (int)HC_OK);
  std::string first_file_error;
  std::mutex file_error_mu;
  auto fail_file = [&](int file, int code, const std::string& why) {
    std::lock_guard<std::mutex> lk(file_error_mu);
    if (file_status[file] == HC_OK) { file_status[file] = code; st.files_failed++; }
    if (first_file_error.empty()) first_file_error = "file " + std::to_string(file) + ": " + why;
  };
  auto parse_batch = [&](int b) -> Parsed {
    Parsed p;
    const int first = b * files_per_batch, n = std::min(files_per_batch, nfiles - first);
    std::lock_guard<std::mutex> one_at_a_time(parse_mu);   // the look-ahead is two batches deep, the thread pool is one
    const auto t0 = clock::now();
    p.share = nbatches > 1 ? share.load() : 0;
    p.job = job_create(e, n, data + first, sizes + first, want_alpha, threads, 0, -1, p.share);
    p.map.resize(n);
    for (int k = 0; k < n; k++) p.map[k] = k;
    if (!p.job) p.error = hc_last_error();   // thread-local: fetch on the parsing thread
    if (!p.job && file_status) {
      // error isolation: find the files that cannot be decoded (each on its own, headers only unless the device parser
      // cannot take the picture), report them through file_status and go on with the others
      std::vector<const uint8_t*> gd; std::vector<size_t> gs;
      p.map.clear();
      for (int k = 0; k < n; k++) {
        hc_heic_job* probe = job_create(e, 1, data + first + k, sizes + first + k, want_alpha, 1, 0, -1, 0);
        if (probe) {
          hc_heic_job_destroy(probe);
          gd.push_back(data[first + k]); gs.push_back(sizes[first + k]); p.map.push_back(k);
        } else {
          fail_file(first + k, HC_ERR_BITSTREAM, hc_last_error());
        }
      }
      p.error.clear();
      if (!gd.empty() && (int)gd.size() < n) {
        p.share = 0;
        p.job = job_create(e, (int)gd.size(), gd.data(), gs.data(), want_alpha, threads, 0, -1, 0);
        if (!p.job) p.error = hc_last_error();
      } else if (!gd.empty()) {
        p.error = "batch failed although every file of it decodes alone";   // e.g. out of memory: not a property of one file
      }
    }
    p.seconds = secs(t0, clock::now());
    return p;
  };

  // stage 2 (this thread): submit — upload, [K0,] K1..K5 and the read-back into a pinned buffer are only ENQUEUED on the
  // batch's streams; stage 3 (this thread, depth-1 batches behind): deliver — wait for the stream, hand the images out,
  // release the batch. Three batches in flight keep two queued on the GPU behind the one that is about to be
  // delivered: K0 is a wavefront per picture, so the head and the tail of one batch's K0 leave most of the resident chain
  // slots idle (16 files: 22 CTB slots of time for 16.6 slots of work); with the next batch's K0 already queued on its own
  // low-priority stream, its chains take those slots, and K1..K5 + D2H of the finished batch run at high priority meanwhile.
  // The K0 kernels of the batches in flight share the GPU and finish together, so their read-backs come as a burst. When a
  // read-back is short against the period (one GPU on its own host link: 42 of 185 ms) three in flight is the best depth
  // (4.6 against 4.1-4.2 GP/s with four or six); when eight GPUs read back over one host link (200 ms per batch, the period
  // itself) the GPU idles through the burst unless another group of batches is parsing meanwhile: six in flight give 28.7
  // GP/s against 23.0 on the 8-GPU box. The depth therefore follows the measured read-back time (HEIFCUDA_STREAM_DEPTH fixes it).
  constexpr int MAX_DEPTH = 6;
  // fixed by the engine option "stream_depth" or HEIFCUDA_STREAM_DEPTH; otherwise automatic, starting from what the
  // engine's previous call ended with
  int depth_fixed = hc_engine_get_option(e, "stream_depth");
  if (const char* m = getenv("HEIFCUDA_STREAM_DEPTH")) {
    const int v = atoi(m);
    if (v > 0) depth_fixed = std::max(2, std::min(MAX_DEPTH, v));
  }
  const int depth_env = depth_fixed;       // 0: automatic
  const int learned = hc_engine_get_option(e, "stream_depth_learned");
  int depth = depth_env ? depth_env : (learned >= 2 && learned <= MAX_DEPTH ? learned : 3);
  struct InFlight { hc_heic_job* job = nullptr; int index = 0; int slot = -1; std::vector<size_t> offs; std::vector<uint8_t*> ptrs; std::vector<size_t> strides; std::vector<int> map; clock::time_point t0; double host_s = 0, host_wait_s = 0; int share = 0; int rc = HC_OK; };
  void* pinned[MAX_DEPTH] = {};
  size_t pinned_cap[MAX_DEPTH] = {};
  bool pinned_busy[MAX_DEPTH] = {};
  bool pin_failed = false, depth_locked = false;
  double last_period = 0;               // seconds between completions, smoothed (below)
  double best_d2h_ms = 0;               // shortest read-back among the last six batches
  double recent_d2h[6] = {0, 0, 0, 0, 0, 0};
  int n_d2h = 0;
  double t_done[5] = {0, 0, 0, 0, 0};   // host time at which the last five batches were seen complete
  int rc = HC_OK;
  std::string err;
  auto submit = [&](hc_heic_job* j, int b, InFlight& f) -> int {
    f.job = j; f.index = b; f.t0 = clock::now();
    f.slot = 0;
    for (int k = 0; k < MAX_DEPTH; k++)
      if (!pinned_busy[k]) { f.slot = k; break; }     // at most `depth` <= MAX_DEPTH batches are in flight
    pinned_busy[f.slot] = true;
    size_t need = 0;
    f.offs.resize(j->images.size());
    f.ptrs.assign(j->images.size(), nullptr);
    f.strides.assign(j->images.size(), 0);
    for (size_t i = 0; i < j->images.size(); i++) {
      const hc_image_desc& d = j->images[i].desc;
      const size_t row = (size_t)d.width * d.bytes_per_pixel;
      f.offs[i] = need;
      // external destination (the reference's heif_decoding_options::ext_dst, heif.h:1605-1615, pixelimage.cc:221-266): the
      // final pixels land in the caller's buffer with the caller's stride when it is large enough, else in our own memory
      const hc_stream_dest* xd = dests ? &dests[(size_t)b * files_per_batch + f.map[i]] : nullptr;
      const bool fits = d.out_format == HC_OUT_YCBCR
                            ? xd && xd->dst && (xd->stride == 0 || xd->stride == row) && xd->len >= image_bytes(d)   // packed planes
                            : xd && xd->dst && xd->stride >= row && xd->len >= xd->stride * (size_t)(d.height - 1) + row;
      if (fits) {
        f.ptrs[i] = (uint8_t*)xd->dst;
        f.strides[i] = d.out_format == HC_OUT_YCBCR ? row : xd->stride;
        continue;
      }
      f.strides[i] = row;
      need += (image_bytes(d) + 255) & ~(size_t)255;
    }
    if (need > pinned_cap[f.slot]) {
      if (pinned[f.slot]) hc_engine_give_out_pinned(e, pinned[f.slot], pinned_cap[f.slot]);
      pinned[f.slot] = hc_engine_take_out_pinned(e, need + need / 8, &pinned_cap[f.slot]);
      if (!pinned[f.slot]) {
        // the host cannot pin another output buffer: the caller falls back to a shallower pipeline (below)
        pinned_cap[f.slot] = 0;
        pinned_busy[f.slot] = false;
        f.slot = -1;
        pin_failed = true;
        return HC_ERR_MEMORY;
      }
    }
    const double ta = now_s();
    int r = (pinned[f.slot] || need == 0) ? hc_heic_job_upload(j) : HC_ERR_MEMORY;
    const double tb = now_s();
    if (r == HC_OK) r = hc_heic_job_run(j);
    if (r == HC_OK) hc_batch_mark_d2h(j->batch, 0);
    for (size_t i = 0; r == HC_OK && i < j->images.size(); i++) {
      if (!f.ptrs[i]) f.ptrs[i] = (uint8_t*)pinned[f.slot] + f.offs[i];
      r = hc_batch_read_rgb_async(j->batch, j->images[i].canvas, f.ptrs[i], f.strides[i]);
    }
    if (r == HC_OK) hc_batch_mark_d2h(j->batch, 1);
    if (trace_on()) fprintf(stderr, "[heifcuda] batch %d submit: pinned %.2f ms, upload %.2f ms, enqueue %.2f ms\n", b, (ta - std::chrono::duration<double>(f.t0.time_since_epoch()).count()) * 1e3, (tb - ta) * 1e3, (now_s() - tb) * 1e3);
    return r;
  };
  auto deliver = [&](InFlight& f, int r) {
    hc_heic_job* j = f.job;
    const double ta = now_s();
    if (r == HC_OK) r = hc_heic_job_sync(j);
    const double d2h_ms = r == HC_OK || r == HC_ERR_BITSTREAM ? (double)hc_batch_async_d2h_ms(j->batch) : 0.0;
    std::vector<char> bad(j->images.size(), 0);
    if (r == HC_ERR_BITSTREAM && file_status) {
      // slice data the device parser rejected: the pictures are known, the other files of the batch are intact
      const int* pics = nullptr;
      const int nbad = hc_batch_failed_pictures(j->batch, &pics);
      const std::string why = hc_last_error();
      for (int q = 0; q < nbad; q++) {
        const int file = pics[q] < (int)j->pic_file.size() ? j->pic_file[pics[q]] : -1;
        if (file < 0) continue;
        bad[file] = 1;
        fail_file(f.index * files_per_batch + f.map[file], HC_ERR_BITSTREAM, why);
      }
      if (nbad > 0) r = HC_OK;
    }
    const double tb = now_s();
    double tc = tb;
    if (r == HC_OK) {
      float ms[8];
      if (hc_heic_job_stage_ms(j, ms) == HC_OK) {
        if (trace_on()) {
          float tl[5];
          if (hc_batch_timeline_ms(j->batch, tl) == HC_OK)
            fprintf(stderr, "[heifcuda] batch %d timeline (ms on the GPU clock): upload %.1f, K0 %.1f .. %.1f, K1 %.1f .. K4 end %.1f\n", f.index, tl[0], tl[1], tl[2], tl[3], tl[4]);
        }
        const double gpu_ms = ms[1] + ms[2] + ms[3] + ms[4] + ms[5] + ms[7];
        st.device_ms += gpu_ms;
        for (int q = 0; q < 4; q++) t_done[q] = t_done[q + 1];
        t_done[4] = tb;
        // overlapping batches finish in pairs or triplets (60 ms, 250 ms, 60 ms, ...): the period between completions is taken
        // over four of them when there are that many, else over two
        if (t_done[2] > 0) last_period = t_done[0] > 0 ? (t_done[4] - t_done[0]) / 4 : (t_done[4] - t_done[2]) / 2;
        if (share_opt < 0 && f.index > 3 && f.host_s > 0 && t_done[2] > 0) {
          // Cost per coded item on either side, smoothed; the balanced share is c_dev / (c_host + c_dev). The K0 kernels of
          // consecutive batches overlap, so a batch's own event times say little; what the device costs per item is the
          // pipeline period (completion to completion, averaged over two batches because overlapping batches tend to finish
          // in pairs) — but only while the GPU is what the pipeline waits for, i.e. this thread did not have to wait for the
          // host parse of the batch.
          const double n_items = (double)j->items.size();
          const double n_host = n_items * f.share / 100.0, n_dev = std::max(1.0, n_items - n_host);
          const double period = last_period, cd = period / n_dev;
          // slow, outlier-resistant tracking: one noisy batch (a host thread descheduled) must not swing the share
          if (n_host < 1.0) c_hdr = 0.5 * c_hdr + 0.5 * std::min(f.host_s / n_items, 2.0 * c_hdr);
          else c_host = 0.5 * c_host + 0.5 * std::min(std::max(0.0, f.host_s - n_items * c_hdr) / n_host, 2.0 * c_host);
          const bool gpu_bound = f.host_wait_s < 0.05 * period;
          if (gpu_bound) c_dev = 0.5 * c_dev + 0.5 * std::min(cd, 2.0 * c_dev);
          share.store(balanced_share(c_dev, c_host, c_hdr));
          if (trace_on()) fprintf(stderr, "[heifcuda] batch %d: host %.1f ms (waited %.1f ms for it), period %.1f ms, own gpu events %.1f ms, share %d%% -> %d%%\n", f.index, f.host_s * 1e3, f.host_wait_s * 1e3, period * 1e3, gpu_ms, f.share, share.load());
        }
      }
      st.bytes_h2d += hc_heic_job_upload_bytes(j);
      st.launches += hc_heic_job_launch_count(j);
      for (size_t i = 0; i < j->images.size(); i++) {
        if (bad[i]) continue;
        const hc_image_desc& d = j->images[i].desc;
        st.bytes_d2h += image_bytes(d);
        st.pixels += (int64_t)d.width * d.height;
        if (on_image) on_image(user, f.index * files_per_batch + f.map[i], &d, f.ptrs[i], f.strides[i]);
      }
      tc = now_s();
    } else if (rc == HC_OK) {
      rc = r;
      err = hc_last_error();
    }
    hc_heic_job_destroy(j);
    if (trace_on()) fprintf(stderr, "[heifcuda] batch %d deliver: wait %.2f ms, callbacks %.2f ms, destroy %.2f ms\n", f.index, (tb - ta) * 1e3, (tc - tb) * 1e3, (now_s() - tc) * 1e3);
    st.seconds_gpu_phase += secs(f.t0, clock::now());
    st.batches++;
    f.job = nullptr;
    if (f.slot >= 0) pinned_busy[f.slot] = false;
    // depth of the pipeline: follows how long a batch's read-back takes against the period (see above)
    // (the shortest read-back among the last six batches counts: the others queued behind the copies of the batches that
    // finished with them; a window, not the minimum of the whole call, so that one copy that met an idle link ages out)
    if (d2h_ms > 0) {
      recent_d2h[n_d2h++ % 6] = d2h_ms;
      best_d2h_ms = recent_d2h[0];
      for (int q = 1; q < std::min(n_d2h, 6); q++) best_d2h_ms = std::min(best_d2h_ms, recent_d2h[q]);
    }
    if (!depth_env && !depth_locked && n_d2h >= 3 && best_d2h_ms > 0 && last_period > 0) {
      const double ratio = best_d2h_ms * 1e-3 / last_period;
      const int before = depth;
      if (ratio > 0.4) depth = MAX_DEPTH;
      else if (ratio < 0.3) depth = 3;
      if (trace_on() && (depth != before || f.index == 6)) fprintf(stderr, "[heifcuda] batch %d: read-back %.1f ms of a %.1f ms period: %d batches in flight from now on\n", f.index, best_d2h_ms, last_period * 1e3, depth);
    }
    st.depth = depth;
  };

  std::deque<InFlight> flight;   // submitted, not yet delivered, in submission order
  // the host side runs up to two batches ahead of the submit stage: completions of overlapping batches come in bursts,
  // and a single batch of look-ahead left this thread waiting for the parser right after every burst
  constexpr int PARSE_AHEAD = 2;
  std::deque<std::future<Parsed>> ahead;
  int next_parse = 0;
  auto top_up = [&]() {
    while ((int)ahead.size() < PARSE_AHEAD && next_parse < nbatches) ahead.push_back(std::async(std::launch::async, parse_batch, next_parse++));
  };
  top_up();
  for (int b = 0; b < nbatches; b++) {
    const auto tw = clock::now();
    Parsed cur = ahead.front().get();
    ahead.pop_front();
    const double host_wait = secs(tw, clock::now());
    top_up();
    st.seconds_parse += cur.seconds;
    if (!cur.job) {
      if (rc == HC_OK && !cur.error.empty()) { rc = HC_ERR_BITSTREAM; err = "batch " + std::to_string(b) + ": " + cur.error; }
      continue;   // keep draining the pipeline (with error isolation: every file of the batch failed and is reported)
    }
    if (rc != HC_OK) { hc_heic_job_destroy(cur.job); continue; }
    while ((int)flight.size() >= depth) { deliver(flight.front(), flight.front().rc); flight.pop_front(); }   // room for this one
    flight.emplace_back();
    InFlight& f = flight.back();
    f.host_s = cur.seconds;
    f.map = cur.map;
    f.host_wait_s = host_wait;
    f.share = cur.share;
    f.rc = submit(cur.job, b, f);
    while (flight.back().rc == HC_ERR_MEMORY && pin_failed && flight.size() > 1) {     // (`f` is not used below: the deque moves)
      // no pinned memory for a buffer of its own: deliver the oldest batch, take over its buffer, and stay this shallow
      pin_failed = false;
      InFlight mine = std::move(flight.back());
      flight.pop_back();
      deliver(flight.front(), flight.front().rc);
      flight.pop_front();
      depth = std::max(2, (int)flight.size() + 1);
      depth_locked = true;
      flight.push_back(std::move(mine));
      InFlight& again = flight.back();
      again.rc = submit(cur.job, b, again);
    }
    while ((int)flight.size() > depth - 1) { deliver(flight.front(), flight.front().rc); flight.pop_front(); }   // depth - 1 stay queued
  }
  while (!flight.empty()) { deliver(flight.front(), flight.front().rc); flight.pop_front(); }   // drain in submission order
  for (int k = 0; k < MAX_DEPTH; k++)
    if (pinned[k]) hc_engine_give_out_pinned(e, pinned[k], pinned_cap[k]);     // kept by the engine for the next call
  if (!depth_env) hc_engine_set_option(e, "stream_depth_learned", depth);
  st.seconds_total = secs(t_begin, clock::now());
  if (stats) *stats = st;
  if (rc != HC_OK) hc::set_last_error(err);
  else if (!first_file_error.empty()) hc::set_last_error(first_file_error);
  return rc;
}

}  // extern "C"
