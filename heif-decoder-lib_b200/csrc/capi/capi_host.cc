// capi_host.cc — C ABI over the host front-end (include/heifcuda.h, section "host front-end").
#include <algorithm>
#include "capi_internal.h"
#include "../host/k0_host.h"
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

namespace {
thread_local std::string g_last_error;
}

namespace hc {
void set_last_error(const std::string& s) { g_last_error = s; }
}  // namespace hc


extern "C" {

const char* hc_last_error(void) { return g_last_error.c_str(); }

hc_parser* hc_parser_new(void) { return new (std::nothrow) hc_parser; }
void hc_parser_free(hc_parser* p) { delete p; }

int hc_parser_push(hc_parser* p, const uint8_t* data, size_t size, int stream_format) {
  if (!p || (!data && size)) {
    g_last_error = "hc_parser_push: null argument";
    return HC_ERR_ARGUMENT;
  }
  std::string e;
  try {
    switch (stream_format) {
      case HC_STREAM_LENGTH_PREFIXED: e = p->parser.push_length_prefixed(data, size); break;
      case HC_STREAM_ANNEXB: e = p->parser.push_annexb(data, size); break;
      case HC_STREAM_SINGLE_NAL: e = p->parser.push_nal(data, size); break;
      default: g_last_error = "hc_parser_push: unknown stream format"; return HC_ERR_ARGUMENT;
    }
  } catch (const std::bad_alloc&) {
    g_last_error = "out of memory while parsing";
    return HC_ERR_MEMORY;
  }
  if (!e.empty()) {
    g_last_error = e;
    return HC_ERR_BITSTREAM;
  }
  return HC_OK;
}

hc_records* hc_parser_take_picture(hc_parser* p) {
  if (!p) {
    g_last_error = "hc_parser_take_picture: null parser";
    return nullptr;
  }
  std::string e;
  std::unique_ptr<hc::PictureRecords> rec = p->parser.take_picture(&e);
  if (!rec) {
    g_last_error = e;
    return nullptr;
  }
  hc_records* r = new (std::nothrow) hc_records;
  if (!r) {
    g_last_error = "out of memory";
    return nullptr;
  }
  r->rec = std::move(rec);
  return r;
}

void hc_records_free(hc_records* r) { delete r; }
const hc_pic* hc_records_pic(const hc_records* r) { return &r->rec->pic; }
const hc_ctu* hc_records_ctus(const hc_records* r, size_t* n) { if (n) *n = r->rec->ctus.size(); return r->rec->ctus.data(); }
const hc_blk* hc_records_blks(const hc_records* r, size_t* n) { if (n) *n = r->rec->blks.size(); return r->rec->blks.data(); }
const hc_tb* hc_records_tbs(const hc_records* r, size_t* n) { if (n) *n = r->rec->tbs.size(); return r->rec->tbs.data(); }
const hc_coeff* hc_records_coeffs(const hc_records* r, size_t* n) { if (n) *n = r->rec->coeffs.size(); return r->rec->coeffs.data(); }
const uint8_t* hc_records_edge_map(const hc_records* r, size_t* n) { if (n) *n = r->rec->edge_map.size(); return r->rec->edge_map.data(); }
const int8_t* hc_records_qp_map(const hc_records* r, size_t* n) { if (n) *n = r->rec->qp_map.size(); return r->rec->qp_map.data(); }
const uint8_t* hc_records_scaling(const hc_records* r, size_t* n) {
  if (n) *n = r->rec->scaling.size();
  return r->rec->scaling.empty() ? nullptr : r->rec->scaling.data();
}
size_t hc_records_upload_bytes(const hc_records* r) {
  const hc::PictureRecords& p = *r->rec;
  return sizeof(hc_pic) + p.ctus.size() * sizeof(hc_ctu) + p.blks.size() * sizeof(hc_blk) +
         p.tbs.size() * sizeof(hc_tb) + p.coeffs.size() * sizeof(hc_coeff) + p.edge_map.size() + p.qp_map.size() +
         p.scaling.size();
}

hc_records* hc_parse_picture(const uint8_t* data, size_t size, int stream_format) {
  hc_parser p;
  if (hc_parser_push(&p, data, size, stream_format) != HC_OK) return nullptr;
  return hc_parser_take_picture(&p);
}

hc_heif* hc_heif_open(const uint8_t* data, size_t size) {
  if (!data) { g_last_error = "hc_heif_open: null data"; return nullptr; }
  hc_heif* f = new (std::nothrow) hc_heif;
  if (!f) { g_last_error = "out of memory"; return nullptr; }
  std::string e = f->file.parse(data, size);
  if (!e.empty()) { g_last_error = e; delete f; return nullptr; }
  return f;
}
void hc_heif_close(hc_heif* f) { delete f; }
uint32_t hc_heif_primary_id(const hc_heif* f) { return f->file.primary_id(); }
int hc_heif_top_level_ids(const hc_heif* f, uint32_t* ids, int max) {
  std::vector<uint32_t> v = f->file.top_level_images();
  for (int i = 0; i < (int)v.size() && i < max; i++) ids[i] = v[i];
  return (int)v.size();
}
int hc_heif_get_overlay(const hc_heif* f, uint32_t id, hc_heif_overlay_info* info) {
  if (!f || !info || !f->file.is_overlay(id)) { g_last_error = "hc_heif_get_overlay: not an overlay item"; return HC_ERR_ARGUMENT; }
  hc::HeifOverlay o;
  std::string e = f->file.overlay(id, o);
  if (!e.empty()) { g_last_error = e; return HC_ERR_BITSTREAM; }
  if (o.children.size() > HC_OVERLAY_MAX_CHILDREN || o.children.size() != o.offsets.size()) { g_last_error = "overlay: too many or mismatched references"; return HC_ERR_UNSUPPORTED; }
  memset(info, 0, sizeof(*info));
  info->canvas_w = o.canvas_w; info->canvas_h = o.canvas_h;
  for (int k = 0; k < 4; k++) info->background[k] = o.background[k];
  info->n = (int32_t)o.children.size();
  for (int k = 0; k < info->n; k++) { info->children[k] = o.children[k]; info->dx[k] = o.offsets[k].first; info->dy[k] = o.offsets[k].second; }
  return HC_OK;
}

int hc_heif_get_image_info(const hc_heif* f, uint32_t id, hc_heif_image_info* info) {
  const hc::HeifItem* it = f->file.item(id);
  if (!it || !info) { g_last_error = "hc_heif_get_image_info: no such item"; return HC_ERR_ARGUMENT; }
  memset(info, 0, sizeof(*info));
  info->id = id;
  info->rows = info->cols = 1;
  info->width = it->ispe_w;
  info->height = it->ispe_h;
  if (f->file.is_grid(id)) {
    hc::HeifGrid g;
    std::string e = f->file.grid(id, g);
    if (!e.empty()) { g_last_error = e; return HC_ERR_BITSTREAM; }
    info->is_grid = 1;
    info->rows = g.rows;
    info->cols = g.cols;
    info->width = g.out_w;
    info->height = g.out_h;
  }
  info->alpha_id = f->file.alpha_item(id);
  info->premultiplied_alpha = f->file.premultiplied(id) ? 1 : 0;
  info->rot = it->rot;
  info->mirror = it->mirror;
  info->n_transforms = (int32_t)std::min<size_t>(it->xforms.size(), 8);
  for (int k = 0; k < info->n_transforms; k++) info->transforms[k] = it->xforms[k];
  info->has_clap = (int32_t)std::min<size_t>(it->claps.size(), 4);
  for (int k = 0; k < info->has_clap; k++) {
    const hc::HeifItem::Clap& cl = it->claps[k];
    const uint32_t v[8] = {cl.w_num, cl.w_den, cl.h_num, cl.h_den, (uint32_t)cl.hoff_num, cl.hoff_den, (uint32_t)cl.voff_num, cl.voff_den};
    for (int q = 0; q < 8; q++) info->claps[k][q] = v[q];
  }
  info->nclx_present = it->nclx.present;
  info->primaries = it->nclx.primaries;
  info->transfer = it->nclx.transfer;
  info->matrix = it->nclx.matrix;
  info->full_range = it->nclx.full_range;
  return HC_OK;
}
int hc_heif_grid_tiles(const hc_heif* f, uint32_t id, uint32_t* tiles, int max) {
  hc::HeifGrid g;
  std::string e = f->file.grid(id, g);
  if (!e.empty()) { g_last_error = e; return HC_ERR_BITSTREAM; }
  for (int i = 0; i < (int)g.tiles.size() && i < max; i++) tiles[i] = g.tiles[i];
  return (int)g.tiles.size();
}
int hc_heif_thumbnail_ids(const hc_heif* f, uint32_t id, uint32_t* ids, int max) {
  std::vector<uint32_t> v = f->file.thumbnails(id);
  for (int i = 0; i < (int)v.size() && i < max; i++) ids[i] = v[i];
  return (int)v.size();
}
int hc_heif_auxiliary_ids(const hc_heif* f, uint32_t id, int include_alpha, uint32_t* ids, int max) {
  std::vector<uint32_t> v = f->file.auxiliaries(id, include_alpha != 0);
  for (int i = 0; i < (int)v.size() && i < max; i++) ids[i] = v[i];
  return (int)v.size();
}
int hc_heif_aux_type(const hc_heif* f, uint32_t id, char* buf, size_t len) {
  const hc::HeifItem* it = f ? f->file.item(id) : nullptr;
  if (!it || it->aux_type.empty()) { g_last_error = "hc_heif_aux_type: item " + std::to_string(id) + " has no auxC property"; return HC_ERR_ARGUMENT; }
  if (buf && len) {
    const size_t n = std::min(len - 1, it->aux_type.size());
    memcpy(buf, it->aux_type.data(), n);
    buf[n] = 0;
  }
  return (int)it->aux_type.size();
}
int hc_heif_coded_stream(const hc_heif* f, uint32_t id, uint8_t** out, size_t* size) {
  std::vector<uint8_t> v;
  std::string e = f->file.coded_stream(id, v);
  if (!e.empty()) { g_last_error = e; return HC_ERR_BITSTREAM; }
  uint8_t* p = (uint8_t*)malloc(v.size() ? v.size() : 1);
  if (!p) { g_last_error = "out of memory"; return HC_ERR_MEMORY; }
  memcpy(p, v.data(), v.size());
  *out = p;
  *size = v.size();
  return HC_OK;
}
void hc_free(void* p) { free(p); }

}  // extern "C"

extern "C" {

hc_k0_picture* hc_k0_prepare(const uint8_t* data, size_t size, int stream_format) {
  if (!data || !size) { g_last_error = "hc_k0_prepare: null argument"; return nullptr; }
  try {
    std::unique_ptr<hc_k0_picture> k(new hc_k0_picture);
    std::string e = hc::k0_prepare(data, size, stream_format, k->hp);
    if (!e.empty()) { g_last_error = e; return nullptr; }
    return k.release();
  } catch (const std::bad_alloc&) {
    g_last_error = "out of memory";
    return nullptr;
  }
}
void hc_k0_free(hc_k0_picture* k) { delete k; }
int hc_k0_eligible(const hc_k0_picture* k) { return k && k->hp.eligible; }
const char* hc_k0_why_not(const hc_k0_picture* k) { return k ? k->hp.why_not.c_str() : ""; }
const hc_pic* hc_k0_pic(const hc_k0_picture* k) { return k ? &k->hp.hpic : nullptr; }
size_t hc_k0_upload_bytes(const hc_k0_picture* k) {
  return k ? k->hp.bytes.size() + k->hp.slices.size() * sizeof(hc::k0::Slice) + k->hp.ctb_slice.size() * 8 + k->hp.subs.size() * sizeof(hc::k0::Sub) : 0;
}

// Test scaffold: parses one picture with the K0 core (the device CABAC parser, kernels/k0_core.cuh) executed
// on the CPU and returns its records in the host parser's form. NULL when the picture is not eligible for K0
// (hc_last_error starts with "not eligible") or malformed.
hc_records* hc_parse_picture_k0(const uint8_t* data, size_t size, int stream_format) {
  hc::K0HostPicture hp;
  std::string e;
  try {
    e = hc::k0_prepare(data, size, stream_format, hp);
    if (e.empty() && !hp.eligible) e = "not eligible for K0: " + hp.why_not;
    if (!e.empty()) { g_last_error = e; return nullptr; }
    std::unique_ptr<hc::PictureRecords> rec = hc::k0_parse_on_cpu(hp, &e);
    if (!rec) { g_last_error = e; return nullptr; }
    hc_records* r = new hc_records;
    r->rec = std::move(rec);
    return r;
  } catch (const std::bad_alloc&) {
    g_last_error = "out of memory";
    return nullptr;
  }
}

size_t hc_image_plane_layout(const hc_image_desc* d, size_t offset[4], size_t stride[4], int32_t width[4], int32_t height[4]) {
  if (!d || d->out_format != HC_OUT_YCBCR || d->width <= 0 || d->height <= 0 || d->chroma_format < 0 || d->chroma_format > 3 ||
      d->bit_depth < 8 || d->bit_depth > 16)
    return 0;
  const size_t ps = d->bit_depth == 8 ? 1 : 2;
  size_t total = 0;
  for (int k = 0; k < 4; k++) {
    const bool present = k == 3 ? d->has_alpha != 0 : hc::plane_w(d->width, d->chroma_format, k) > 0;
    const int w = present ? hc::plane_w(d->width, d->chroma_format, k) : 0, h = present ? hc::plane_h(d->height, d->chroma_format, k) : 0;
    if (offset) offset[k] = total;
    if (stride) stride[k] = (size_t)w * ps;
    if (width) width[k] = w;
    if (height) height[k] = h;
    total += (size_t)w * ps * h;
  }
  return total;
}

}  // extern "C"
