// heif_reader.cc — see heif_reader.h.
#include "heif_reader.h"
#include <algorithm>
#include <cstring>

namespace hc {

namespace {

constexpr uint32_t fourcc(const char* s) {
  return ((uint32_t)(uint8_t)s[0] << 24) | ((uint32_t)(uint8_t)s[1] << 16) | ((uint32_t)(uint8_t)s[2] << 8) |
         (uint32_t)(uint8_t)s[3];
}

struct Cursor {
  const uint8_t* p;
  size_t n, pos = 0;
  bool bad = false;
  Cursor(const uint8_t* d, size_t s) : p(d), n(s) {}
  size_t left() const { return n > pos ? n - pos : 0; }
  uint64_t be(int bytes) {
    if (left() < (size_t)bytes) { bad = true; pos = n; return 0; }
    uint64_t v = 0;
    for (int i = 0; i < bytes; i++) v = (v << 8) | p[pos++];
    return v;
  }
  uint32_t u8() { return (uint32_t)be(1); }
  uint32_t u16() { return (uint32_t)be(2); }
  uint32_t u32() { return (uint32_t)be(4); }
  void skip(size_t k) { if (left() < k) { bad = true; pos = n; } else pos += k; }
  std::string cstr() {
    std::string s;
    while (pos < n && p[pos]) s.push_back((char)p[pos++]);
    if (pos < n) pos++; else bad = true;
    return s;
  }
};

struct Box {
  uint32_t type = 0;
  const uint8_t* body = nullptr;
  size_t size = 0;
};

// reads the next box header at c; returns false at the end or on a malformed header
bool next_box(Cursor& c, Box& b) {
  if (c.left() < 8) return false;
  uint64_t sz = c.u32();
  b.type = c.u32();
  size_t hdr = 8;
  if (sz == 1) { sz = c.be(8); hdr = 16; }
  else if (sz == 0) sz = c.left() + hdr;
  if (b.type == fourcc("uuid")) { c.skip(16); hdr += 16; }
  if (c.bad || sz < hdr || sz - hdr > c.left()) { c.bad = true; return false; }
  b.body = c.p + c.pos;
  b.size = (size_t)(sz - hdr);
  c.pos += b.size;
  return true;
}

// the auxC types that make an auxiliary image an alpha image
bool is_alpha_urn(const std::string& urn) {
  return urn == "urn:mpeg:avc:2015:auxid:1" || urn == "urn:mpeg:hevc:2015:auxid:1" || urn == "urn:mpeg:mpegB:cicp:systems:auxiliary:alpha";
}

}  // namespace

const HeifItem* HeifFile::item(uint32_t id) const {
  auto it = items_.find(id);
  return it == items_.end() ? nullptr : &it->second;
}

std::string HeifFile::parse(const uint8_t* data, size_t size) {
  data_ = data;
  size_ = size;
  items_.clear();
  hvcc_.clear();
  refs_.clear();
  primary_ = 0;
  idat_ = nullptr;
  idat_size_ = 0;

  Cursor top(data, size);
  Box b;
  bool have_ftyp = false, have_meta = false;
  Box meta;
  while (next_box(top, b)) {
    if (b.type == fourcc("ftyp")) have_ftyp = true;
    else if (b.type == fourcc("meta") && !have_meta) { meta = b; have_meta = true; }
  }
  if (!have_ftyp) return "not a HEIF file: no ftyp box";
  if (!have_meta) return "HEIF file without a meta box";

  Cursor m(meta.body, meta.size);
  m.skip(4);  // FullBox version/flags
  struct Prop { uint32_t type; const uint8_t* body; size_t size; };
  std::vector<Prop> props;
  struct Assoc { uint32_t item; std::vector<int> idx; };
  std::vector<Assoc> assocs;
  struct Loc { uint32_t id; int cm; uint64_t base; std::vector<HeifItem::Extent> ext; };
  std::vector<Loc> locs;

  while (next_box(m, b)) {
    Cursor c(b.body, b.size);
    if (b.type == fourcc("pitm")) {
      uint32_t vf = c.u32();
      primary_ = (vf >> 24) == 0 ? c.u16() : c.u32();
    } else if (b.type == fourcc("idat")) {
      idat_ = b.body;
      idat_size_ = b.size;
    } else if (b.type == fourcc("iinf")) {
      uint32_t vf = c.u32();
      uint32_t n = (vf >> 24) == 0 ? c.u16() : c.u32();
      Box e;
      for (uint32_t i = 0; i < n && next_box(c, e); i++) {
        if (e.type != fourcc("infe")) continue;
        Cursor ec(e.body, e.size);
        uint32_t evf = ec.u32();
        int ver = (int)(evf >> 24);
        if (ver < 2) continue;
        HeifItem it;
        it.id = ver == 2 ? ec.u16() : ec.u32();
        ec.u16();
        it.type = ec.u32();
        it.hidden = (evf & 1) != 0;
        if (!ec.bad) items_[it.id] = it;
      }
    } else if (b.type == fourcc("iloc")) {
      uint32_t vf = c.u32();
      int ver = (int)(vf >> 24);
      uint32_t a = c.u8(), bb = c.u8();
      int offset_size = (int)(a >> 4), length_size = (int)(a & 15), base_size = (int)(bb >> 4), index_size = (int)(bb & 15);
      if (ver == 0) index_size = 0;
      uint32_t n = ver < 2 ? c.u16() : c.u32();
      for (uint32_t i = 0; i < n && !c.bad; i++) {
        Loc l;
        l.id = ver < 2 ? c.u16() : c.u32();
        l.cm = 0;
        if (ver == 1 || ver == 2) l.cm = (int)(c.u16() & 15);
        c.u16();  // data_reference_index
        l.base = c.be(base_size);
        uint32_t ne = c.u16();
        for (uint32_t k = 0; k < ne && !c.bad; k++) {
          if ((ver == 1 || ver == 2) && index_size > 0) c.be(index_size);
          HeifItem::Extent e;
          e.offset = c.be(offset_size);
          e.length = c.be(length_size);
          l.ext.push_back(e);
        }
        locs.push_back(l);
      }
      if (c.bad) return "malformed iloc box";
    } else if (b.type == fourcc("iref")) {
      uint32_t vf = c.u32();
      int ver = (int)(vf >> 24);
      Box e;
      while (next_box(c, e)) {
        Cursor rc(e.body, e.size);
        Ref r;
        r.type = e.type;
        r.from = ver == 0 ? rc.u16() : rc.u32();
        uint32_t cnt = rc.u16();
        for (uint32_t i = 0; i < cnt && !rc.bad; i++) r.to.push_back(ver == 0 ? rc.u16() : rc.u32());
        if (!rc.bad) refs_.push_back(r);
      }
    } else if (b.type == fourcc("iprp")) {
      Box e;
      while (next_box(c, e)) {
        if (e.type == fourcc("ipco")) {
          Cursor pc(e.body, e.size);
          Box pb;
          while (next_box(pc, pb)) props.push_back({pb.type, pb.body, pb.size});
        } else if (e.type == fourcc("ipma")) {
          Cursor ac(e.body, e.size);
          uint32_t vf = ac.u32();
          int ver = (int)(vf >> 24);
          uint32_t n = ac.u32();
          for (uint32_t i = 0; i < n && !ac.bad; i++) {
            Assoc as;
            as.item = ver < 1 ? ac.u16() : ac.u32();
            uint32_t cnt = ac.u8();
            for (uint32_t k = 0; k < cnt; k++) {
              uint32_t v = (vf & 1) ? (ac.u16() & 0x7FFF) : (ac.u8() & 0x7F);
              as.idx.push_back((int)v);
            }
            assocs.push_back(as);
          }
        }
      }
    }
  }
  if (m.bad) return "malformed meta box";

  for (auto& l : locs) {
    auto it = items_.find(l.id);
    if (it == items_.end()) continue;
    it->second.construction_method = l.cm;
    it->second.base_offset = l.base;
    it->second.extents = l.ext;
  }
  // resolve properties
  std::map<int, int> hvcc_of_prop;
  for (auto& as : assocs) {
    auto it = items_.find(as.item);
    if (it == items_.end()) continue;
    HeifItem& item = it->second;
    for (int idx : as.idx) {
      if (idx < 1 || idx > (int)props.size()) continue;
      item.props.push_back(idx);
      const Prop& p = props[idx - 1];
      Cursor c(p.body, p.size);
      if (p.type == fourcc("ispe")) {
        c.u32();
        item.ispe_w = (int)c.u32();
        item.ispe_h = (int)c.u32();
      } else if (p.type == fourcc("hvcC")) {
        auto f = hvcc_of_prop.find(idx);
        if (f != hvcc_of_prop.end()) { item.hvcc_prop = f->second; continue; }
        HeifHvcC h;
        c.skip(21);
        h.length_size = (int)(c.u8() & 3) + 1;
        uint32_t narr = c.u8();
        for (uint32_t a = 0; a < narr && !c.bad; a++) {
          c.u8();
          uint32_t nn = c.u16();
          for (uint32_t k = 0; k < nn && !c.bad; k++) {
            uint32_t len = c.u16();
            if (c.left() < len) { c.bad = true; break; }
            h.nals.emplace_back(c.p + c.pos, c.p + c.pos + len);
            c.skip(len);
          }
        }
        if (c.bad) return "malformed hvcC box";
        hvcc_.push_back(std::move(h));
        hvcc_of_prop[idx] = (int)hvcc_.size() - 1;
        item.hvcc_prop = (int)hvcc_.size() - 1;
      } else if (p.type == fourcc("colr")) {
        uint32_t ct = c.u32();
        if (ct == fourcc("nclx") && !item.nclx.present) {
          item.nclx.present = true;
          item.nclx.primaries = (int)c.u16();
          item.nclx.transfer = (int)c.u16();
          item.nclx.matrix = (int)c.u16();
          item.nclx.full_range = (int)(c.u8() >> 7);
        }
      } else if (p.type == fourcc("irot")) {
        item.rot = (int)(c.u8() & 3);
        if (item.rot) item.xforms.push_back((uint8_t)item.rot);
      } else if (p.type == fourcc("imir")) {
        item.mirror = (int)(c.u8() & 1);
        item.xforms.push_back((uint8_t)(item.mirror ? 4 : 5));   // box.cc:3626-3636: axis & 1 -> "horizontal"
      } else if (p.type == fourcc("clap")) {
        item.has_clap = true;
        HeifItem::Clap cl;
        cl.w_num = c.u32(); cl.w_den = c.u32(); cl.h_num = c.u32(); cl.h_den = c.u32();
        cl.hoff_num = (int32_t)c.u32(); cl.hoff_den = c.u32(); cl.voff_num = (int32_t)c.u32(); cl.voff_den = c.u32();
        if (c.bad) return "malformed clap box";
        item.claps.push_back(cl);
        item.xforms.push_back(6);
      } else if (p.type == fourcc("auxC")) {
        c.u32();
        item.aux_type = c.cstr();
      } else if (p.type == fourcc("pixi")) {
        c.u32();
        uint32_t nch = c.u8();
        if (nch) item.pixi_bits = (int)c.u8();
      }
    }
  }
  if (!primary_ || !items_.count(primary_)) {
    // fall back to the first image item like a tolerant reader would
    for (auto& kv : items_)
      if (kv.second.type == fourcc("hvc1") || kv.second.type == fourcc("grid")) { primary_ = kv.first; break; }
    if (!primary_) return "HEIF file has no image item";
  }
  return "";
}

std::vector<uint32_t> HeifFile::top_level_images() const {
  std::vector<uint32_t> out;
  for (auto& kv : items_) {
    const HeifItem& it = kv.second;
    if (it.type != fourcc("hvc1") && it.type != fourcc("grid")) continue;
    if (it.hidden) continue;
    bool sub = false;
    for (auto& r : refs_)
      if (r.from == it.id && (r.type == fourcc("thmb") || r.type == fourcc("auxl"))) sub = true;
    if (!sub) out.push_back(it.id);
  }
  return out;
}

bool HeifFile::is_grid(uint32_t id) const {
  const HeifItem* it = item(id);
  return it && it->type == fourcc("grid");
}

std::string HeifFile::read_item_data(const HeifItem& it, std::vector<uint8_t>& out) const {
  const uint8_t* base = it.construction_method == 1 ? idat_ : data_;
  size_t bsize = it.construction_method == 1 ? idat_size_ : size_;
  if (it.construction_method > 1) return "iloc construction method 2 is not supported";
  if (!base) return "item data refers to a missing idat box";
  for (auto& e : it.extents) {
    uint64_t off = it.base_offset + e.offset;
    uint64_t len = e.length;
    if (len == 0 && it.extents.size() == 1) len = bsize > off ? bsize - off : 0;  // "to the end"
    if (off > bsize || len > bsize - off) return "item extent outside the file";
    out.insert(out.end(), base + off, base + off + len);
  }
  return "";
}

std::string HeifFile::grid(uint32_t id, HeifGrid& g) const {
  const HeifItem* it = item(id);
  if (!it || it->type != fourcc("grid")) return "item is not a grid";
  std::vector<uint8_t> d;
  std::string e = read_item_data(*it, d);
  if (!e.empty()) return e;
  if (d.size() < 8) return "grid item payload too short";   // context.cc:172-221
  int flags = d[1];
  g.rows = d[2] + 1;
  g.cols = d[3] + 1;
  if (flags & 1) {
    if (d.size() < 12) return "grid item payload too short";
    g.out_w = (int)(((uint32_t)d[4] << 24) | (d[5] << 16) | (d[6] << 8) | d[7]);
    g.out_h = (int)(((uint32_t)d[8] << 24) | (d[9] << 16) | (d[10] << 8) | d[11]);
  } else {
    g.out_w = (d[4] << 8) | d[5];
    g.out_h = (d[6] << 8) | d[7];
  }
  g.tiles.clear();
  for (auto& r : refs_)
    if (r.from == id && r.type == fourcc("dimg")) g.tiles = r.to;
  if ((int)g.tiles.size() != g.rows * g.cols) return "grid: number of tile references does not match rows*cols";
  if (g.out_w <= 0 || g.out_h <= 0) return "grid: empty output size";
  return "";
}

bool HeifFile::is_overlay(uint32_t id) const {
  const HeifItem* it = item(id);
  return it && it->type == fourcc("iovl");
}

std::string HeifFile::overlay(uint32_t id, HeifOverlay& o) const {
  const HeifItem* it = item(id);
  if (!it || it->type != fourcc("iovl")) return "not an overlay item";
  std::vector<uint8_t> d;
  std::string e = read_item_data(*it, d);
  if (!e.empty()) return e;
  o = HeifOverlay();
  for (auto& r : refs_)
    if (r.from == id && r.type == fourcc("dimg")) o.children = r.to;
  if (d.size() < 2 + 4 * 2) return "Overlay image data incomplete";
  if (d[0] != 0) return "Overlay image data version " + std::to_string((int)d[0]) + " is not implemented yet";
  const size_t fl = (d[1] & 1) ? 4 : 2;
  if (2 + 4 * 2 + 2 * fl + o.children.size() * 2 * fl > d.size()) return "Overlay image data incomplete";
  size_t p = 2;
  auto rd = [&](size_t n) { uint32_t v = 0; for (size_t k = 0; k < n; k++) v = (v << 8) | d[p++]; return v; };
  for (int k = 0; k < 4; k++) o.background[k] = (uint16_t)rd(2);
  const uint32_t w = rd(fl), h = rd(fl);
  if (w == 0 || h == 0) return "Overlay image with zero width or height.";
  if (w > 0x7fffffffu || h > 0x7fffffffu || (uint64_t)w * h > (uint64_t)32768 * 32768) return "overlay canvas exceeds the maximum image size";
  o.canvas_w = (int)w; o.canvas_h = (int)h;
  for (size_t k = 0; k < o.children.size(); k++) {
    const uint32_t x = rd(fl), y = rd(fl);
    o.offsets.push_back({fl == 2 ? (int32_t)(int16_t)x : (int32_t)x, fl == 2 ? (int32_t)(int16_t)y : (int32_t)y});
  }
  return "";
}

bool HeifFile::premultiplied(uint32_t id) const {
  for (auto& r : refs_)
    if (r.type == fourcc("prem") && r.from == id) return true;
  return false;
}

uint32_t HeifFile::alpha_item(uint32_t id) const {
  for (auto& r : refs_) {
    if (r.type != fourcc("auxl")) continue;
    bool to_me = false;
    for (uint32_t t : r.to) if (t == id) to_me = true;
    if (!to_me) continue;
    const HeifItem* a = item(r.from);
    if (a && is_alpha_urn(a->aux_type)) return a->id;
  }
  return 0;
}

bool HeifFile::is_image_item(uint32_t id) const {
  const HeifItem* it = item(id);
  return it && (it->type == fourcc("hvc1") || it->type == fourcc("grid") || it->type == fourcc("iovl"));
}

// the items with a `ref_type` reference to `id`, ascending and each once
std::vector<uint32_t> HeifFile::referring(uint32_t ref_type, uint32_t id) const {
  std::vector<uint32_t> out;
  for (auto& r : refs_) {
    if (r.type != ref_type || !item(r.from)) continue;
    for (uint32_t t : r.to)
      if (t == id) { out.push_back(r.from); break; }
  }
  std::sort(out.begin(), out.end());
  out.erase(std::unique(out.begin(), out.end()), out.end());
  return out;
}

std::vector<uint32_t> HeifFile::thumbnails(uint32_t id) const { return referring(fourcc("thmb"), id); }

std::vector<uint32_t> HeifFile::auxiliaries(uint32_t id, bool include_alpha) const {
  std::vector<uint32_t> out = referring(fourcc("auxl"), id);
  if (!include_alpha) out.erase(std::remove_if(out.begin(), out.end(), [&](uint32_t a) { return is_alpha_urn(item(a)->aux_type); }), out.end());
  return out;
}

std::string HeifFile::coded_stream(uint32_t id, std::vector<uint8_t>& out) const {
  const HeifItem* it = item(id);
  if (!it) return "no such item";
  if (it->type != fourcc("hvc1")) return "item is not an HEVC image (hvc1)";
  if (it->hvcc_prop < 0) return "HEVC item without hvcC configuration";
  const HeifHvcC& h = hvcc_[it->hvcc_prop];
  out.clear();
  for (auto& nal : h.nals) {
    uint32_t n = (uint32_t)nal.size();
    out.push_back((uint8_t)(n >> 24)); out.push_back((uint8_t)(n >> 16));
    out.push_back((uint8_t)(n >> 8)); out.push_back((uint8_t)n);
    out.insert(out.end(), nal.begin(), nal.end());
  }
  std::vector<uint8_t> d;
  std::string e = read_item_data(*it, d);
  if (!e.empty()) return e;
  if (h.length_size == 4) {
    out.insert(out.end(), d.begin(), d.end());
  } else {
    size_t pos = 0;
    while (pos + h.length_size <= d.size()) {
      uint32_t n = 0;
      for (int i = 0; i < h.length_size; i++) n = (n << 8) | d[pos++];
      if (n > d.size() - pos) return "NAL length exceeds the item data";
      out.push_back((uint8_t)(n >> 24)); out.push_back((uint8_t)(n >> 16));
      out.push_back((uint8_t)(n >> 8)); out.push_back((uint8_t)n);
      out.insert(out.end(), d.begin() + pos, d.begin() + pos + n);
      pos += n;
    }
  }
  return "";
}

}  // namespace hc
