// heif_reader.h — minimal ISO-BMFF / HEIF item resolver for the batch driver (SURVEY.md §8f N1).
//
// The plugin path does not need this (libheif parses the container and hands the plugin NAL
// units); the batch API (hc_decode_heic*) does: it must find, for every image of a file, the
// coded HEVC items (single image or all grid tiles, plus an alpha auxiliary image), their hvcC
// parameter sets and the paste geometry, so that all tiles of all images can be in flight on the
// GPU at once instead of libheif's one-decoder-per-tile call pattern (context.cc:2361-2415).
//
// New code written from ISO/IEC 14496-12 (box structure, iloc/iinf/iref/iprp) and ISO/IEC 23008-12
// (hvc1/grid items, ispe/colr/pixi/auxC/irot/imir). Reference counterparts: libheif/box.cc,
// libheif/file.cc:1246-1536 (get_compressed_image_data), libheif/context.cc:172-221 (ImageGrid::parse),
// :710-1240 (interpret_heif_file), codecs/hevc.cc:226-247 (hvcC headers).
#pragma once
#include <cstdint>
#include <map>
#include <string>
#include <vector>

namespace hc {

struct HeifNclx {
  bool present = false;
  int primaries = 2, transfer = 2, matrix = 2, full_range = 0;
};

struct HeifItem {
  uint32_t id = 0;
  uint32_t type = 0;            // fourcc
  bool hidden = false;
  int construction_method = 0;  // 0 file offset, 1 idat
  uint64_t base_offset = 0;
  struct Extent { uint64_t offset, length; };
  std::vector<Extent> extents;
  std::vector<int> props;       // 1-based indices into ipco
  // resolved properties
  int ispe_w = 0, ispe_h = 0;
  int hvcc_prop = -1;           // index into HeifFile::hvcc
  HeifNclx nclx;
  int rot = 0;                  // irot: anti-clockwise quarter turns
  int mirror = -1;              // imir: -1 none, 0 vertical axis, 1 horizontal axis
  bool has_clap = false;
  struct Clap { uint32_t w_num, w_den, h_num, h_den; int32_t hoff_num; uint32_t hoff_den; int32_t voff_num; uint32_t voff_den; };
  std::vector<Clap> claps;      // clap boxes in ipma order; xforms code 6 consumes the next one
  std::vector<uint8_t> xforms;  // irot / imir in ipma order (context.cc:1955-1978): 1..3 = quarter turns anti-clockwise,
                                // 4 = mirror direction horizontal (rows reversed), 5 = vertical (row order reversed), 6 = clap
  std::string aux_type;         // auxC
  int pixi_bits = 0;
};

struct HeifHvcC {
  int length_size = 4;
  std::vector<std::vector<uint8_t>> nals;   // parameter set NAL units
};

struct HeifGrid {
  int rows = 0, cols = 0;
  int out_w = 0, out_h = 0;
  std::vector<uint32_t> tiles;  // item ids, row-major
};

// 'iovl' derived image item (ISO/IEC 23008-12 6.6.2.2; libheif ImageOverlay::parse, context.cc:318-369)
struct HeifOverlay {
  int canvas_w = 0, canvas_h = 0;
  uint16_t background[4] = {0, 0, 0, 0};   // R, G, B, A, 16 bit each
  std::vector<uint32_t> children;          // 'dimg' references, bottom first
  std::vector<std::pair<int32_t, int32_t>> offsets;
};

class HeifFile {
 public:
  // Parses the box structure. `data` must stay valid while the object is used.
  std::string parse(const uint8_t* data, size_t size);

  uint32_t primary_id() const { return primary_; }
  const HeifItem* item(uint32_t id) const;
  // image items that are not hidden, thumbnails or auxiliary images (libheif's "top level images")
  std::vector<uint32_t> top_level_images() const;
  bool is_grid(uint32_t id) const;
  std::string grid(uint32_t id, HeifGrid& g) const;
  bool is_overlay(uint32_t id) const;
  std::string overlay(uint32_t id, HeifOverlay& o) const;
  // the item types that are decoded as images: 'hvc1', 'grid' and 'iovl'
  bool is_image_item(uint32_t id) const;
  // alpha auxiliary image item of `id`, or 0
  uint32_t alpha_item(uint32_t id) const;
  // items with a 'thmb' reference to `id`, in ascending item id
  std::vector<uint32_t> thumbnails(uint32_t id) const;
  // items with an 'auxl' reference to `id`, in ascending item id; alpha images only when `include_alpha`
  std::vector<uint32_t> auxiliaries(uint32_t id, bool include_alpha) const;
  // a 'prem' item reference from the colour image: its samples are stored premultiplied by alpha (context.cc:1150-1161)
  bool premultiplied(uint32_t id) const;
  // hvcC parameter sets followed by the item's coded data, every NAL prefixed by a 4-byte
  // big-endian length: exactly what libheif passes to heif_decoder_plugin::push_data
  // (file.cc:1496-1536, codecs/hevc.cc:226-247).
  std::string coded_stream(uint32_t id, std::vector<uint8_t>& out) const;

 private:
  std::string read_item_data(const HeifItem& it, std::vector<uint8_t>& out) const;
  std::vector<uint32_t> referring(uint32_t ref_type, uint32_t id) const;
  const uint8_t* data_ = nullptr;
  size_t size_ = 0;
  uint32_t primary_ = 0;
  std::map<uint32_t, HeifItem> items_;
  std::vector<HeifHvcC> hvcc_;
  struct Ref { uint32_t type, from; std::vector<uint32_t> to; };
  std::vector<Ref> refs_;
  const uint8_t* idat_ = nullptr;
  size_t idat_size_ = 0;
};

}  // namespace hc
