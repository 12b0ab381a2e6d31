// capi_internal.h — definitions shared by the C-ABI translation units.
#pragma once
#include <memory>
#include <string>
#include "../../../include/heifcuda.h"
#include "../host/hevc_parse.h"
#include "../host/heif_reader.h"
#include "../host/k0_host.h"

struct hc_parser {
  hc::HevcIntraParser parser;
};
struct hc_records {
  std::unique_ptr<hc::PictureRecords> rec;
};
struct hc_k0_picture {
  hc::K0HostPicture hp;
};
struct hc_heif {
  hc::HeifFile file;
};

namespace hc {
void set_last_error(const std::string& s);
// samples of plane c (0 Y, 1 Cb, 2 Cr, 3 A) of a w x h image: chroma planes round up; 0 for the chroma of monochrome
inline int plane_w(int w, int chroma, int c) { return (c == 0 || c == 3 || chroma == 3) ? w : (chroma == 0 ? 0 : (w + 1) / 2); }
inline int plane_h(int h, int chroma, int c) { return (c == 0 || c == 3 || chroma != 1) ? (chroma == 0 && c != 0 && c != 3 ? 0 : h) : (h + 1) / 2; }
}
