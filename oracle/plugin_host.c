/* plugin_host.c — the part of libheif's public API a decoder plugin calls back into (heif_image_create / add_plane /
 * get_plane / release, the nclx profile setters, heif_image_add_decoding_warning; heif.h:1414-1456,1731-1781,2342-2376),
 * restated as plain memory so that the tests can drive libheif-cuda.so through its plugin ABI when the reference
 * libheif (oracle/_ref) is not built. Test infrastructure (the checker): grid paste, alpha and colour conversion of the
 * decoded images are done by tests/heic_oracle.py, pinned against the reference's golden MD5s.
 * The plugin finds these symbols through HEIFCUDA_LIBHEIF (decoder_cuda.cc, resolve_api). */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "../include/heifcuda_plugin.h"

#define PH_EXPORT __attribute__((visibility("default")))

typedef struct {
  int width, height, bits, stride;
  uint8_t* data;
} ph_plane;

typedef struct {
  int width, height, colorspace, chroma;
  ph_plane planes[4]; /* heif_channel_Y / Cb / Cr / (3: unused) */
  hcp_nclx nclx;
  int has_nclx, warnings;
} ph_image;

static const hcp_error ph_ok = {HCP_ERROR_OK, 0, "Success"};
static const hcp_error ph_bad = {HCP_ERROR_DECODER_PLUGIN, 0, "plugin_host: invalid argument"};
static const hcp_error ph_nomem = {HCP_ERROR_MEMORY_ALLOCATION, 0, "plugin_host: out of memory"};

PH_EXPORT hcp_error heif_image_create(int width, int height, int colorspace, int chroma, void** out) {
  ph_image* img = (ph_image*)calloc(1, sizeof(ph_image));
  if (!img) return ph_nomem;
  img->width = width;
  img->height = height;
  img->colorspace = colorspace;
  img->chroma = chroma;
  *out = img;
  return ph_ok;
}

PH_EXPORT hcp_error heif_image_add_plane(void* raw, int channel, int width, int height, int bits) {
  ph_image* img = (ph_image*)raw;
  if (!img || channel < 0 || channel > 2 || width <= 0 || height <= 0 || bits <= 0 || bits > 16 || img->planes[channel].data)
    return ph_bad;
  ph_plane* p = &img->planes[channel];
  p->stride = (width * ((bits + 7) / 8) + 63) & ~63; /* padded rows, as libheif's planes have */
  p->data = (uint8_t*)calloc((size_t)p->stride, (size_t)height);
  if (!p->data) return ph_nomem;
  p->width = width;
  p->height = height;
  p->bits = bits;
  return ph_ok;
}

PH_EXPORT uint8_t* heif_image_get_plane(void* raw, int channel, int* stride) {
  ph_image* img = (ph_image*)raw;
  if (!img || channel < 0 || channel > 2 || !img->planes[channel].data) return NULL;
  if (stride) *stride = img->planes[channel].stride;
  return img->planes[channel].data;
}

PH_EXPORT void heif_image_release(const void* raw) {
  ph_image* img = (ph_image*)raw;
  if (!img) return;
  for (int c = 0; c < 4; c++) free(img->planes[c].data);
  free(img);
}

PH_EXPORT hcp_nclx* heif_nclx_color_profile_alloc(void) {
  hcp_nclx* n = (hcp_nclx*)calloc(1, sizeof(hcp_nclx));
  if (n) {
    n->version = 1;
    n->color_primaries = n->transfer_characteristics = n->matrix_coefficients = 2; /* unspecified */
    n->full_range_flag = 1;
  }
  return n;
}

PH_EXPORT void heif_nclx_color_profile_free(hcp_nclx* n) { free(n); }

PH_EXPORT hcp_error heif_nclx_color_profile_set_color_primaries(hcp_nclx* n, uint16_t v) {
  if (!n) return ph_bad;
  n->color_primaries = v;
  return ph_ok;
}

PH_EXPORT hcp_error heif_nclx_color_profile_set_transfer_characteristics(hcp_nclx* n, uint16_t v) {
  if (!n) return ph_bad;
  n->transfer_characteristics = v;
  return ph_ok;
}

PH_EXPORT hcp_error heif_nclx_color_profile_set_matrix_coefficients(hcp_nclx* n, uint16_t v) {
  if (!n) return ph_bad;
  n->matrix_coefficients = v;
  return ph_ok;
}

PH_EXPORT hcp_error heif_image_set_nclx_color_profile(void* raw, const hcp_nclx* n) {
  ph_image* img = (ph_image*)raw;
  if (!img || !n) return ph_bad;
  img->nclx = *n;
  img->has_nclx = 1;
  return ph_ok;
}

PH_EXPORT void heif_image_add_decoding_warning(void* raw, hcp_error e) {
  (void)e;
  if (raw) ((ph_image*)raw)->warnings++;
}

/* read-back for the tests: plane geometry (0 when the plane is absent) and the nclx the decoder attached */
PH_EXPORT int ph_image_plane(const void* raw, int channel, int* width, int* height, int* bits, int* stride) {
  const ph_image* img = (const ph_image*)raw;
  if (!img || channel < 0 || channel > 2 || !img->planes[channel].data) return 0;
  const ph_plane* p = &img->planes[channel];
  *width = p->width;
  *height = p->height;
  *bits = p->bits;
  *stride = p->stride;
  return 1;
}

PH_EXPORT int ph_image_nclx(const void* raw, int out[4]) {
  const ph_image* img = (const ph_image*)raw;
  if (!img || !img->has_nclx) return 0;
  out[0] = img->nclx.color_primaries;
  out[1] = img->nclx.transfer_characteristics;
  out[2] = img->nclx.matrix_coefficients;
  out[3] = img->nclx.full_range_flag;
  return 1;
}
