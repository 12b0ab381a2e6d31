// launch.h — host-callable launchers of the sm_100a kernels (defined in the k*.cu files).
#pragma once
#include <cuda_runtime.h>
#include "common.cuh"
#include "../../../include/heifcuda.h"

namespace hc {

// largest gridDim.y (and gridDim.z) of a launch
constexpr int kMaxGridY = 65535;

struct CscArgs {
  const uint8_t* y;  const uint8_t* cb;  const uint8_t* cr;  const uint8_t* a;   // plane bases (bytes)
  int y_stride, c_stride, a_stride;   // in samples
  int width, height;                  // written (delivered) image
  int chroma_format;                  // 0..3
  uint8_t* out;
  long long out_stride;               // bytes
  hc_csc_params p;
  // gather != 0: the planes are src_w x src_h and output pixel (x, y) is converted from source pixel
  // (x * src_w / width, y * src_h / height), nearest neighbour like HeifPixelImage::scale_nearest_neighbor
  int src_w, src_h, gather;
};

// up to CSC_BATCH_MAX canvases of one sample size converted by one launch (kernel parameter space: 4 KB)
constexpr int CSC_BATCH_MAX = 24;
struct CscBatch {
  CscArgs a[CSC_BATCH_MAX];
  int n;
};

// K6: one plane through one dihedral map (see hc_batch_set_canvas_transform); strides in samples
struct XformArgs {
  const uint8_t* src;
  uint8_t* dst;
  int w, h;                  // input plane size
  int src_stride, dst_stride;
  int swap, flip_x, flip_y;
};

// K7: one 'iovl' derived image composed from up to OVERLAY_MAX child canvases (8-bit 4:4:4, optional alpha plane)
constexpr int OVERLAY_MAX = 16;
struct OverlayChild {
  const uint8_t* y; const uint8_t* cb; const uint8_t* cr; const uint8_t* a;
  int y_stride, c_stride, a_stride;
  int w, h, dx, dy;
  int mode, full_range;            // HC_CSC_FLOAT / GBR / YCGCO of Op_YCbCr_to_RGB<uint8_t>
  float r_cr, g_cb, g_cr, b_cb;
};
struct OverlayArgs {
  OverlayChild child[OVERLAY_MAX];
  int n;
  int width, height;               // written (delivered) image
  int bkg[3];                      // background colour, already reduced to 8 bit
  int out_format;
  uint8_t* out;
  long long out_stride;
  // canvas size; when it differs from width x height, output pixel (x, y) is the composition at canvas pixel
  // (x * src_w / width, y * src_h / height)
  int src_w, src_h;
  int row0, full_h;                // set by launch_k7 for each band of a scaled image: its first row, all delivered rows
};
void launch_k7(const OverlayArgs& a, cudaStream_t stream);

// K8: planes copied from the plane pool (pitched rows) into packed HC_OUT_YCBCR images (tight rows, one plane after the
// other). Plane by plane, whatever the sample size: a plane is row_bytes x rows bytes.
struct PackPlane {
  const uint8_t* src;        // first row of the plane in the pool
  uint8_t* dst;              // packed destination, any alignment
  unsigned src_pitch;        // bytes between source rows
  unsigned row_bytes;        // plane width x sample bytes
  unsigned rows;
  unsigned pad;
};
// planes of up to 24 canvases per launch (kernel parameter space: 4 KB)
constexpr int PACK_BATCH_MAX = 96;
struct PackBatch {
  PackPlane p[PACK_BATCH_MAX];
  int n;
};
void launch_k8_batch(const PackBatch& b, cudaStream_t stream);

namespace k0 { struct Tables; struct Pic; struct Sub; struct Chain; }
// K0: device CABAC parse of the pictures added as bitstreams (one CTA per substream chain)
void launch_k0(const k0::Tables* tables, const k0::Pic* pics, const k0::Sub* subs, const k0::Chain* chains, int nchains,
               cudaStream_t stream);
void launch_k0_finish(const k0::Pic* pics, int npics, int max_ctbs, cudaStream_t stream);
void launch_k1(const BatchView& bv, const uint32_t* const tb_index[4], const int counts[4], cudaStream_t stream);
// lists built on the device (K0): capacity[l] entries at most, the real lengths are d_counts[0..3] in device memory
void launch_k1_indirect(const BatchView& bv, const uint32_t* const tb_index[4], const long long capacity[4], const unsigned* d_counts,
                        int sm_count, cudaStream_t stream);
// shared-memory bytes one K2 row task needs (CTB of ctb_w x ctb_h samples of this component)
int k2_task_smem_bytes(int ctb_w, int ctb_h, int pixel_bytes);
// per-warp task lists: `work` holds 3 entries per CTA; smem_bytes: dynamic shared memory per CTA = max over CTAs of the
// bytes its lists need
void launch_k2(const BatchView& bv, const RowTask* tasks, const WarpWork* work, int nctas, int smem_bytes, int* progress, cudaStream_t stream);
void launch_k3(const BatchView& bv, long long max_units, int planes, cudaStream_t stream);
void launch_k4(const BatchView& bv, long long max_ctbs, int planes, cudaStream_t stream);
void launch_k5(const CscArgs& a, bool sixteen_bit, cudaStream_t stream);
void launch_k5_batch(const CscBatch& b, bool sixteen_bit, cudaStream_t stream);
void launch_k6(const XformArgs& a, bool sixteen_bit, cudaStream_t stream);
// nearest-neighbour rescale of one plane (strides in samples): dst(x, y) = src(x * sw / dw, y * sh / dh)
void launch_k6_scale(const uint8_t* src, int sw, int sh, int src_stride, uint8_t* dst, int dw, int dh, int dst_stride, bool sixteen_bit,
                     cudaStream_t stream);

}  // namespace hc
