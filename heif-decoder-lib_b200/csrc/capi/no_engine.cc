// no_engine.cc — hc_engine_* entry points of the host-only library (libheifcuda_host.so).
// There is NO CPU implementation of the reconstruction path: every call fails loudly.
#include "capi_internal.h"

#define NO_ENGINE() (hc::set_last_error("this build has no CUDA engine and there is no CPU fallback"), HC_ERR_NO_DEVICE)

extern "C" {
int hc_has_cuda_engine(void) { return 0; }
hc_engine* hc_engine_create(int) { NO_ENGINE(); return nullptr; }
void hc_engine_destroy(hc_engine*) {}
int hc_engine_set_option(hc_engine*, const char*, int) { return NO_ENGINE(); }
int hc_engine_get_option(const hc_engine*, const char*) { return 0; }
hc_batch* hc_batch_create(hc_engine*) { NO_ENGINE(); return nullptr; }
void hc_batch_destroy(hc_batch*) {}
int hc_batch_add_canvas(hc_batch*, int, int, int, int, int) { return NO_ENGINE(); }
int hc_batch_add_picture(hc_batch*, const hc_records*, int, int, int, int, int) { return NO_ENGINE(); }
int hc_batch_add_k0_picture(hc_batch*, const hc_k0_picture*, int, int, int, int, int) { return NO_ENGINE(); }
int hc_batch_k0_pictures(const hc_batch*) { return 0; }
int hc_batch_set_canvas_transform(hc_batch*, int, int, int, int) { return NO_ENGINE(); }
int hc_batch_add_canvas_pass(hc_batch*, int, int, int, int, int, int) { return NO_ENGINE(); }
int hc_batch_link_alpha(hc_batch*, int, int) { return NO_ENGINE(); }
int hc_batch_set_canvas_output_size(hc_batch*, int, int, int) { return NO_ENGINE(); }
int hc_batch_upload(hc_batch*) { return NO_ENGINE(); }
int hc_batch_reconstruct(hc_batch*, int) { return NO_ENGINE(); }
int hc_batch_reconstruct_async(hc_batch*, int) { return NO_ENGINE(); }
int hc_batch_convert(hc_batch*, int, const hc_csc_params*) { return NO_ENGINE(); }
int hc_batch_convert_many(hc_batch*, int, const int*, const hc_csc_params*) { return NO_ENGINE(); }
int hc_batch_sync(hc_batch*) { return NO_ENGINE(); }
int hc_batch_read_plane(hc_batch*, int, int, void*, size_t) { return NO_ENGINE(); }
int hc_batch_read_planes(hc_batch*, int, int, void* const*, const size_t*) { return NO_ENGINE(); }
int hc_batch_read_rgb(hc_batch*, int, void*, size_t) { return NO_ENGINE(); }
int hc_batch_copy_rgb_device(hc_batch*, int, void*, size_t) { return NO_ENGINE(); }
int hc_batch_read_rgb_async(hc_batch*, int, void*, size_t) { return NO_ENGINE(); }
int hc_batch_read_residual(hc_batch*, int, int16_t*, size_t) { return NO_ENGINE(); }
int hc_batch_stage_ms(hc_batch*, float*) { return NO_ENGINE(); }
int hc_batch_timer_start(hc_batch*) { return NO_ENGINE(); }
int hc_batch_timer_stop_ms(hc_batch*, float*) { return NO_ENGINE(); }
int hc_batch_launch_count(const hc_batch*) { return 0; }
size_t hc_batch_upload_bytes(const hc_batch*) { return 0; }
int hc_batch_set_rgb_target(hc_batch*, int, void*, size_t) { return NO_ENGINE(); }
void hc_batch_set_pack_threads(hc_batch*, int) {}
int hc_batch_failed_pictures(const hc_batch*, const int**) { return 0; }
int hc_batch_timeline_ms(hc_batch*, float*) { return NO_ENGINE(); }
void hc_batch_mark_d2h(hc_batch*, int) {}
void* hc_engine_take_out_pinned(hc_engine*, size_t, size_t*) { NO_ENGINE(); return nullptr; }
void hc_engine_give_out_pinned(hc_engine*, void*, size_t) {}
float hc_batch_async_d2h_ms(hc_batch*) { return 0.f; }
int hc_batch_add_overlay_canvas(hc_batch*, int, int, const uint16_t*) { return NO_ENGINE(); }
int hc_batch_overlay_add_child(hc_batch*, int, int, int, int, const hc_csc_params*) { return NO_ENGINE(); }
hc_shared_image* hc_shared_image_create(hc_engine*, int, int, int) { NO_ENGINE(); return nullptr; }
int hc_shared_image_export(const hc_shared_image*, uint8_t*) { return NO_ENGINE(); }
hc_shared_image* hc_shared_image_open(hc_engine*, const uint8_t*, int, int, int) { NO_ENGINE(); return nullptr; }
hc_shared_image* hc_shared_image_attach(hc_engine*, const hc_shared_image*) { NO_ENGINE(); return nullptr; }
void hc_shared_image_destroy(hc_shared_image*) {}
void* hc_shared_image_device_ptr(const hc_shared_image*) { return nullptr; }
size_t hc_shared_image_stride(const hc_shared_image*) { return 0; }
int hc_shared_image_read(hc_shared_image*, int, int, void*, size_t) { return NO_ENGINE(); }
int hc_shared_image_geometry(const hc_shared_image*, int*, int*, int*) { return NO_ENGINE(); }
void* hc_host_alloc(size_t) { NO_ENGINE(); return nullptr; }
void hc_host_free(void*) {}
}
