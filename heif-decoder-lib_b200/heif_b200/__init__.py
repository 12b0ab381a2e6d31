"""heif_b200 — Python host-side mirror of the reference's decoder interface for the B200 HEVC-intra
engine (tests and bench use it; the product boundary is the C ABI in include/heifcuda.h)."""
from ._lib import load, lib_path, HeifCudaError, Pic, CscParams  # noqa: F401
from .api import (Records, K0Picture, HeifFile, Engine, Batch, HeicJob, parse_picture, parse_picture_k0, csc_select, decode_heic, decode_stream,  # noqa: F401
                  plane_layout, split_planes, OUT_YCBCR,
                  STREAM_LENGTH_PREFIXED, STREAM_ANNEXB, OUT_RGB, OUT_RGBA, OUT_RRGGBB_BE, OUT_RRGGBBAA_BE,
                  OUT_RRGGBB_LE, OUT_RRGGBBAA_LE, STAGE_DEBLOCK, STAGE_SAO, STAGE_ALL)
