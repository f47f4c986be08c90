/*
 * scgib_private.h - entry points of libscgib.so that are NOT part of the drop-in boundary (include/scgib.h):
 * implementation selection for cross-checks and the role-timeline dumps of the warp-specialised kernels.
 * Used by tests/ and the experiment scripts only.
 */
#ifndef SCGIB_PRIVATE_H_
#define SCGIB_PRIVATE_H_
#include "../../include/scgib.h"
#ifdef __cplusplus
extern "C" {
#endif
/* GIN forward: 1 = tcgen05 kernels (gin_tc3.cu fp32 / gin_bf16.cu bf16; default), 0 = FP32 FFMA register tiles
 * (gin_kernels.cu).  Also the environment variable SCGIB_TC; mode < 0 restores the default. */
SCGIB_API void scgib_set_tensor_cores(int mode);
/* fp32 GIN, head MLP and compressor backward at hidden 64: 1 = tcgen05 two-term fp16 splits (gin_bwd_h.cu; default),
 * 0 = FP32 FFMA register tiles (gin_kernels.cu).  Also the environment variable SCGIB_TC_BWD; mode < 0 restores the default. */
SCGIB_API void scgib_set_tensor_cores_bwd(int mode);
/* Per-tile role timestamps of the last gin_fwd_tc3 launch run with SCGIB_DBG bit 1024
 * ([cta < 160][tile < 16][event < 12] SM clocks) copied to host memory. */
SCGIB_API int scgib_debug_tc2_trace(long long* host_out, int n);
SCGIB_API int scgib_debug_bf16_trace(long long* host_out, int n);     /* gin_fwd_bf16 (bf16 mode), same layout */
SCGIB_API int scgib_debug_bwdh_trace(long long* host_out, int n);     /* gin_bwd_h (SCGIB_DBG bit 2048), same layout */
#ifdef __cplusplus
}
#endif
#endif
