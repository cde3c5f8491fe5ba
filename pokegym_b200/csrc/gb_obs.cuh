// gb_obs.cuh -- packed observations (gbenv_step_packed / gbenv_reset_packed / gbenv_unpack_obs), kernels in gb_obs.cu.
//
// The kernels live in their own translation unit so that adding them leaves the code generated for gbenv.cu's kernels
// exactly as it was (see gb_frames.cuh).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

// k_obs_pack on `st`: the packed observation (include/gbenv.h) of every env e < n_envs with mask[e] != 0 (invert: == 0;
// mask NULL: all) into packed[e][GBENV_OBS_PACKED_WORDS]; other rows are untouched.  `mem` / `fb` are the interleaved
// emulator arrays, `vis_pt` / `vis_pool` the visited-bitmap page tables and pages.  `packed` is 16-byte aligned.
cudaError_t launch_obs_pack(const uint32_t *mem, const uint32_t *fb, const uint32_t *vis_pt, const uint32_t *vis_pool, int n_envs, int n_tiles,
                            const uint8_t *mask, int invert, uint32_t *packed, cudaStream_t st);
// k_obs_unpack on `st`: n packed rows -> out[n][GBENV_OBS_BYTES] in the reference layout (both 16-byte aligned).
cudaError_t launch_obs_unpack(const uint32_t *packed, int n, uint8_t *out, cudaStream_t st);
