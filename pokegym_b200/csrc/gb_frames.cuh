// gb_frames.cuh -- batched frame capture and decode (gbenv_capture_frames / gbenv_frames_to_rgb), kernels in gb_frames.cu.
//
// The kernels live in their own translation unit so that adding them leaves the code generated for gbenv.cu's kernels (the
// emulation, render, wrapper and reduction kernels) exactly as it was: nvcc's register numbering, and with it ptxas'
// schedule, depends on everything else in the module.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

// k_frames_capture on `st`: the framebuffer words of the envs ids[0..n) (ids NULL: 0..n-1) from the interleaved array `fb`
// into frames[n][FB_WORDS]; an entry whose id is outside [0, n_envs) is neither read nor written.
cudaError_t launch_frames_capture(const uint32_t *fb, const int32_t *ids, int n, int n_envs, uint32_t *frames, cudaStream_t st);
// k_frames_to_rgb on `st`: n_frames packed frames -> out[n_frames][144][160][channels] (channels 1 or 3, out 16-byte aligned).
cudaError_t launch_frames_to_rgb(const uint32_t *frames, int n_frames, int channels, uint8_t *out, cudaStream_t st);
