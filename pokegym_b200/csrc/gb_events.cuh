// gb_events.cuh -- the reference's 130 event flags of a list of envs (gbenv_event_flags), kernel in gb_events.cu.
//
// The kernel lives in its own translation unit so that adding it leaves the code generated for gbenv.cu's kernels exactly as
// it was: nvcc's register numbering, and with it ptxas' schedule, depends on everything else in the module.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

// k_event_flags on `st`: the event flags of the envs ids[0..n) (ids NULL: 0..n-1), read from the interleaved plain-RAM
// array `mem`, into flags[n][GBENV_EVENT_WORDS]; an entry whose id is outside [0, n_envs) is neither read nor written.
cudaError_t launch_event_flags(const uint32_t *mem, const int32_t *ids, int n, int n_envs, uint32_t *flags, cudaStream_t st);
