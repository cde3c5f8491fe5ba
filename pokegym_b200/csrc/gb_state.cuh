// gb_state.cuh -- batched PyBoy v9 save-states (gbenv_save_states, and gbenv_save_state on top of it) and load-states
// (gbenv_load_states), kernels in gb_state.cu.
//
// The kernel lives in its own translation unit so that adding it leaves the code generated for gbenv.cu's kernels exactly
// as it was (see gb_frames.cuh).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "gb_layout.cuh"

// k_save_states on `st`: the v9 file of the envs ids[0..n) (ids NULL: id0 .. id0 + n - 1) into blobs[n][GBENV_STATE_BYTES],
// rows contiguous; `blobs` is 16-byte aligned.  A row whose id is outside [0, d.n_envs) is left untouched and nothing is
// read for it.
cudaError_t launch_save_states(const DevArrays &d, const int32_t *ids, int id0, int n, uint8_t *blobs, cudaStream_t st);

// gbenv_load_states on `st`: k_load_check, then k_load_states.  Entry i loads env ids[i] (ids NULL: i) from row i of
// blobs[n][GBENV_STATE_BYTES] (16-byte aligned) and reports into status[i] (may be NULL).  claim is uint64[d.n_envs] that only
// ever grows; seq must exceed the seq of every earlier call with the same claim array.
cudaError_t launch_load_states(const DevArrays &d, const int32_t *ids, int n, const uint8_t *blobs, int32_t *status, unsigned long long *claim,
                               uint32_t seq, cudaStream_t st);
