// tools/obs_kernels.cu -- timing harness of tools/bench_obs_packed.py, not part of the library: the two observation writers,
// k_wrap_obs (reference rows, gb_wrap.cuh) and k_obs_pack (packed rows, gb_obs.cu), launched alone on the same synthetic
// batch and timed with CUDA events, the L2 overwritten before every timed launch.
//
// The batch: WRAM, framebuffer and bitmap pages filled with hashed bits, so positions and maps are spread over 0..255 / 0..247
// and every page-table entry of every env points to a page of a pool of 4 pages per env.  Every obs row of every env then has
// a bitmap row to read, which is the most work either kernel can have.
#include <cuda_runtime.h>
#include "../pokegym_b200/csrc/gb_wrap.cuh"
#include "../pokegym_b200/csrc/gb_obs.cu"

__global__ void k_hash_fill(uint32_t *p, size_t n, uint32_t seed, uint32_t modulo) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        uint32_t x = (uint32_t)i * 0x9E3779B9u ^ seed;
        x ^= x >> 16; x *= 0x7FEB352Du; x ^= x >> 15; x *= 0x846CA68Bu; x ^= x >> 16;
        p[i] = modulo ? x % modulo + 1 : x;
    }
}

// mean device ms of one launch of k_wrap_obs (ms[0]) and k_obs_pack (ms[1]) over `reps` alternated launches of each at n envs
extern "C" int obs_kernel_ms(int n, int reps, float *ms) {
    const int tiles = (n + GB_TILE - 1) / GB_TILE;
    const size_t pages = (size_t)n * 4, flush_bytes = (size_t)256 << 20;
    DevArrays d{};
    WrapArrays w{};
    uint8_t *obs = nullptr, *flush = nullptr;
    uint32_t *packed = nullptr;
    cudaEvent_t e0, e1;
    if (cudaMalloc(&d.mem, (size_t)tiles * GB_TILE * MEM_WORDS * 4) || cudaMalloc(&d.fb, (size_t)tiles * GB_TILE * FB_WORDS * 4) ||
        cudaMalloc(&w.vis_pt, (size_t)n * VIS_PT_ENTRIES * 4) || cudaMalloc(&w.vis_pool, pages * VIS_PAGE_WORDS * 4) ||
        cudaMalloc(&obs, (size_t)n * GBENV_OBS_BYTES) || cudaMalloc(&packed, (size_t)n * GBENV_OBS_PACKED_BYTES) || cudaMalloc(&flush, flush_bytes))
        return -1;
    d.n_envs = n;
    d.n_tiles = tiles;
    k_hash_fill<<<1024, 256>>>(d.mem, (size_t)tiles * GB_TILE * MEM_WORDS, 1u, 0u);
    k_hash_fill<<<1024, 256>>>(d.fb, (size_t)tiles * GB_TILE * FB_WORDS, 2u, 0u);
    k_hash_fill<<<1024, 256>>>(w.vis_pt, (size_t)n * VIS_PT_ENTRIES, 3u, (uint32_t)pages);
    k_hash_fill<<<1024, 256>>>(w.vis_pool, pages * VIS_PAGE_WORDS, 4u, 0u);
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    double total[2] = {0.0, 0.0};
    for (int r = -2; r < reps; r++) {  // two untimed rounds first
        for (int which = 0; which < 2; which++) {
            cudaMemsetAsync(flush, r & 0xFF, flush_bytes, 0);
            cudaEventRecord(e0, 0);
            if (which == 0)
                k_wrap_obs<<<tiles, 256>>>(d, w, nullptr, obs, GBENV_OBS_BYTES, 0);
            else
                launch_obs_pack(d.mem, d.fb, w.vis_pt, w.vis_pool, n, tiles, nullptr, 0, packed, 0);
            cudaEventRecord(e1, 0);
            cudaEventSynchronize(e1);
            float t = 0.f;
            cudaEventElapsedTime(&t, e0, e1);
            if (r >= 0) total[which] += t;
        }
    }
    const int rc = cudaGetLastError() == cudaSuccess ? 0 : -3;
    ms[0] = (float)(total[0] / reps);
    ms[1] = (float)(total[1] / reps);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d.mem); cudaFree(d.fb); cudaFree(w.vis_pt); cudaFree(w.vis_pool); cudaFree(obs); cudaFree(packed); cudaFree(flush);
    return rc;
}
