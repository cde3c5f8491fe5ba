// gbenv.cu -- host side of libgbenv.so: the C ABI of include/gbenv.h over the CUDA kernels.
// There is no CPU fallback anywhere in this file: every entry point either launches kernels on the
// handle's device or fails with GBENV_E_CUDA.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/gbenv.h"
#include "gb_events.cuh"
#include "gb_frames.cuh"
#include "gb_image.h"
#include "gb_kernels.cuh"
#include "gb_obs.cuh"
#include "gb_state.cuh"
#include "gb_wrap.cuh"

struct StateTemplate {
    uint32_t *d_image;  // IMG_WORDS words, canonical per-env image
    int version;
};

struct gbenv {
    int n = 0, n_tiles = 0, device = 0;
    DevArrays d{};
    WrapArrays w{};
    cudaStream_t stream = nullptr;
    std::vector<StateTemplate> templates;
    std::vector<int> initial_template;  // per env, -1 = none (host copy; the device copy d_init_tmpl is what resets read)
    int32_t *d_init_tmpl = nullptr;     // [n]
    uint32_t **d_tmpl_images = nullptr; // [MAX_TEMPLATES] device pointers of the template images
    int32_t *d_tmpl_versions = nullptr; // [MAX_TEMPLATES]
    bool tmpl_dirty = false;            // host-side template tables changed since the last upload
    bool loads_pending = false;         // some env may still have its first reset (which loads its save-state) ahead
    unsigned long long *d_counters = nullptr;
    uint32_t *d_stage_image = nullptr;
    uint8_t *d_stage_blob = nullptr;  // GBENV_STATE_BYTES, gbenv_save_state
    unsigned long long *d_load_claim = nullptr;  // [n] gbenv_load_states: (call << 32 | entry) of the entry an env takes
    uint32_t load_calls = 0;                     // gbenv_load_states calls so far (the high half of the claim keys)
    uint8_t *d_stage_buf = nullptr;  // 64 KiB scratch for bus access
    double *d_info_rows = nullptr;
    int32_t *d_env_ids = nullptr;
    uint8_t *d_mask = nullptr;
    // staging for the *_host entry points
    // two slots: step t+1 is emulated while the results of step t travel to the host (gbenv_submit_host / gbenv_fetch_host)
    uint8_t *d_actions[2] = {nullptr, nullptr}, *d_obs[2] = {nullptr, nullptr}, *d_done[2] = {nullptr, nullptr};
    double *d_reward[2] = {nullptr, nullptr};
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_stepped[2] = {nullptr, nullptr}, ev_copied[2] = {nullptr, nullptr};
    unsigned long long submitted = 0, fetched = 0;
    // cross-stream ordering of the calls on this handle (use_stream)
    cudaStream_t last_stream = nullptr;
    bool last_stream_valid = false;
    cudaEvent_t ev_order = nullptr;
    // CUDA-event ring: slot k holds {start, after k_run_frames, after k_wrap_*} of step k (mod EV_RING)
    static const int EV_RING = 64;
    cudaEvent_t ev[EV_RING][3] = {};
    unsigned long long ev_step = 0, ev_folded = 0;  // steps recorded / steps folded into the totals
    double ms_total[2] = {0.0, 0.0};
    bool ev_valid = false;
    unsigned long long launches = 0;
    int lanes = 32;  // envs per warp in k_run_frames
    int defer = 1;   // deferred PPU (GBENV_DEFER=0: draw inside the emulation kernel)
    size_t smem_opted = 48 * 1024;
    int32_t *pool_err_host = nullptr;  // pinned copy of WrapArrays.ctl[CTL_ERROR], refreshed asynchronously after every step / reset
    int32_t *d_cm_dense = nullptr;     // staging for gbenv_counts_map
    int cm_sum_chunk = 0;              // envs per block row of k_cm_sum (0 = not chosen yet)
    std::string err;
};

static thread_local std::string g_err;
static const int MAX_TEMPLATES = 1024;

#define CK(call)                                                                                       \
    do {                                                                                               \
        cudaError_t _e = (call);                                                                       \
        if (_e != cudaSuccess) {                                                                       \
            char _b[512];                                                                              \
            snprintf(_b, sizeof(_b), "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
            if (h) h->err = _b; else g_err = _b;                                                       \
            return GBENV_E_CUDA;                                                                       \
        }                                                                                              \
    } while (0)

static int fail(gbenv *h, int code, const char *msg) {
    if (h) h->err = msg; else g_err = msg;
    return code;
}

// Every entry point does its work on ONE stream: the caller's (`stream` argument; NULL = the legacy default stream, which
// is what PyTorch uses unless told otherwise) or the handle's own.  Calls on one handle take effect in call order whatever
// streams they use: when the stream changes, the new one first waits for an event recorded on the previous one, so e.g.
// gbenv_save_state (own stream) after gbenv_step on a PyTorch side stream sees the stepped state.
static cudaStream_t use_stream(gbenv *h, cudaStream_t s) {
    if (h->last_stream_valid && s != h->last_stream && h->ev_order) {
        cudaEventRecord(h->ev_order, h->last_stream);
        cudaStreamWaitEvent(s, h->ev_order, 0);
    }
    h->last_stream = s;
    h->last_stream_valid = true;
    return s;
}
static cudaStream_t pick(gbenv *h, void *stream) { return use_stream(h, (cudaStream_t)stream); }
static cudaStream_t own(gbenv *h) { return use_stream(h, h->stream); }

// all bitmap pages start on the free stack
__global__ void k_pool_init(WrapArrays w) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < w.vis_pages) w.vis_free[i] = i;
    if (i == 0) { w.ctl[CTL_VIS_FREE] = w.vis_pages; w.ctl[CTL_CM_NEXT] = 0; w.ctl[CTL_ERROR] = 0; }
}

// A pool of the exploration storage ran dry in an earlier step: the bits are sticky and the handle refuses further work.
static int pool_error(gbenv *h) {
    const int32_t e = h->pool_err_host ? *(volatile int32_t *)h->pool_err_host : 0;
    if (!e) return GBENV_OK;
    std::string msg = "exploration storage exhausted:";
    if (e & POOL_ERR_VISITED) msg += " visited-bitmap page pool (GBENV_VISITED_PAGES)";
    if (e & POOL_ERR_HEATMAP) msg += " heat-map block pool (GBENV_COUNTS_BLOCKS)";
    if (e & POOL_ERR_CUT_COORDS) msg += " cut_coords table (64 distinct tiles per episode)";
    msg += "; rewards / observations of the affected envs no longer match the reference";
    return fail(h, GBENV_E_NOMEM, msg.c_str());
}
static void queue_pool_error_copy(gbenv *h, cudaStream_t st) {
    cudaMemcpyAsync(h->pool_err_host, h->w.ctl + CTL_ERROR, sizeof(int32_t), cudaMemcpyDeviceToHost, st);
}

// ------------------------------------------------------------------------------- lifetime

extern "C" int gbenv_abi_version(void) { return GBENV_ABI_VERSION; }

extern "C" const char *gbenv_last_error(const gbenv *h) { return h ? h->err.c_str() : g_err.c_str(); }

extern "C" int gbenv_num_envs(const gbenv *h) { return h ? h->n : GBENV_E_ARG; }

static int scatter(gbenv *h, const uint32_t *d_image, int version, const int32_t *env_ids_host, int n, cudaStream_t st) {
    const int32_t *d_ids = nullptr;
    if (env_ids_host) {
        for (int i = 0; i < n; i++)
            if (env_ids_host[i] < 0 || env_ids_host[i] >= h->n) return fail(h, GBENV_E_ARG, "env id out of range");
        CK(cudaMemcpyAsync(h->d_env_ids, env_ids_host, sizeof(int32_t) * n, cudaMemcpyHostToDevice, st));
        d_ids = h->d_env_ids;
    } else {
        n = h->n;
    }
    if (n <= 0) return GBENV_OK;
    dim3 block(32, 8), grid((n + 31) / 32, (IMG_WORDS + 7) / 8);
    k_scatter_image<<<grid, block, 0, st>>>(h->d, d_image, d_ids, n, version);
    h->launches++;
    CK(cudaGetLastError());
    if (env_ids_host) CK(cudaStreamSynchronize(st));  // d_env_ids is reused by the next call
    return GBENV_OK;
}

extern "C" int gbenv_destroy(gbenv *h) {
    if (!h) return GBENV_E_ARG;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    for (auto &t : h->templates) cudaFree(t.d_image);
    cudaFree(h->d.mem); cudaFree(h->d.cram); cudaFree(h->d.fb); cudaFree(h->d.lp); cudaFree(h->d.regs); cudaFree(h->d.dl); cudaFree((void *)h->d.rom); cudaFree((void *)h->d.rom_dec);
    cudaFree(h->w.state); cudaFree(h->w.vis_pt); cudaFree(h->w.vis_pool); cudaFree(h->w.vis_free); cudaFree(h->w.cm_dir); cudaFree(h->w.cm_pool);
    cudaFree(h->w.ctl);
    if (h->pool_err_host) cudaFreeHost(h->pool_err_host);
    cudaFree(h->d_cm_dense);
    cudaFree(h->d_counters); cudaFree(h->d_stage_image); cudaFree(h->d_stage_blob); cudaFree(h->d_load_claim); cudaFree(h->d_stage_buf); cudaFree(h->d_info_rows);
    cudaFree(h->d_env_ids); cudaFree(h->d_mask); cudaFree(h->d_init_tmpl); cudaFree(h->d_tmpl_images); cudaFree(h->d_tmpl_versions);
    for (int k = 0; k < 2; k++) {
        cudaFree(h->d_actions[k]); cudaFree(h->d_obs[k]); cudaFree(h->d_done[k]); cudaFree(h->d_reward[k]);
        if (h->ev_stepped[k]) cudaEventDestroy(h->ev_stepped[k]);
        if (h->ev_copied[k]) cudaEventDestroy(h->ev_copied[k]);
    }
    if (h->ev_order) cudaEventDestroy(h->ev_order);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    for (auto &slot : h->ev)
        for (auto &e : slot)
            if (e) cudaEventDestroy(e);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return GBENV_OK;
}

static int create_impl(gbenv *&h, int n_envs, const uint8_t *rom_host, size_t rom_len, int device_id);

extern "C" int gbenv_create(int n_envs, const uint8_t *rom_host, size_t rom_len, int device_id, gbenv **out) {
    if (!out) return fail(nullptr, GBENV_E_ARG, "gbenv_create: bad argument");
    gbenv *h = nullptr;
    int rc = create_impl(h, n_envs, rom_host, rom_len, device_id);
    if (rc != GBENV_OK) {  // nothing is leaked on a failed create: the message moves to the global slot, the handle goes
        if (h) {
            if (!h->err.empty()) g_err = h->err;
            gbenv_destroy(h);
        }
        return rc;
    }
    *out = h;
    return GBENV_OK;
}

static int create_impl(gbenv *&h, int n_envs, const uint8_t *rom_host, size_t rom_len, int device_id) {
    if (n_envs <= 0 || !rom_host || rom_len < 0x8000 || (rom_len & 0x3FFF)) return fail(nullptr, GBENV_E_ARG, "gbenv_create: bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(nullptr, GBENV_E_CUDA, "gbenv_create: no CUDA device (this library has no CPU fallback)");
    if (device_id < 0 || device_id >= ndev) return fail(nullptr, GBENV_E_ARG, "gbenv_create: bad device id");
    CK(cudaSetDevice(device_id));
    h = new gbenv();
    h->n = n_envs;
    h->n_tiles = (n_envs + GB_TILE - 1) / GB_TILE;
    h->device = device_id;
    h->initial_template.assign(n_envs, -1);
#define ALLOC(ptr, bytes)                                              \
    do {                                                               \
        if (cudaMalloc((void **)&(ptr), (bytes)) != cudaSuccess) {     \
            h->err = "gbenv_create: cudaMalloc failed for " #ptr;      \
            return GBENV_E_NOMEM;                                      \
        }                                                              \
        cudaMemset((ptr), 0, (bytes));                                 \
    } while (0)
    size_t T = (size_t)h->n_tiles * GB_TILE * sizeof(uint32_t);
    ALLOC(h->d.mem, T * MEM_WORDS);
    ALLOC(h->d.cram, T * CRAM_WORDS);
    ALLOC(h->d.fb, T * FB_WORDS);
    ALLOC(h->d.lp, T * LP_WORDS);
    ALLOC(h->d.dl, T * DL_WORDS);  // deferred-line records (scratch between k_run_frames and k_render_pending)
    ALLOC(h->d.regs, T * R_WORDS);
    uint8_t *d_rom = nullptr;
    ALLOC(d_rom, rom_len + 16);  // padded: the instruction fetch reads two aligned words
    h->d.rom = d_rom;
    uint4 *d_rom_dec = nullptr;
    ALLOC(d_rom_dec, rom_len * sizeof(uint4));
    h->d.rom_dec = d_rom_dec;
    h->d.rom_banks = (uint32_t)(rom_len / 0x4000);
    h->d.n_envs = n_envs;
    h->d.n_tiles = h->n_tiles;
    {   // envs per warp: the interpreter is latency-bound, so spread the batch over as many warps as are resident
        // at once (one wave: SMs x STEP_MIN_BLOCKS blocks) and no more; GBENV_LANES / gbenv_set_lanes_per_warp override.
        int sms = 148;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device_id);
        const int resident_warps = sms * 32;  // warp slots the policy was tuned with (16 two-warp blocks per SM; 32 single-thread blocks)
        // measured on B200 (tools/quick_bench.sh): the smallest power of two that keeps every warp resident wins; counts
        // that are not powers of two make warps straddle 32-env tiles (partial 128-byte lines) and lose 3-5 %
        // and past one env per warp, the next power of two (half a wave of warps) wins: 8,192 envs 198 k env-steps/s at 4
        // lanes vs 181 k at 2; 16,384: 339 k at 8 vs 304 k at 4; 32,768: 578 k at 16 vs 522 k at 8; 65,536: 957 k at 32 vs 924 k at 16
        int lanes = 1;
        if (n_envs > resident_warps)
            while (lanes < 32 && (n_envs + lanes - 1) / lanes > resident_warps / 2) lanes <<= 1;
        if (const char *ev = getenv("GBENV_LANES")) {
            int v = atoi(ev);
            if (v >= 1 && v <= 32) lanes = v;
        }
        h->lanes = lanes;
        if (const char *ev = getenv("GBENV_DEFER")) h->defer = atoi(ev) != 0;
    }
    ALLOC(h->w.state, sizeof(WrapState) * (size_t)n_envs);
    {   // exploration storage (gb_wrap.cuh): page tables / directories per env, pages and blocks from shared pools.  A pool
        // holds everything the batch could ever use when that fits its budget (8 GiB of 2 KiB bitmap pages, 4 GiB of 1 KiB
        // heat-map blocks), otherwise the budget: e.g. 32,768 envs share 4.2 M bitmap pages -- 128 per env on average, all
        // 992 for any one of them.  GBENV_VISITED_PAGES / GBENV_COUNTS_BLOCKS override the pool sizes (tests);
        // GBENV_COUNTS_MAP=0 switches the heat maps off.
        size_t pages = (size_t)n_envs * VIS_PT_ENTRIES, max_pages = ((size_t)8 << 30) / (VIS_PAGE_WORDS * 4);
        if (pages > max_pages) pages = max_pages;
        if (const char *ev = getenv("GBENV_VISITED_PAGES")) {
            long v = atol(ev);
            if (v >= 1 && (size_t)v <= max_pages) pages = (size_t)v;
        }
        h->w.vis_pages = (int)pages;
        ALLOC(h->w.vis_pt, (size_t)n_envs * VIS_PT_ENTRIES * sizeof(uint32_t));
        ALLOC(h->w.vis_pool, pages * VIS_PAGE_WORDS * sizeof(uint32_t));
        ALLOC(h->w.vis_free, pages * sizeof(int32_t));
        ALLOC(h->w.ctl, 8 * sizeof(int32_t));
        bool heat = true;
        if (const char *ev = getenv("GBENV_COUNTS_MAP")) heat = strcmp(ev, "0") != 0;
        if (heat) {
            size_t blocks = (size_t)n_envs * CM_DIR_ENTRIES, max_blocks = ((size_t)4 << 30) / (CM_BLOCK * CM_BLOCK * 4);
            if (blocks > max_blocks) blocks = max_blocks;
            if (const char *ev = getenv("GBENV_COUNTS_BLOCKS")) {
                long v = atol(ev);
                if (v >= 1 && (size_t)v <= max_blocks) blocks = (size_t)v;
            }
            h->w.cm_blocks = (int)blocks;
            ALLOC(h->w.cm_dir, (size_t)n_envs * CM_DIR_ENTRIES * sizeof(uint32_t));
            ALLOC(h->w.cm_pool, blocks * CM_BLOCK * CM_BLOCK * sizeof(int32_t));
        }
    }
    ALLOC(h->d_counters, 8 * sizeof(unsigned long long));
    ALLOC(h->d_stage_image, IMG_WORDS * sizeof(uint32_t));
    ALLOC(h->d_stage_blob, GBENV_STATE_BYTES);
    ALLOC(h->d_load_claim, (size_t)n_envs * sizeof(unsigned long long));
    ALLOC(h->d_stage_buf, 0x10000);
    ALLOC(h->d_info_rows, (size_t)n_envs * GBENV_INFO_SCALARS * sizeof(double));
    ALLOC(h->d_env_ids, (size_t)n_envs * sizeof(int32_t));
    ALLOC(h->d_mask, (size_t)n_envs);
    ALLOC(h->d_init_tmpl, (size_t)n_envs * sizeof(int32_t));
    ALLOC(h->d_tmpl_images, MAX_TEMPLATES * sizeof(uint32_t *));
    ALLOC(h->d_tmpl_versions, MAX_TEMPLATES * sizeof(int32_t));
#undef ALLOC
    CK(cudaMemset(h->d_init_tmpl, 0xFF, (size_t)n_envs * sizeof(int32_t)));  // -1: no save-state to load
    CK(cudaStreamCreate(&h->stream));
    CK(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&h->ev_order, cudaEventDisableTiming));
    for (int k = 0; k < 2; k++) {
        CK(cudaEventCreateWithFlags(&h->ev_stepped[k], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_copied[k], cudaEventDisableTiming));
    }
    for (auto &slot : h->ev)
        for (auto &e : slot) CK(cudaEventCreate(&e));
    CK(cudaMemcpy(d_rom, rom_host, rom_len, cudaMemcpyHostToDevice));
    {   // decode the shared ROM once (gb_predecode.h): 16 bytes per ROM offset, L2-resident
        static uint4 base[512];
        pd_build_base(base);
        CK(cudaMemcpyToSymbol(c_base_desc, base, sizeof(base)));
        k_predecode_rom<<<(unsigned)((rom_len + 255) / 256), 256, 0, h->stream>>>(d_rom, (uint32_t)rom_len, d_rom_dec);
        CK(cudaGetLastError());
    }
    k_wrap_init<<<(n_envs + 127) / 128, 128, 0, h->stream>>>(h->w, n_envs);
    k_pool_init<<<(h->w.vis_pages + 255) / 256, 256, 0, h->stream>>>(h->w);
    CK(cudaGetLastError());
    CK(cudaHostAlloc((void **)&h->pool_err_host, sizeof(int32_t), cudaHostAllocDefault));
    *h->pool_err_host = 0;
    std::vector<uint32_t> img;
    power_on_image(img);
    CK(cudaMemcpyAsync(h->d_stage_image, img.data(), IMG_WORDS * 4, cudaMemcpyHostToDevice, h->stream));
    int rc = scatter(h, h->d_stage_image, 0 /* raw image, no load_state merge */, nullptr, 0, h->stream);
    if (rc) return rc;
    CK(cudaStreamSynchronize(h->stream));
    return GBENV_OK;
}

extern "C" int gbenv_set_lanes_per_warp(gbenv *h, int lanes) {
    if (!h || lanes < 1 || lanes > 32) return fail(h, GBENV_E_ARG, "gbenv_set_lanes_per_warp: lanes must be in 1..32");
    h->lanes = lanes;
    return GBENV_OK;
}

extern "C" int gbenv_get_lanes_per_warp(const gbenv *h) { return h ? h->lanes : GBENV_E_ARG; }

extern "C" int gbenv_sync(gbenv *h) {
    if (!h) return GBENV_E_ARG;
    CK(cudaSetDevice(h->device));
    own(h);  // ordered after whatever was last queued on this handle, on any stream
    CK(cudaStreamSynchronize(h->stream));
    return GBENV_OK;
}

// ------------------------------------------------------------------------------- templates / state

extern "C" int gbenv_add_state_template(gbenv *h, const uint8_t *blob, size_t len, int *id_out) {
    if (!h || !blob || !id_out) return fail(h, GBENV_E_ARG, "gbenv_add_state_template: bad argument");
    CK(cudaSetDevice(h->device));
    std::vector<uint32_t> img;
    int ver = 0;
    std::string err;
    int rc = blob_to_image(blob, len, img, &ver, err);
    if (rc) return fail(h, rc, err.c_str());
    if ((int)h->templates.size() >= MAX_TEMPLATES) return fail(h, GBENV_E_ARG, "gbenv_add_state_template: too many templates");
    StateTemplate t{nullptr, ver};
    CK(cudaMalloc((void **)&t.d_image, IMG_WORDS * sizeof(uint32_t)));
    CK(cudaMemcpy(t.d_image, img.data(), IMG_WORDS * sizeof(uint32_t), cudaMemcpyHostToDevice));
    h->templates.push_back(t);
    h->tmpl_dirty = true;
    *id_out = (int)h->templates.size() - 1;
    return GBENV_OK;
}

extern "C" int gbenv_load_template(gbenv *h, const int32_t *env_ids, int n, int tid) {
    if (!h || tid < 0 || tid >= (int)h->templates.size()) return fail(h, GBENV_E_ARG, "gbenv_load_template: bad template id");
    CK(cudaSetDevice(h->device));
    own(h);  // ordered after whatever was last queued on this handle, on any stream
    return scatter(h, h->templates[tid].d_image, h->templates[tid].version, env_ids, n, h->stream);
}

extern "C" int gbenv_set_initial_template(gbenv *h, const int32_t *env_ids, int n, int tid) {
    if (!h || tid < 0 || tid >= (int)h->templates.size()) return fail(h, GBENV_E_ARG, "gbenv_set_initial_template: bad template id");
    if (env_ids) {
        for (int i = 0; i < n; i++) {
            if (env_ids[i] < 0 || env_ids[i] >= h->n) return fail(h, GBENV_E_ARG, "env id out of range");
            h->initial_template[env_ids[i]] = tid;
        }
    } else {
        for (auto &t : h->initial_template) t = tid;
    }
    h->tmpl_dirty = true;
    h->loads_pending = true;
    return GBENV_OK;
}

extern "C" int gbenv_power_on(gbenv *h, const int32_t *env_ids, int n) {
    if (!h) return GBENV_E_ARG;
    CK(cudaSetDevice(h->device));
    own(h);  // ordered after whatever was last queued on this handle, on any stream
    // a power-on is a complete re-initialisation: unlike a state load it also resets STAT mode / ly_window
    std::vector<uint32_t> img;
    power_on_image(img);
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpyAsync(h->d_stage_image, img.data(), IMG_WORDS * 4, cudaMemcpyHostToDevice, h->stream));
    return scatter(h, h->d_stage_image, 0 /* version 0 = raw, no merge */, env_ids, n, h->stream);
}

// gbenv_save_states for one env on the handle's stream, then to the host
extern "C" int gbenv_save_state(gbenv *h, int env, uint8_t *blob) {
    if (!h || env < 0 || env >= h->n || !blob) return fail(h, GBENV_E_ARG, "gbenv_save_state: bad argument");
    CK(cudaSetDevice(h->device));
    CK(launch_save_states(h->d, nullptr, env, 1, h->d_stage_blob, own(h)));
    h->launches++;
    CK(cudaMemcpyAsync(blob, h->d_stage_blob, GBENV_STATE_BYTES, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return GBENV_OK;
}

extern "C" int gbenv_save_states(gbenv *h, const int32_t *env_ids_dev, int n, uint8_t *blobs_dev, void *stream) {
    if (!h || n < 0 || (!env_ids_dev && n > h->n) || (n && !blobs_dev) || ((uintptr_t)blobs_dev & 15) || ((uintptr_t)env_ids_dev & 3))
        return fail(h, GBENV_E_ARG, "gbenv_save_states: bad argument (NULL or misaligned buffer, n < 0, or NULL ids with n > n_envs)");
    if (n == 0) return GBENV_OK;
    CK(cudaSetDevice(h->device));
    CK(launch_save_states(h->d, env_ids_dev, 0, n, blobs_dev, pick(h, stream)));
    h->launches++;
    return GBENV_OK;
}

extern "C" int gbenv_load_states(gbenv *h, const int32_t *env_ids_dev, int n, const uint8_t *blobs_dev, int32_t *status_dev, void *stream) {
    if (!h || n < 0 || (!env_ids_dev && n > h->n) || (n && !blobs_dev) || ((uintptr_t)blobs_dev & 15) || ((uintptr_t)env_ids_dev & 3) ||
        ((uintptr_t)status_dev & 3))
        return fail(h, GBENV_E_ARG, "gbenv_load_states: bad argument (NULL or misaligned buffer, n < 0, or NULL ids with n > n_envs)");
    if (n == 0) return GBENV_OK;
    CK(cudaSetDevice(h->device));
    cudaStream_t st = pick(h, stream);
    if (++h->load_calls == 0) {  // the call counter wrapped: older keys would outrank the new ones
        CK(cudaMemsetAsync(h->d_load_claim, 0, (size_t)h->n * sizeof(unsigned long long), st));
        h->load_calls = 1;
    }
    CK(launch_load_states(h->d, env_ids_dev, n, blobs_dev, status_dev, h->d_load_claim, h->load_calls, st));
    h->launches += 2;
    return GBENV_OK;
}

// ------------------------------------------------------------------------------- emulator

// deferred PPU, second half: the lines the emulation kernel recorded are drawn with one thread per (env, line slot)
static int launch_render(gbenv *h, const RunParams &p, cudaStream_t st) {
    if (!p.defer) return GBENV_OK;
    k_render_pending<<<dim3(h->n_tiles, 144 / RENDER_LINES_PER_BLOCK), dim3(32, RENDER_LINES_PER_BLOCK), 0, st>>>(p.d, p.skip);
    h->launches++;
    CK(cudaGetLastError());
    return GBENV_OK;
}

static int launch_run(gbenv *h, const uint8_t *actions_dev, int n_frames, int render_mode, cudaStream_t st, const uint8_t *skip_dev = nullptr) {
    RunParams p;
    p.d = h->d;
    p.actions = actions_dev;
    p.skip = skip_dev;
    p.n_frames = n_frames;
    p.render_mode = render_mode;
    p.release_frame = 8;
    p.counters = h->d_counters;
    p.lanes = h->lanes;
    p.defer = h->defer && render_mode != 0;
    p.bank_mask = (h->d.rom_banks & (h->d.rom_banks - 1)) == 0 ? h->d.rom_banks - 1 : 0;
    if (h->lanes == 1) {  // one env per warp: the single-thread-block build of the same kernel
        k_run_frames_1<<<h->n, 1, ENV_SMEM_BYTES(1), st>>>(p);
        h->launches++;
        CK(cudaGetLastError());
        return launch_render(h, p, st);
    }
    int warps = (h->n + h->lanes - 1) / h->lanes;
    int blocks = (warps * 32 + STEP_THREADS - 1) / STEP_THREADS;
    size_t smem = ENV_SMEM_BYTES((STEP_THREADS / 32) * h->lanes);
    if (smem > h->smem_opted) {  // beyond the 48 KiB default: opt in once per size
        CK(cudaFuncSetAttribute(k_run_frames, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        h->smem_opted = smem;
    }
    k_run_frames<<<blocks, STEP_THREADS, smem, st>>>(p);
    h->launches++;
    CK(cudaGetLastError());
    return launch_render(h, p, st);
}

extern "C" int gbenv_run_action(gbenv *h, const uint8_t *actions_dev, int frame_skip, void *stream) {
    if (!h || !actions_dev || frame_skip <= 0) return fail(h, GBENV_E_ARG, "gbenv_run_action: bad argument");
    CK(cudaSetDevice(h->device));
    return launch_run(h, actions_dev, frame_skip, 2, pick(h, stream));
}

extern "C" int gbenv_tick(gbenv *h, int n_frames, int render, void *stream) {
    if (!h || n_frames <= 0) return fail(h, GBENV_E_ARG, "gbenv_tick: bad argument");
    CK(cudaSetDevice(h->device));
    return launch_run(h, nullptr, n_frames, render ? 1 : 0, pick(h, stream));
}

extern "C" int gbenv_send_input(gbenv *h, int button, int pressed, void *stream) {
    if (!h || button < 0 || button > 7) return fail(h, GBENV_E_ARG, "gbenv_send_input: bad argument");
    CK(cudaSetDevice(h->device));
    k_send_input<<<(h->n + 127) / 128, 128, 0, pick(h, stream)>>>(h->d, button, pressed);
    h->launches++;
    CK(cudaGetLastError());
    return GBENV_OK;
}

static int bus_access(gbenv *h, int env, uint32_t addr, uint32_t n, uint8_t *host, int write) {
    if (!h || env < 0 || env >= h->n || !host || addr + n > 0x10000 || n == 0) return fail(h, GBENV_E_ARG, "bus access: bad argument");
    CK(cudaSetDevice(h->device));
    own(h);
    if (write) CK(cudaMemcpyAsync(h->d_stage_buf, host, n, cudaMemcpyHostToDevice, h->stream));
    k_bus_access<<<1, 1, 0, h->stream>>>(h->d, env, addr, n, h->d_stage_buf, write);
    h->launches++;
    CK(cudaGetLastError());
    if (!write) CK(cudaMemcpyAsync(host, h->d_stage_buf, n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return GBENV_OK;
}

extern "C" int gbenv_read_mem(gbenv *h, int env, uint32_t addr, uint32_t n, uint8_t *out) { return bus_access(h, env, addr, n, out, 0); }
extern "C" int gbenv_write_mem(gbenv *h, int env, uint32_t addr, uint32_t n, const uint8_t *in) {
    return bus_access(h, env, addr, n, (uint8_t *)in, 1);
}

extern "C" int gbenv_screen(gbenv *h, int env, uint8_t *rgb) {
    if (!h || env < 0 || env >= h->n || !rgb) return fail(h, GBENV_E_ARG, "gbenv_screen: bad argument");
    CK(cudaSetDevice(h->device));
    own(h);  // ordered after whatever was last queued on this handle, on any stream
    k_gather_image<<<(IMG_WORDS + 255) / 256, 256, 0, h->stream>>>(h->d, h->d_stage_image, env);
    h->launches++;
    CK(cudaGetLastError());
    std::vector<uint32_t> fb(FB_WORDS);
    CK(cudaMemcpyAsync(fb.data(), h->d_stage_image + IMG_FB, FB_WORDS * 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    static const uint8_t grey[4] = {0xFF, 0x99, 0x55, 0x00};
    for (uint32_t i = 0; i < 144 * 160; i++) {
        uint8_t g = grey[(fb[i >> 4] >> (2 * (i & 15))) & 3];
        rgb[3 * i] = rgb[3 * i + 1] = rgb[3 * i + 2] = g;
    }
    return GBENV_OK;
}

extern "C" int gbenv_capture_frames(gbenv *h, const int32_t *env_ids_dev, int n, uint32_t *frames_dev, void *stream) {
    if (!h || n < 0 || (!env_ids_dev && n > h->n) || (n && !frames_dev) || ((uintptr_t)frames_dev & 3) || ((uintptr_t)env_ids_dev & 3))
        return fail(h, GBENV_E_ARG, "gbenv_capture_frames: bad argument (NULL or misaligned buffer, n < 0, or NULL ids with n > n_envs)");
    if (n == 0) return GBENV_OK;
    CK(cudaSetDevice(h->device));
    CK(launch_frames_capture(h->d.fb, env_ids_dev, n, h->n, frames_dev, pick(h, stream)));
    h->launches++;
    return GBENV_OK;
}

extern "C" int gbenv_frames_to_rgb(gbenv *h, const uint32_t *frames_dev, int n_frames, int channels, uint8_t *out_dev, void *stream) {
    if (!h || n_frames < 0 || (channels != 1 && channels != 3) || (n_frames && (!frames_dev || !out_dev)) || ((uintptr_t)frames_dev & 3) ||
        ((uintptr_t)out_dev & 15))
        return fail(h, GBENV_E_ARG, "gbenv_frames_to_rgb: bad argument (NULL or misaligned buffer, n_frames < 0, or channels not 1 or 3)");
    if (n_frames == 0) return GBENV_OK;
    CK(cudaSetDevice(h->device));
    CK(launch_frames_to_rgb(frames_dev, n_frames, channels, out_dev, pick(h, stream)));
    h->launches++;
    return GBENV_OK;
}

extern "C" int gbenv_event_flags(gbenv *h, const int32_t *env_ids_dev, int n, uint32_t *flags_dev, void *stream) {
    if (!h || n < 0 || (!env_ids_dev && n > h->n) || (n && !flags_dev) || ((uintptr_t)flags_dev & 3) || ((uintptr_t)env_ids_dev & 3))
        return fail(h, GBENV_E_ARG, "gbenv_event_flags: bad argument (NULL or misaligned buffer, n < 0, or NULL ids with n > n_envs)");
    if (n == 0) return GBENV_OK;
    CK(cudaSetDevice(h->device));
    CK(launch_event_flags(h->d.mem, env_ids_dev, n, h->n, flags_dev, pick(h, stream)));
    h->launches++;
    return GBENV_OK;
}

// ------------------------------------------------------------------------------- Environment API

// environment.py:1241-1242: the save-state is loaded on an env's FIRST reset only.  Which envs that concerns is decided on
// the device (WrapState.reset_count == 0 and a template assigned), so a reset never needs the host to look at per-env data.
// grid: (ceil(n / 32), ceil(IMG_WORDS / 8)); block (32, 8) as k_scatter_image
__global__ void k_reset_load(DevArrays d, const WrapState *st, const int32_t *init_tmpl, uint32_t *const *tmpl_images, const int32_t *tmpl_versions,
                             const uint8_t *mask, int n) {
    int env = blockIdx.x * 32 + threadIdx.x;
    uint32_t j = blockIdx.y * 8 + threadIdx.y;
    if (env >= n || j >= IMG_WORDS || (mask && !mask[env])) return;
    int tid = init_tmpl[env];
    if (tid < 0 || st[env].reset_count != 0) return;
    const uint32_t *image = tmpl_images[tid];
    uint32_t v = image[j];
    uint32_t *slot = image_slot(d, env, j);
    if (j >= IMG_REGS) v = merge_loaded_reg(j - IMG_REGS, *slot, v, tmpl_versions[tid], image[IMG_REGS + R_LCD0] & 0xFF);
    *slot = v;
}

static int upload_template_tables(gbenv *h, cudaStream_t st) {
    if (!h->tmpl_dirty) return GBENV_OK;
    std::vector<uint32_t *> ptrs(h->templates.size());
    std::vector<int32_t> vers(h->templates.size());
    for (size_t i = 0; i < h->templates.size(); i++) { ptrs[i] = h->templates[i].d_image; vers[i] = h->templates[i].version; }
    std::vector<int32_t> init(h->initial_template.begin(), h->initial_template.end());
    // pageable host vectors: these copies return after the data has been staged, so the vectors may go out of scope
    if (!ptrs.empty()) {
        CK(cudaMemcpyAsync(h->d_tmpl_images, ptrs.data(), ptrs.size() * sizeof(uint32_t *), cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(h->d_tmpl_versions, vers.data(), vers.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    }
    CK(cudaMemcpyAsync(h->d_init_tmpl, init.data(), init.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st));
    h->tmpl_dirty = false;
    return GBENV_OK;
}

// Where a step or a reset puts the observation: reference rows (obs, stride) by k_wrap_obs, or packed rows (packed non-null)
// by k_obs_pack.  The rows of the envs with mask[e] != 0 are written (== 0 when `invert` is set; mask null: all).
struct ObsOut {
    uint8_t *obs;
    size_t stride;
    uint32_t *packed;
};

static void launch_obs(gbenv *h, const ObsOut &o, const uint8_t *mask, int invert, cudaStream_t st) {
    if (o.packed)
        launch_obs_pack(h->d.mem, h->d.fb, h->w.vis_pt, h->w.vis_pool, h->n, h->n_tiles, mask, invert, o.packed, st);
    else
        k_wrap_obs<<<h->n_tiles, 256, 0, st>>>(h->d, h->w, mask, o.obs, o.stride, invert);
}

// Environment.reset for the envs with mask_dev[e] != 0 (mask_dev == NULL: all), everything on the device, asynchronous.
static int reset_impl(gbenv *h, const uint8_t *mask_dev, int max_episode_steps, double reward_scale, const ObsOut &o, void *stream) {
    CK(cudaSetDevice(h->device));
    cudaStream_t st = pick(h, stream);
    int rc = pool_error(h);
    if (rc) return rc;
    rc = upload_template_tables(h, st);
    if (rc) return rc;
    int blocks = (h->n + 127) / 128;
    k_wrap_reset_pre<<<blocks, 128, 0, st>>>(h->d, h->w, mask_dev);  // environment.py:1239: D778 |= 0x10 before the load
    h->launches++;
    if (h->loads_pending) {
        dim3 block(32, 8), grid((h->n + 31) / 32, (IMG_WORDS + 7) / 8);
        k_reset_load<<<grid, block, 0, st>>>(h->d, h->w.state, h->d_init_tmpl, h->d_tmpl_images, h->d_tmpl_versions, mask_dev, h->n);
        h->launches++;
        if (!mask_dev) h->loads_pending = false;  // every env has had its first reset now
    }
    k_vis_release<<<h->n, 256, 0, st>>>(h->w, mask_dev, h->n);  // the envs' bitmap pages go back to the pool
    k_wrap_reset_post<<<blocks, 128, 0, st>>>(h->d, h->w, mask_dev, max_episode_steps, reward_scale);
    launch_obs(h, o, mask_dev, 0, st);
    h->launches += 3;
    CK(cudaGetLastError());
    queue_pool_error_copy(h, st);
    return GBENV_OK;
}

extern "C" int gbenv_reset_dev(gbenv *h, const uint8_t *mask_dev, int max_episode_steps, double reward_scale, uint8_t *obs_dev, size_t obs_stride,
                               void *stream) {
    if (!h || !obs_dev || obs_stride < GBENV_OBS_BYTES || (obs_stride & 3)) return fail(h, GBENV_E_ARG, "gbenv_reset: bad argument");
    return reset_impl(h, mask_dev, max_episode_steps, reward_scale, ObsOut{obs_dev, obs_stride, nullptr}, stream);
}

extern "C" int gbenv_reset_packed(gbenv *h, const uint8_t *mask_dev, int max_episode_steps, double reward_scale, uint32_t *packed_dev, void *stream) {
    if (!h || !packed_dev || ((uintptr_t)packed_dev & 15)) return fail(h, GBENV_E_ARG, "gbenv_reset_packed: bad argument (NULL or misaligned buffer)");
    return reset_impl(h, mask_dev, max_episode_steps, reward_scale, ObsOut{nullptr, 0, packed_dev}, stream);
}

extern "C" int gbenv_reset(gbenv *h, const uint8_t *mask_host, int max_episode_steps, double reward_scale, uint8_t *obs_dev, size_t obs_stride,
                           void *stream) {
    if (!h) return GBENV_E_ARG;
    if (!mask_host) return gbenv_reset_dev(h, nullptr, max_episode_steps, reward_scale, obs_dev, obs_stride, stream);
    CK(cudaSetDevice(h->device));
    cudaStream_t st = pick(h, stream);
    CK(cudaMemcpyAsync(h->d_mask, mask_host, h->n, cudaMemcpyHostToDevice, st));
    int rc = gbenv_reset_dev(h, h->d_mask, max_episode_steps, reward_scale, obs_dev, obs_stride, stream);
    if (rc) return rc;
    CK(cudaStreamSynchronize(st));  // d_mask is reused by the next call
    return GBENV_OK;
}

// accumulate the device time of recorded steps [ev_folded, upto) into ms_total (blocks on their events)
static int fold_events(gbenv *h, unsigned long long upto) {
    while (h->ev_folded < upto && h->ev_folded < h->ev_step) {
        cudaEvent_t *ev = h->ev[h->ev_folded % gbenv::EV_RING];
        CK(cudaEventSynchronize(ev[2]));
        float a = 0, b = 0;
        CK(cudaEventElapsedTime(&a, ev[0], ev[1]));
        CK(cudaEventElapsedTime(&b, ev[1], ev[2]));
        h->ms_total[0] += a;
        h->ms_total[1] += b;
        h->ev_folded++;
    }
    return GBENV_OK;
}

extern "C" int gbenv_step(gbenv *h, const uint8_t *actions_dev, uint8_t *obs_dev, size_t obs_stride, double *reward_dev, uint8_t *done_dev,
                          void *stream) {
    return gbenv_step_masked(h, actions_dev, nullptr, obs_dev, obs_stride, reward_dev, done_dev, stream);
}

// Environment.step for the envs with skip_dev[e] == 0 (null: all).  A skipped env is not emulated, its wrapper state, info row
// and observation row stay as they are, and it reports reward 0 / done 0.
static int step_impl(gbenv *h, const uint8_t *actions_dev, const uint8_t *skip_dev, const ObsOut &o, double *reward_dev, uint8_t *done_dev,
                     void *stream) {
    CK(cudaSetDevice(h->device));
    {
        int rce = pool_error(h);
        if (rce) return rce;
    }
    cudaStream_t st = pick(h, stream);
    if (h->ev_step - h->ev_folded >= (unsigned long long)gbenv::EV_RING) {  // slot about to be reused: fold it first
        int rcf = fold_events(h, h->ev_folded + 1);
        if (rcf) return rcf;
    }
    cudaEvent_t *ev = h->ev[h->ev_step % gbenv::EV_RING];
    CK(cudaEventRecord(ev[0], st));
    int rc = launch_run(h, actions_dev, GBENV_ACT_FREQ, 2, st, skip_dev);
    if (rc) return rc;
    CK(cudaEventRecord(ev[1], st));
    int blocks = (h->n_tiles * GB_TILE + 127) / 128;
    k_wrap_step<<<blocks, 128, 0, st>>>(h->d, h->w, reward_dev, done_dev, h->d_info_rows, skip_dev);
    launch_obs(h, o, skip_dev, 1, st);
    h->launches += 2;
    CK(cudaGetLastError());
    CK(cudaEventRecord(ev[2], st));
    queue_pool_error_copy(h, st);
    h->ev_step++;
    h->ev_valid = true;
    return GBENV_OK;
}

extern "C" int gbenv_step_masked(gbenv *h, const uint8_t *actions_dev, const uint8_t *skip_dev, uint8_t *obs_dev, size_t obs_stride, double *reward_dev,
                                 uint8_t *done_dev, void *stream) {
    if (!h || !actions_dev || !obs_dev || !reward_dev || !done_dev || obs_stride < GBENV_OBS_BYTES || (obs_stride & 3))
        return fail(h, GBENV_E_ARG, "gbenv_step: bad argument");
    return step_impl(h, actions_dev, skip_dev, ObsOut{obs_dev, obs_stride, nullptr}, reward_dev, done_dev, stream);
}

extern "C" int gbenv_step_packed(gbenv *h, const uint8_t *actions_dev, const uint8_t *skip_dev, uint32_t *packed_dev, double *reward_dev,
                                 uint8_t *done_dev, void *stream) {
    if (!h || !actions_dev || !packed_dev || !reward_dev || !done_dev || ((uintptr_t)packed_dev & 15))
        return fail(h, GBENV_E_ARG, "gbenv_step_packed: bad argument (NULL or misaligned buffer)");
    return step_impl(h, actions_dev, skip_dev, ObsOut{nullptr, 0, packed_dev}, reward_dev, done_dev, stream);
}

extern "C" int gbenv_unpack_obs(gbenv *h, const uint32_t *packed_dev, int n, uint8_t *out_dev, void *stream) {
    if (!h || n < 0 || (n && (!packed_dev || !out_dev)) || ((uintptr_t)packed_dev & 15) || ((uintptr_t)out_dev & 15))
        return fail(h, GBENV_E_ARG, "gbenv_unpack_obs: bad argument (NULL or misaligned buffer, or n < 0)");
    if (n == 0) return GBENV_OK;
    CK(cudaSetDevice(h->device));
    CK(launch_obs_unpack(packed_dev, n, out_dev, pick(h, stream)));
    h->launches++;
    return GBENV_OK;
}

static int ensure_host_staging(gbenv *h) {
    if (h->d_actions[0]) return GBENV_OK;
    for (int k = 0; k < 2; k++) {
        CK(cudaMalloc((void **)&h->d_actions[k], h->n));
        CK(cudaMalloc((void **)&h->d_obs[k], (size_t)h->n * GBENV_OBS_BYTES));
        CK(cudaMalloc((void **)&h->d_done[k], h->n));
        CK(cudaMalloc((void **)&h->d_reward[k], (size_t)h->n * sizeof(double)));
    }
    return GBENV_OK;
}

// Queues one Environment.step with HOST buffers and returns at once: actions H2D, the three kernels, then -- on a second
// stream -- obs / reward / done D2H into the caller's buffers.  gbenv_fetch_host blocks until the OLDEST queued step has
// landed.  At most two steps may be in flight (two device staging slots), which is what lets the 23 KB-per-env observation
// copy of step t overlap the emulation of step t+1.
extern "C" int gbenv_submit_host(gbenv *h, const uint8_t *actions, uint8_t *obs, double *reward, uint8_t *done) {
    if (!h || !actions || !obs || !reward || !done) return fail(h, GBENV_E_ARG, "gbenv_submit_host: bad argument");
    if (h->submitted - h->fetched >= 2) return fail(h, GBENV_E_ARG, "gbenv_submit_host: two steps already in flight, fetch one first");
    CK(cudaSetDevice(h->device));
    int rc = ensure_host_staging(h);
    if (rc) return rc;
    const int k = (int)(h->submitted & 1);
    cudaStream_t st = own(h);
    CK(cudaStreamWaitEvent(st, h->ev_copied[k], 0));  // slot k's previous results have left the device
    CK(cudaMemcpyAsync(h->d_actions[k], actions, h->n, cudaMemcpyHostToDevice, st));
    rc = gbenv_step(h, h->d_actions[k], h->d_obs[k], GBENV_OBS_BYTES, h->d_reward[k], h->d_done[k], st);
    if (rc) return rc;
    CK(cudaEventRecord(h->ev_stepped[k], st));
    CK(cudaStreamWaitEvent(h->copy_stream, h->ev_stepped[k], 0));
    CK(cudaMemcpyAsync(obs, h->d_obs[k], (size_t)h->n * GBENV_OBS_BYTES, cudaMemcpyDeviceToHost, h->copy_stream));
    CK(cudaMemcpyAsync(reward, h->d_reward[k], (size_t)h->n * sizeof(double), cudaMemcpyDeviceToHost, h->copy_stream));
    CK(cudaMemcpyAsync(done, h->d_done[k], h->n, cudaMemcpyDeviceToHost, h->copy_stream));
    CK(cudaEventRecord(h->ev_copied[k], h->copy_stream));
    h->submitted++;
    return GBENV_OK;
}

extern "C" int gbenv_fetch_host(gbenv *h) {
    if (!h) return GBENV_E_ARG;
    if (h->fetched == h->submitted) return fail(h, GBENV_E_ARG, "gbenv_fetch_host: nothing in flight");
    CK(cudaSetDevice(h->device));
    CK(cudaEventSynchronize(h->ev_copied[h->fetched & 1]));
    h->fetched++;
    return GBENV_OK;
}

// Same call, synchronous: copies in, steps, copies out.  This is the entry point a pokegym worker would call.
extern "C" int gbenv_step_host(gbenv *h, const uint8_t *actions, uint8_t *obs, double *reward, uint8_t *done) {
    if (!h) return GBENV_E_ARG;
    while (h->fetched < h->submitted) {
        int rc = gbenv_fetch_host(h);
        if (rc) return rc;
    }
    int rc = gbenv_submit_host(h, actions, obs, reward, done);
    if (rc) return rc;
    return gbenv_fetch_host(h);
}

extern "C" int gbenv_reset_host(gbenv *h, const uint8_t *mask, int max_episode_steps, double reward_scale, uint8_t *obs) {
    if (!h || !obs) return fail(h, GBENV_E_ARG, "gbenv_reset_host: bad argument");
    CK(cudaSetDevice(h->device));
    int rc = ensure_host_staging(h);
    if (rc) return rc;
    // rows of envs that are not reset keep the caller's bytes: stage the caller's buffer in first
    while (h->fetched < h->submitted) {
        rc = gbenv_fetch_host(h);
        if (rc) return rc;
    }
    cudaStream_t st = own(h);
    if (mask) CK(cudaMemcpyAsync(h->d_obs[0], obs, (size_t)h->n * GBENV_OBS_BYTES, cudaMemcpyHostToDevice, st));
    rc = gbenv_reset(h, mask, max_episode_steps, reward_scale, h->d_obs[0], GBENV_OBS_BYTES, st);
    if (rc) return rc;
    CK(cudaMemcpyAsync(obs, h->d_obs[0], (size_t)h->n * GBENV_OBS_BYTES, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return GBENV_OK;
}

extern "C" int gbenv_get_info(gbenv *h, double *info_dev, void *stream) {
    if (!h || !info_dev) return fail(h, GBENV_E_ARG, "gbenv_get_info: bad argument");
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(info_dev, h->d_info_rows, (size_t)h->n * GBENV_INFO_SCALARS * sizeof(double), cudaMemcpyDeviceToDevice, pick(h, stream)));
    return GBENV_OK;
}

extern "C" int gbenv_reduce_info_masked(gbenv *h, const uint8_t *mask_dev, double *sum_dev, void *stream) {
    if (!h || !sum_dev) return fail(h, GBENV_E_ARG, "gbenv_reduce_info: bad argument");
    CK(cudaSetDevice(h->device));
    k_reduce_info<<<GBENV_INFO_SCALARS, 256, 0, pick(h, stream)>>>(h->d_info_rows, mask_dev, h->n, sum_dev);
    h->launches++;
    CK(cudaGetLastError());
    return GBENV_OK;
}

extern "C" int gbenv_reduce_info(gbenv *h, double *sum_dev, void *stream) { return gbenv_reduce_info_masked(h, nullptr, sum_dev, stream); }

static const char *const CM_DISABLED = "gbenv_counts_map: exploration map tracking is disabled (GBENV_COUNTS_MAP=0)";

extern "C" int gbenv_counts_map_sum(gbenv *h, const uint8_t *mask_dev, int64_t *sum_dev, void *stream) {
    if (!h || !sum_dev) return fail(h, GBENV_E_ARG, "gbenv_counts_map_sum: bad argument");
    if (!h->w.cm_dir) return fail(h, GBENV_E_ARG, CM_DISABLED);
    CK(cudaSetDevice(h->device));
    int rc = pool_error(h);  // a sum over maps that stopped being tracked would look valid
    if (rc) return rc;
    if (!h->cm_sum_chunk) {
        // env chunks: enough blocks for four waves of the GPU, but at least 1,024 envs per chunk so that a block's reads of
        // the maps outweigh its 256 atomics into the sum
        int sms = 148, per_sm = 1;
        CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device));
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_cm_sum, CM_SUM_THREADS, 0));
        const int wanted = (4 * sms * per_sm + CM_DIR_ENTRIES - 1) / CM_DIR_ENTRIES, most = (h->n + 1023) / 1024;
        const int chunks = wanted < most ? (wanted > 1 ? wanted : 1) : most;
        h->cm_sum_chunk = ((h->n + chunks - 1) / chunks + CM_SUM_GROUP - 1) / CM_SUM_GROUP * CM_SUM_GROUP;
    }
    cudaStream_t st = pick(h, stream);
    CK(cudaMemsetAsync(sum_dev, 0, (size_t)COUNTS_H * COUNTS_W * sizeof(int64_t), st));
    const dim3 grid(CM_DIR_ENTRIES, (h->n + h->cm_sum_chunk - 1) / h->cm_sum_chunk);
    k_cm_sum<<<grid, CM_SUM_THREADS, 0, st>>>(h->w, mask_dev, h->n, h->cm_sum_chunk, (long long *)sum_dev);
    h->launches++;
    CK(cudaGetLastError());
    return GBENV_OK;
}

extern "C" int gbenv_counts_map(gbenv *h, int env, int32_t *map_host) {
    if (!h || env < 0 || env >= h->n || !map_host) return fail(h, GBENV_E_ARG, "gbenv_counts_map: bad argument");
    if (!h->w.cm_dir) return fail(h, GBENV_E_ARG, CM_DISABLED);
    CK(cudaSetDevice(h->device));
    cudaStream_t st = own(h);  // ordered after whatever was last queued on this handle, on any stream
    if (!h->d_cm_dense) CK(cudaMalloc((void **)&h->d_cm_dense, (size_t)COUNTS_H * COUNTS_W * sizeof(int32_t)));
    k_cm_gather<<<CM_DIR_ENTRIES, CM_BLOCK * CM_BLOCK, 0, st>>>(h->w, env, h->d_cm_dense);  // the env's blocks -> dense 444 x 436
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(map_host, h->d_cm_dense, (size_t)COUNTS_H * COUNTS_W * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return GBENV_OK;
}

// Blocks until everything queued on the handle is done; GBENV_E_NOMEM when a pool of the exploration storage ran dry.
extern "C" int gbenv_check(gbenv *h) {
    if (!h) return GBENV_E_ARG;
    int rc = gbenv_sync(h);
    if (rc) return rc;
    return pool_error(h);
}

// ------------------------------------------------------------------------------- diagnostics

__global__ void k_count_faults(DevArrays d, WrapArrays w, unsigned long long *out) {
    int env = blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= d.n_envs) return;
    uint32_t in = d.regs[il_index(env >> 5, R_WORDS, R_INT, env & 31)];
    if (((in >> 4) & 1) || w.state[env].overflow) atomicAdd(out, 1ull);
}

extern "C" int gbenv_get_counters(gbenv *h, gbenv_counters_t *out) {
    if (!h || !out) return fail(h, GBENV_E_ARG, "gbenv_get_counters: bad argument");
    CK(cudaSetDevice(h->device));
    own(h);  // ordered after whatever was last queued on this handle, on any stream
    CK(cudaMemsetAsync(h->d_counters + 3, 0, sizeof(unsigned long long), h->stream));
    k_count_faults<<<(h->n + 127) / 128, 128, 0, h->stream>>>(h->d, h->w, h->d_counters + 3);
    CK(cudaGetLastError());
    unsigned long long c[4];
    CK(cudaMemcpyAsync(c, h->d_counters, sizeof(c), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    out->instructions = c[0];
    out->cycles = c[1];
    out->frames = c[2];
    out->faults = c[3];
    out->kernel_launches = h->launches;
    return GBENV_OK;
}

extern "C" int gbenv_last_kernel_ms(gbenv *h, int which, float *ms) {
    if (!h || !ms || which < 0 || which > 1) return fail(h, GBENV_E_ARG, "gbenv_last_kernel_ms: bad argument");
    if (!h->ev_valid || h->ev_step == 0) return fail(h, GBENV_E_ARG, "gbenv_last_kernel_ms: no step recorded yet");
    CK(cudaSetDevice(h->device));
    cudaEvent_t *ev = h->ev[(h->ev_step - 1) % gbenv::EV_RING];
    CK(cudaEventSynchronize(ev[2]));
    CK(cudaEventElapsedTime(ms, ev[which], ev[which + 1]));
    return GBENV_OK;
}

extern "C" int gbenv_kernel_time_total(gbenv *h, int which, double *ms_total, uint64_t *steps) {
    if (!h || which < 0 || which > 1 || !ms_total || !steps) return fail(h, GBENV_E_ARG, "gbenv_kernel_time_total: bad argument");
    CK(cudaSetDevice(h->device));
    int rc = fold_events(h, h->ev_step);
    if (rc) return rc;
    *ms_total = h->ms_total[which];
    *steps = h->ev_folded;
    return GBENV_OK;
}

extern "C" int gbenv_get_core_extra(gbenv *h, int env, gbenv_core_extra_t *out) {
    if (!h || env < 0 || env >= h->n || !out) return fail(h, GBENV_E_ARG, "gbenv_get_core_extra: bad argument");
    CK(cudaSetDevice(h->device));
    own(h);  // ordered after whatever was last queued on this handle, on any stream
    CK(cudaStreamSynchronize(h->stream));
    uint32_t lcd2 = 0, joy = 0, in = 0;
    int tile = env >> 5, lane = env & 31;
    CK(cudaMemcpy(&lcd2, h->d.regs + il_index(tile, R_WORDS, R_LCD2, lane), 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(&joy, h->d.regs + il_index(tile, R_WORDS, R_JOY, lane), 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(&in, h->d.regs + il_index(tile, R_WORDS, R_INT, lane), 4, cudaMemcpyDeviceToHost));
    out->stat_mode = (lcd2 >> 24) & 3;
    out->ly_window = (int)(int8_t)((joy >> 16) & 0xFF);
    out->fault = (in >> 4) & 1;
    out->reserved = 0;
    return GBENV_OK;
}

extern "C" int gbenv_debug_render_frame(gbenv *h, int env) {
    if (!h || env < 0 || env >= h->n) return fail(h, GBENV_E_ARG, "gbenv_debug_render_frame: bad argument");
    CK(cudaSetDevice(h->device));
    own(h);  // ordered after whatever was last queued on this handle, on any stream
    k_debug_render_frame<<<1, 1, 0, h->stream>>>(h->d, env);
    h->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream));
    return GBENV_OK;
}
