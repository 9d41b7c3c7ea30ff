// api.cu — the C ABI of include/orbit_cuda.h: argument checking, scratch ownership, kernel launches.
// No torch types, no host synchronisation on the stage calls, no CPU fallback.
#include <cuda_runtime.h>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include "params.cuh"


using namespace orbit;

namespace orbit {
bool pdl_enabled() {
    // Programmatic dependent launch between the stage kernels (every kernel waits — griddepcontrol.wait — before its first
    // global access, and triggers at the end of its main work). Round 1 (profiles/r1_pdl.txt): C2 frame 1.3% faster but a
    // pass-0 sweep with 1.2M survivors 15% slower -> opt-in. Round 2, with the emit kernel's trigger after its emission and
    // the per-lane emission path (profiles/r2_pdl.txt): C2 frame 84.5 -> 83.4 us, pass-0 sweep 52.4 -> 52.2 us, C3 1220 ->
    // 1213 us, C5 185.7 -> 188.7 us per view -> on by default; ORBIT_NO_PDL=1 turns it off.
    static const bool on = std::getenv("ORBIT_NO_PDL") == nullptr;
    return on;
}
}  // namespace orbit

static thread_local int g_last_cuda_error = 0;
static constexpr size_t kViewChunkWords = 2u * 2048u;   // per view: two parities of chunk counts
static constexpr size_t kViewCounterWords = ORBIT_MAX_BATCH_VIEWS * (kViewChunkWords + 4u);
#define CK(expr)                                                       \
    do {                                                               \
        cudaError_t e_ = (expr);                                       \
        if (e_ != cudaSuccess) { g_last_cuda_error = (int)e_; return ORBIT_ERR_CUDA; } \
    } while (0)

// Makes `device` current for the duration of an entry point and restores the caller's device afterwards: a context may be
// used from any thread (the reference records its passes from rayon workers), whatever device that thread has current.
struct DeviceGuard {
    int prev = -1;
    bool ok = true;
    explicit DeviceGuard(int device) {
        int cur = -1;
        if (cudaGetDevice(&cur) != cudaSuccess) cur = -1;
        if (cur != device) { ok = cudaSetDevice(device) == cudaSuccess; prev = cur; }
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define GUARD(c) DeviceGuard guard_((c)->device); if (!guard_.ok) { g_last_cuda_error = (int)cudaGetLastError(); return ORBIT_ERR_CUDA; }

struct orbit_ctx {
    int device = 0;
    int sm_count = 0;
    // scan scratch
    unsigned long long* status = nullptr;
    size_t status_capacity = 0;       // descriptors
    uint4* main_masks = nullptr;      // record entries of the fused MAIN pass
    size_t main_mask_capacity = 0;
    unsigned int* counters = nullptr; // 32 words: [0] ticket, [1] done, [2] hiz ticket, [3] scan epoch (device-advanced), [4,5] meshlet survivor
                                      // totals per parity, [6,7] parity words A/B of the meshlet stage, [8] scene-update cursor snapshot,
                                      // [10..13] the same four words for test-only calls, [16..18] dispatch header of orbit_draws_from_masks
    // device-written status, pinned + mapped
    OrbitStatus* status_host = nullptr;
    OrbitStatus* status_dev = nullptr;
    uint32_t* chunk_counts = nullptr; // 2 x 2048 per-chunk survivor counts
    uint32_t* view_counters = nullptr;// batched views (orbit_meshlet_cull_views): 16 x 2 x 2048 chunk counts, then 16 x {survivor totals
                                      // per parity, parity words A/B} — apart from the single-view words, so both forms may interleave.
                                      // Allocated by the first batched call, never in orbit_ctx_create: an allocation there moves the
                                      // buffers created after it (the scan descriptors the entity kernel polls), and the single-view
                                      // entity stage measured ~1 us slower on C2 with its descriptors at the shifted address
    // meshlet stage scratch: one draw mask per dispatch record
    uint4* draw_masks = nullptr;
    uint4* cmd_side = nullptr;        // 32 entries per dispatch record, same capacity as draw_masks
    size_t draw_mask_capacity = 0;
    // scene-update scratch: per-tile sums (kept apart from `status`, whose words carry scan epochs)
    unsigned long long* tile_sums = nullptr;
    size_t tile_sums_capacity = 0;
    // light scratch
    float4* light_view = nullptr;
    size_t light_capacity = 0;
    uint64_t light_hits_budget = 0;   // bytes the bit matrix may take (ORBIT_LIGHT_HITS_BUDGET_MB, default 256)
    uint32_t* light_hits = nullptr;   // bit matrix [active cluster][light / 32] of the light-parallel culling path
    size_t light_hits_words = 0;
    // tuning (ORBIT_MC_CTAS_PER_SM environment override, read once)
    int mc_ctas_per_sm = 0;
    int emit_occupancy = 0;
    int debug_skip = 0;               // ORBIT_DEBUG_SKIP: 1 = skip emit kernel, 2 = skip test kernel (timing experiments only)
    int entity_occupancy = 0;
    int entity_views_occupancy[3] = {0, 0, 0};        // the same for the batched entity kernel, per pass (more registers: fewer CTAs per SM)
    int mc_occupancy[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // cached occupancy per meshlet test-kernel variant
    int views_occupancy[8] = {0, 0, 0, 0, 0, 0, 0, 0}; // the same for the batched test kernels, per variant
    int emit_ctas_per_sm = 0;         // ORBIT_EMIT_CTAS_PER_SM (tuning knob, read once at creation)
    bool views_pass2_configured = false;   // meshlet_cull_configure_views_pass2 done (first batched pass-2 call with meshlet occlusion)
    // Scratch that was outgrown is parked here until the context is destroyed: freeing it would need a device
    // synchronisation (work that uses it may still be in flight), and a stage call never synchronises.
    void* retired[64] = {};
    int n_retired = 0;
    unsigned long long* trace = nullptr;   // -DORBIT_TRACE builds only: 16 blocks of 1024 x 16 stamps
    unsigned trace_seq = 0;
    std::atomic<uint64_t> launches{0};
};

struct orbit_hiz {
    OrbitHizInfo info;
    uint32_t depth_w, depth_h;
    bool owns;
    int device;
};

// Outgrown scratch is retired, not freed (see orbit_ctx::retired). With doubling capacities a context retires a handful of
// buffers in its life; if the list ever fills up the oldest entries are freed after one device synchronisation.
static int retire(orbit_ctx* c, void* p) {
    if (!p) return ORBIT_OK;
    if (c->n_retired == 64) {
        CK(cudaDeviceSynchronize());
        for (int i = 0; i < 64; ++i) cudaFree(c->retired[i]);
        c->n_retired = 0;
    }
    c->retired[c->n_retired++] = p;
    return ORBIT_OK;
}

// Scan descriptors; a fresh array is zeroed on `stream` (epoch 0 never matches a launch: epochs start at 1).
static int ensure_status(orbit_ctx* c, size_t tiles, cudaStream_t stream) {
    if (tiles <= c->status_capacity) return ORBIT_OK;
    size_t cap = c->status_capacity ? c->status_capacity : 4096;
    while (cap < tiles) cap *= 2;
    int rc = retire(c, c->status);
    if (rc != ORBIT_OK) return rc;
    c->status = nullptr; c->status_capacity = 0;
    CK(cudaMalloc(&c->status, cap * sizeof(unsigned long long)));
    CK(cudaMemsetAsync(c->status, 0, cap * sizeof(unsigned long long), stream));
    c->status_capacity = cap;
    return ORBIT_OK;
}

static int ensure_tile_sums(orbit_ctx* c, size_t tiles) {
    if (tiles <= c->tile_sums_capacity) return ORBIT_OK;
    size_t cap = c->tile_sums_capacity ? c->tile_sums_capacity : 1024;
    while (cap < tiles) cap *= 2;
    int rc = retire(c, c->tile_sums);
    if (rc != ORBIT_OK) return rc;
    c->tile_sums = nullptr; c->tile_sums_capacity = 0;
    CK(cudaMalloc(&c->tile_sums, cap * sizeof(unsigned long long)));
    c->tile_sums_capacity = cap;
    return ORBIT_OK;
}

// record entries of the fused MAIN pass (orbit_meshlet_cull_late_main)
static int ensure_main_masks(orbit_ctx* c, uint64_t max_records) {
    if (max_records <= c->main_mask_capacity) return ORBIT_OK;
    int rc = retire(c, c->main_masks);
    if (rc != ORBIT_OK) return rc;
    c->main_masks = nullptr; c->main_mask_capacity = 0;
    size_t cap = 65536; while (cap < max_records) cap *= 2;
    CK(cudaMalloc(&c->main_masks, cap * sizeof(uint4)));
    c->main_mask_capacity = cap;
    return ORBIT_OK;
}

static int ensure_record_scratch(orbit_ctx* c, uint64_t max_records) {
    if (max_records <= c->draw_mask_capacity) return ORBIT_OK;
    int rc = retire(c, c->draw_masks);
    if (rc == ORBIT_OK) rc = retire(c, c->cmd_side);
    if (rc != ORBIT_OK) return rc;
    c->draw_masks = nullptr; c->cmd_side = nullptr; c->draw_mask_capacity = 0;
    size_t cap = 65536; while (cap < max_records) cap *= 2;
    CK(cudaMalloc(&c->draw_masks, cap * sizeof(uint4)));
    CK(cudaMalloc(&c->cmd_side, cap * 32u * sizeof(uint4)));
    c->draw_mask_capacity = cap;
    return ORBIT_OK;
}

// The light-parallel culling path keeps one hit bit per (cluster, light); grids whose matrix would exceed this budget (the
// reference's default 8-pixel tiles: ~10^6 clusters) take the CTA-per-cluster kernel instead.
static constexpr uint64_t kLightHitsBudgetBytes = 256ull << 20;
static uint64_t light_hits_words_needed(uint64_t clusters, uint64_t n_lights) {   // bit matrix + per-(cluster, light block) counts
    return clusters * ((uint64_t)light_hits_blocks((uint32_t)n_lights) * 17u + 9u);   // 16 words of bits + 1 count per (cluster, light block), 8 words of box + 1 hit total per cluster
}

static int ensure_light_hits(orbit_ctx* c, uint64_t words) {
    if (words <= c->light_hits_words) return ORBIT_OK;
    int rc = retire(c, c->light_hits);
    if (rc != ORBIT_OK) return rc;
    c->light_hits = nullptr; c->light_hits_words = 0;
    size_t cap = 1u << 16; while (cap < words) cap *= 2;
    CK(cudaMalloc(&c->light_hits, cap * sizeof(uint32_t)));
    c->light_hits_words = cap;
    return ORBIT_OK;
}

static int ensure_lights(orbit_ctx* c, uint64_t n_lights) {
    if (n_lights <= c->light_capacity) return ORBIT_OK;
    int rc = retire(c, c->light_view);
    if (rc != ORBIT_OK) return rc;
    c->light_view = nullptr; c->light_capacity = 0;
    size_t cap = 1024; while (cap < n_lights) cap *= 2;
    CK(cudaMalloc(&c->light_view, cap * sizeof(float4)));
    c->light_capacity = cap;
    return ORBIT_OK;
}

// block of the timeline buffer for the next kernel launch (development builds), else nullptr
static unsigned long long* next_trace(orbit_ctx* c) {
    if (!c->trace) return nullptr;
    return c->trace + (size_t)(c->trace_seq++ % 16u) * 1024u * 16u;
}

static ScanState next_scan(orbit_ctx* c) {
    return ScanState{next_trace(c), c->status, c->counters + 0, c->counters + 1, c->counters + 3};
}

static HizDevice hiz_device(const orbit_hiz* h) {
    HizDevice d{};
    if (h) {
        d.texels = h->info.texels; d.width = h->info.width; d.height = h->info.height; d.levels = h->info.levels;
        for (int i = 0; i < ORBIT_HIZ_MAX_LEVELS; ++i) d.level_offset[i] = h->info.level_offset[i];
    }
    return d;
}

static uint32_t npot(uint32_t v) { uint32_t p = 1; while (p < v) p <<= 1; return p; }

extern "C" {

int orbit_abi_version(void) { return ORBIT_ABI_VERSION; }

const char* orbit_error_string(int code) {
    switch (code) {
        case ORBIT_OK: return "ok";
        case ORBIT_ERR_INVALID_ARGUMENT: return "invalid argument";
        case ORBIT_ERR_CUDA: return "CUDA runtime error (see orbit_last_cuda_error)";
        case ORBIT_ERR_OUT_OF_MEMORY: return "out of memory";
        case ORBIT_ERR_NO_DEVICE: return "no CUDA device (this library has no CPU fallback)";
        case ORBIT_ERR_CAPACITY: return "an output buffer overflowed its capacity; extra items were dropped";
        default: return "unknown error";
    }
}

int orbit_last_cuda_error(void) { return g_last_cuda_error; }

int orbit_ctx_create(int device, orbit_ctx** out) {
    if (!out) return ORBIT_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) { g_last_cuda_error = (int)e; return ORBIT_ERR_NO_DEVICE; }
    if (device < 0 || device >= n) return ORBIT_ERR_INVALID_ARGUMENT;
    DeviceGuard guard(device);
    if (!guard.ok) { g_last_cuda_error = (int)cudaGetLastError(); return ORBIT_ERR_CUDA; }
    orbit_ctx* c = new (std::nothrow) orbit_ctx();
    if (!c) return ORBIT_ERR_OUT_OF_MEMORY;
    c->device = device;
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    c->sm_count = prop.multiProcessorCount;
    CK(cudaMalloc(&c->counters, 64 * sizeof(unsigned int)));
    CK(cudaMemset(c->counters, 0, 64 * sizeof(unsigned int)));
    { const unsigned int one = 1u; CK(cudaMemcpy(c->counters + 3, &one, sizeof(one), cudaMemcpyHostToDevice)); }
    CK(cudaMalloc(&c->chunk_counts, 6 * 2048 * sizeof(uint32_t)));   // two parities for orbit_meshlet_cull + two (never read) for orbit_meshlet_test + two for the fused MAIN pass
    CK(cudaMemset(c->chunk_counts, 0, 6 * 2048 * sizeof(uint32_t)));
    CK(cudaHostAlloc(&c->status_host, sizeof(OrbitStatus), cudaHostAllocMapped));
    std::memset(c->status_host, 0, sizeof(OrbitStatus));
    CK(cudaHostGetDevicePointer(&c->status_dev, c->status_host, 0));
    int rc = ensure_status(c, 4096, nullptr);
    if (rc != ORBIT_OK) return rc;
    CK(cudaDeviceSynchronize());
    CK(meshlet_cull_configure_device());
    CK(light_cluster_configure_device());
#ifdef ORBIT_TRACE
    CK(cudaMalloc(&c->trace, 16u * 1024u * 16u * sizeof(unsigned long long)));
    CK(cudaMemset(c->trace, 0, 16u * 1024u * 16u * sizeof(unsigned long long)));
#endif
    if (const char* s = std::getenv("ORBIT_DEBUG_SKIP")) c->debug_skip = std::atoi(s);
    if (const char* s = std::getenv("ORBIT_MC_CTAS_PER_SM")) { int v = std::atoi(s); if (v > 0 && v <= 32) c->mc_ctas_per_sm = v; }
    c->light_hits_budget = kLightHitsBudgetBytes;
    if (const char* s = std::getenv("ORBIT_LIGHT_HITS_BUDGET_MB")) { const long v = std::atol(s); if (v >= 0) c->light_hits_budget = (uint64_t)v << 20; }
    if (const char* s = std::getenv("ORBIT_EMIT_CTAS_PER_SM")) { int v = std::atoi(s); if (v > 0 && v <= 32) c->emit_ctas_per_sm = v; }
    *out = c;
    return ORBIT_OK;
}

void orbit_ctx_destroy(orbit_ctx* c) {
    if (!c) return;
    DeviceGuard guard(c->device);
    cudaDeviceSynchronize();
    for (int i = 0; i < c->n_retired; ++i) cudaFree(c->retired[i]);
    cudaFree(c->status); cudaFree(c->counters); cudaFree(c->light_view); cudaFree(c->light_hits); cudaFree(c->draw_masks); cudaFree(c->cmd_side); cudaFree(c->main_masks); cudaFree(c->chunk_counts); cudaFree(c->view_counters); cudaFree(c->tile_sums);
    cudaFree(c->trace);
    cudaFreeHost(c->status_host);
    delete c;
}

int orbit_ctx_poll_status(orbit_ctx* c, OrbitStatus* out) {
    if (!c || !out) return ORBIT_ERR_INVALID_ARGUMENT;
    *out = *c->status_host;
    std::memset(c->status_host, 0, sizeof(OrbitStatus));
    if (out->asset_error) return ORBIT_ERR_INVALID_ARGUMENT;
    if (out->peer_timeout) return ORBIT_ERR_CUDA;
    return (out->dispatch_overflow || out->draw_overflow || out->light_index_overflow || out->visibility_overflow) ? ORBIT_ERR_CAPACITY : ORBIT_OK;
}

uint64_t orbit_ctx_launch_count(const orbit_ctx* c) { return c ? c->launches.load() : 0; }

int orbit_ctx_reserve(orbit_ctx* c, uint64_t entity_draws, uint64_t capacity_records, uint64_t n_lights, uint64_t n_clusters, uint64_t n_entities) {
    if (!c) return ORBIT_ERR_INVALID_ARGUMENT;
    if (capacity_records > 0xFFFFFFFFull) capacity_records = 0xFFFFFFFFull;
    GUARD(c);
    size_t tiles = (size_t)(entity_draws + 255u) / 256u + 1u;
    if ((size_t)n_clusters + 1u > tiles) tiles = (size_t)n_clusters + 1u;
    int rc = ensure_status(c, tiles, nullptr);
    if (rc == ORBIT_OK && capacity_records) rc = ensure_record_scratch(c, capacity_records);
    if (rc == ORBIT_OK && capacity_records) rc = ensure_main_masks(c, capacity_records);        // fused LATE + MAIN
    if (rc == ORBIT_OK && n_lights) rc = ensure_lights(c, n_lights);
    if (rc == ORBIT_OK && n_lights && n_clusters) {                                             // light-parallel culling path
        const uint64_t words = light_hits_words_needed(n_clusters, n_lights);
        if (words * 4u <= c->light_hits_budget) rc = ensure_light_hits(c, words);
    }
    if (rc == ORBIT_OK && n_entities) rc = ensure_tile_sums(c, ((size_t)n_entities + 255u) / 256u);
    if (rc != ORBIT_OK) return rc;
    CK(cudaDeviceSynchronize());   // the one place that may synchronise: after this, stage calls within these sizes never allocate
    return ORBIT_OK;
}

#ifdef ORBIT_TRACE
// development builds only: device pointer and size of the timeline buffer (see scan.cuh)
int orbit_debug_trace(orbit_ctx* c, void** ptr, uint64_t* bytes) {
    if (!c || !ptr || !bytes) return ORBIT_ERR_INVALID_ARGUMENT;
    *ptr = c->trace; *bytes = 16ull * 1024ull * 16ull * sizeof(unsigned long long);
    c->trace_seq = 0;   // the next launch stamps block 0 again
    return ORBIT_OK;
}
#endif

// ---- depth pyramid -------------------------------------------------------------------------------------
int orbit_hiz_geometry(uint32_t dw, uint32_t dh, OrbitHizInfo* out) {
    if (!out || dw == 0 || dh == 0 || dw > 32768u || dh > 32768u) return ORBIT_ERR_INVALID_ARGUMENT;
    std::memset(out, 0, sizeof(*out));
    out->width = npot(dw) / 2u; out->height = npot(dh) / 2u;         // draw_gen.rs:458
    if (out->width == 0 || out->height == 0) return ORBIT_ERR_INVALID_ARGUMENT;  // a 1-texel-wide depth has no pyramid
    uint32_t mx = out->width > out->height ? out->width : out->height;
    uint32_t levels = 0; while (mx) { ++levels; mx >>= 1; }           // math.rs:18-20
    out->levels = levels;
    uint32_t off = 0;
    for (uint32_t l = 0; l < levels; ++l) {
        out->level_offset[l] = off;
        uint32_t w = out->width >> l, h = out->height >> l;
        off += (w ? w : 1u) * (h ? h : 1u);                            // image.rs:531
    }
    out->total_texels = off;
    return ORBIT_OK;
}

static int hiz_make(orbit_ctx* c, uint32_t dw, uint32_t dh, float* texels, bool owns, orbit_hiz** out) {
    if (!c || !out) return ORBIT_ERR_INVALID_ARGUMENT;
    orbit_hiz* h = new (std::nothrow) orbit_hiz();
    if (!h) return ORBIT_ERR_OUT_OF_MEMORY;
    int rc = orbit_hiz_geometry(dw, dh, &h->info);
    if (rc != ORBIT_OK) { delete h; return rc; }
    h->depth_w = dw; h->depth_h = dh; h->owns = owns; h->device = c->device;
    if (owns) {
        DeviceGuard guard(c->device);
        cudaError_t e = guard.ok ? cudaSuccess : cudaErrorInvalidDevice;
        if (e == cudaSuccess) e = cudaMalloc(&texels, (size_t)h->info.total_texels * sizeof(float));
        if (e != cudaSuccess) { g_last_cuda_error = (int)e; delete h; return e == cudaErrorMemoryAllocation ? ORBIT_ERR_OUT_OF_MEMORY : ORBIT_ERR_CUDA; }
    } else if (!texels || ((uintptr_t)texels & 15u)) {
        delete h; return ORBIT_ERR_INVALID_ARGUMENT;
    }
    h->info.texels = texels;
    *out = h;
    return ORBIT_OK;
}

int orbit_hiz_create(orbit_ctx* c, uint32_t dw, uint32_t dh, orbit_hiz** out) { return hiz_make(c, dw, dh, nullptr, true, out); }
int orbit_hiz_wrap(orbit_ctx* c, uint32_t dw, uint32_t dh, float* texels, orbit_hiz** out) { return hiz_make(c, dw, dh, texels, false, out); }

void orbit_hiz_destroy(orbit_hiz* h) {
    if (!h) return;
    if (h->owns) { DeviceGuard guard(h->device); cudaFree(h->info.texels); }
    delete h;
}

int orbit_hiz_info(const orbit_hiz* h, OrbitHizInfo* out) {
    if (!h || !out) return ORBIT_ERR_INVALID_ARGUMENT;
    *out = h->info;
    return ORBIT_OK;
}

int orbit_hiz_build(orbit_ctx* c, orbit_hiz* h, const float* depth, uint32_t dw, uint32_t dh, void* stream) {
    if (!c || !h || !depth || dw != h->depth_w || dh != h->depth_h) return ORBIT_ERR_INVALID_ARGUMENT;
    GUARD(c);
    HizBuildParams p{};
    p.depth = depth; p.texels = h->info.texels; p.depth_w = dw; p.depth_h = dh;
    p.width = h->info.width; p.height = h->info.height; p.levels = h->info.levels;
    for (int i = 0; i < ORBIT_HIZ_MAX_LEVELS; ++i) p.level_offset[i] = h->info.level_offset[i];
    p.ticket = c->counters + 2;
    p.trace = next_trace(c);
    CK(launch_hiz_build(p, (cudaStream_t)stream));
    c->launches += 1;
    return ORBIT_OK;
}

// Batched form: one launch, a row of CTAs per pyramid. Pyramid v's ticket is counter word 40 + v (words 40..55 are used by
// nothing else and were zeroed with the rest at context creation; each row's last CTA re-zeroes its own).
int orbit_hiz_build_views(orbit_ctx* c, orbit_hiz* const* hizs, const float* const* depths, uint32_t n_views, uint32_t dw, uint32_t dh,
                          void* stream) {
    if (!c || !hizs || !depths || n_views == 0u || n_views > ORBIT_MAX_BATCH_VIEWS) return ORBIT_ERR_INVALID_ARGUMENT;
    for (uint32_t v = 0; v < n_views; ++v) {
        const orbit_hiz* h = hizs[v];
        if (!h || !depths[v] || dw != h->depth_w || dh != h->depth_h) return ORBIT_ERR_INVALID_ARGUMENT;
        for (uint32_t u = 0; u < v; ++u) if (hizs[u]->info.texels == h->info.texels) return ORBIT_ERR_INVALID_ARGUMENT;
    }
    GUARD(c);
    HizBuildViewsParams pv{};
    pv.n_views = n_views;
    for (uint32_t v = 0; v < n_views; ++v) {
        const orbit_hiz* h = hizs[v];
        HizBuildParams& p = pv.view[v];
        p.depth = depths[v]; p.texels = h->info.texels; p.depth_w = dw; p.depth_h = dh;
        p.width = h->info.width; p.height = h->info.height; p.levels = h->info.levels;
        for (int i = 0; i < ORBIT_HIZ_MAX_LEVELS; ++i) p.level_offset[i] = h->info.level_offset[i];
        p.ticket = c->counters + 40 + v;
    }
    pv.view[0].trace = next_trace(c);
    CK(launch_hiz_build_views(pv, (cudaStream_t)stream));
    c->launches += 1;
    return ORBIT_OK;
}

// ---- entity stage ----------------------------------------------------------------------------------------
static int check_cull(const OrbitCullInfo* cull, const OrbitSceneBuffers* scene, const orbit_hiz* hiz, bool meshlet_stage) {
    if (!cull || !scene) return ORBIT_ERR_INVALID_ARGUMENT;
    if (cull->cull_plane_count > ORBIT_MAX_CULL_PLANES) return ORBIT_ERR_INVALID_ARGUMENT;  // assert!, draw_gen.rs:334,390
    if (cull->occlusion_pass > 2u) return ORBIT_ERR_INVALID_ARGUMENT;
    if (!scene->entities) return ORBIT_ERR_INVALID_ARGUMENT;
    const bool mocc = cull->meshlet_visibility_buffer != ORBIT_NO_BUFFER;
    if (meshlet_stage) {
        if (!scene->meshlets || !scene->materials) return ORBIT_ERR_INVALID_ARGUMENT;
        if (((uintptr_t)scene->meshlets & 15u) || ((uintptr_t)scene->entities & 15u)) return ORBIT_ERR_INVALID_ARGUMENT;
        if (mocc && cull->occlusion_pass != 0u && !scene->meshlet_visibility) return ORBIT_ERR_INVALID_ARGUMENT;
        if (mocc && cull->occlusion_pass == 2u && !hiz) return ORBIT_ERR_INVALID_ARGUMENT;
    } else {
        if (!scene->entity_draws || !scene->mesh_infos) return ORBIT_ERR_INVALID_ARGUMENT;
        if (((uintptr_t)scene->mesh_infos & 15u) || ((uintptr_t)scene->entities & 15u) || ((uintptr_t)scene->entity_draws & 3u)) return ORBIT_ERR_INVALID_ARGUMENT;
        if (cull->occlusion_pass != 0u && !scene->entity_visibility) return ORBIT_ERR_INVALID_ARGUMENT;
        if (cull->occlusion_pass == 2u && !hiz) return ORBIT_ERR_INVALID_ARGUMENT;
        if (scene->draw_begin % 32u) return ORBIT_ERR_INVALID_ARGUMENT;
    }
    return ORBIT_OK;
}

// draws [begin, end) a call covers (OrbitSceneBuffers::draw_begin / draw_end, 0,0 = all)
static int draw_range(const OrbitSceneBuffers* scene, uint32_t* begin, uint32_t* end) {
    *begin = scene->draw_begin; *end = scene->draw_end;
    if (*begin == 0u && *end == 0u) *end = scene->entity_draw_count;
    if (*end > scene->entity_draw_count) *end = scene->entity_draw_count;
    return *begin > *end ? ORBIT_ERR_INVALID_ARGUMENT : ORBIT_OK;
}

static EntityCullParams entity_params(orbit_ctx* c, const OrbitCullInfo* cull, const OrbitSceneBuffers* scene, const orbit_hiz* hiz,
                                      void* dispatch_buffer, uint64_t capacity_records, uint32_t begin, uint32_t end) {
    EntityCullParams p{};
    p.cull = *cull; p.hiz = hiz_device(hiz);
    p.entity_draw_words = (const uint32_t*)scene->entity_draws;
    p.mesh_infos = (const uint8_t*)scene->mesh_infos;
    p.entities = (const float4*)scene->entities;
    p.entity_visibility = scene->entity_visibility;
    p.dispatch_words = (uint32_t*)dispatch_buffer;
    p.overflow_flag = &c->status_dev->dispatch_overflow;
    p.capacity_records = capacity_records;
    p.draw_begin = begin; p.draw_end = end;
    return p;
}

static uint32_t entity_coresident_ctas(orbit_ctx* c) {
    if (c->entity_occupancy <= 0) c->entity_occupancy = entity_cull_max_ctas_per_sm();
    return (uint32_t)(c->sm_count * (c->entity_occupancy > 0 ? c->entity_occupancy : 1));
}

static uint32_t entity_views_coresident_ctas(orbit_ctx* c, uint32_t pass) {
    int& occ = c->entity_views_occupancy[pass];
    if (occ <= 0) occ = entity_cull_views_max_ctas_per_sm(pass);
    return (uint32_t)(c->sm_count * (occ > 0 ? occ : 1));
}

static int entity_stage(orbit_ctx* c, const OrbitCullInfo* cull, const OrbitSceneBuffers* scene, const orbit_hiz* hiz,
                        void* meshlet_dispatch_buffer, void* mirror_dispatch_buffer, uint64_t capacity_records, void* stream) {
    if (!c || !meshlet_dispatch_buffer || ((uintptr_t)meshlet_dispatch_buffer & 3u)) return ORBIT_ERR_INVALID_ARGUMENT;
    int rc = check_cull(cull, scene, hiz, false);
    if (rc != ORBIT_OK) return rc;
    uint32_t begin, end;
    rc = draw_range(scene, &begin, &end);
    if (rc != ORBIT_OK) return rc;
    const uint32_t n = end - begin;
    GUARD(c);
    rc = ensure_status(c, (size_t)(n + 255u) / 256u + 1u, (cudaStream_t)stream);
    if (rc != ORBIT_OK) return rc;
    EntityCullParams p = entity_params(c, cull, scene, hiz, meshlet_dispatch_buffer, capacity_records, begin, end);
    p.dispatch_mirror = (uint32_t*)mirror_dispatch_buffer;
    p.scan = next_scan(c);
    CK(launch_entity_cull(p, n, entity_coresident_ctas(c), (cudaStream_t)stream));
    c->launches += 1;
    return ORBIT_OK;
}

int orbit_entity_cull(orbit_ctx* c, const OrbitCullInfo* cull, const OrbitSceneBuffers* scene, const orbit_hiz* hiz,
                      void* meshlet_dispatch_buffer, uint64_t capacity_records, void* stream) {
    return entity_stage(c, cull, scene, hiz, meshlet_dispatch_buffer, nullptr, capacity_records, stream);
}

// ---- fused LATE + MAIN -----------------------------------------------------------------------------------
// The MAIN pass (forward.rs:518-548) is pass 1 over the visibility bits the LATE pass (pass 2, forward.rs:266-403) has just
// written. With the same camera, planes, LOD parameters and buffers, and meshlet occlusion culling on:
//   entity level   MAIN: visible = bit_new && frustum = LATE's `visible` (the bit IS that value and already includes the same
//                  frustum test), should_draw = visible; LATE: should_draw = visible && (!bit_old || mocc) = visible
//                  (entity_cull.comp:137-189) -> the two dispatch lists are the same list.
//   meshlet level  MAIN: visible = bit_new && frustum && cone = LATE's `visible`; should_draw = visible && alpha filter
//                  (meshlet_cull.comp:137,207), LATE: visible && !bit_old (or the alpha filter for noskip modes).
// So one entity kernel writes both dispatch buffers and the LATE test kernel fills both record-entry arrays; each list is
// then emitted by its own emit kernel. Everything else falls back to separate calls: orbit_cull_pair_compatible says which.
int orbit_cull_pair_compatible(const OrbitCullInfo* late, const OrbitCullInfo* main_pass) {
    if (!late || !main_pass) return 0;
    if (late->occlusion_pass != 2u || main_pass->occlusion_pass != 1u) return 0;
    if (late->meshlet_visibility_buffer == ORBIT_NO_BUFFER || main_pass->meshlet_visibility_buffer == ORBIT_NO_BUFFER) return 0;
    if (late->visibility_buffer != main_pass->visibility_buffer || late->meshlet_visibility_buffer != main_pass->meshlet_visibility_buffer) return 0;
    // view matrix, reprojection matrix, planes, plane count: bytes [0, 324)
    if (std::memcmp(late, main_pass, offsetof(OrbitCullInfo, alpha_mode_flags)) != 0) return 0;
    // projection type (cone test) and LOD parameters, bytes [372, 400); p00 / p11 / z_near / z_far are only read by the
    // occlusion test and are left zero for pass 1 by CullInfo::to_gpu (draw_gen.rs:150-198)
    if (late->projection_type != main_pass->projection_type) return 0;
    if (std::memcmp(&late->lod_base, &main_pass->lod_base, sizeof(OrbitCullInfo) - offsetof(OrbitCullInfo, lod_base)) != 0) return 0;
    return 1;
}

int orbit_entity_cull_late_main(orbit_ctx* c, const OrbitCullInfo* late, const OrbitCullInfo* main_pass, const OrbitSceneBuffers* scene,
                                const orbit_hiz* hiz, void* late_dispatch_buffer, void* main_dispatch_buffer, uint64_t capacity_records,
                                void* stream) {
    if (!main_dispatch_buffer || ((uintptr_t)main_dispatch_buffer & 3u) || main_dispatch_buffer == late_dispatch_buffer) return ORBIT_ERR_INVALID_ARGUMENT;
    if (!orbit_cull_pair_compatible(late, main_pass)) return ORBIT_ERR_INVALID_ARGUMENT;
    return entity_stage(c, late, scene, hiz, late_dispatch_buffer, main_dispatch_buffer, capacity_records, stream);
}

// ---- meshlet stage ---------------------------------------------------------------------------------------
// The CullInfo and the planes paired for the packed test kernel (MeshletCullParams::planes_t)
static void set_cull(MeshletCullParams& p, const OrbitCullInfo* cull) {
    p.cull = *cull;
    p.pk_one = make_float2(1.0f, 1.0f); p.pk_mone = make_float2(-1.0f, -1.0f);
    for (uint32_t j = 0; j < 6u; ++j) {
        const uint32_t n = cull->cull_plane_count;
        const uint32_t a = 2u * j < n ? 2u * j : (n ? n - 1u : 0u), b = 2u * j + 1u < n ? 2u * j + 1u : a;
        for (int cc = 0; cc < 4; ++cc) p.planes_t[j][cc] = make_float2(cull->cull_planes[a][cc], cull->cull_planes[b][cc]);
    }
}

// Emit grid for a dispatch buffer of max_records records; *small_grid = the CTAs that take part when the list is short.
static uint64_t emit_grids(orbit_ctx* c, uint64_t max_records, uint32_t* small_grid) {
    // emit kernel: two CTAs per SM (every CTA repeats the 2048-entry chunk scan; more CTAs only add to that)
    if (c->emit_occupancy <= 0) c->emit_occupancy = meshlet_emit_max_ctas_per_sm();
    // emit kernel: as many CTAs per SM as fit (3) for long lists; two per SM take part when the list is short (decided on the
    // device from the survivor count, see meshlet_emit_body)
    int emit_per_sm = c->emit_occupancy > 0 ? c->emit_occupancy : 1;
    if (emit_per_sm > 4) emit_per_sm = 4;
    // even CTAs that leave at once cost launch time (C2 frame: +1.6 us over its three emit launches), so a dispatch buffer too
    // small for a long list (capacity below 2^18 records = 8 M meshlets) gets the two per SM of the short case outright
    if (max_records < (1u << 18) && emit_per_sm > 2) emit_per_sm = 2;
    int emit_small_per_sm = emit_per_sm < 2 ? emit_per_sm : 2;
    if (c->emit_ctas_per_sm >= 1 && c->emit_ctas_per_sm <= c->emit_occupancy) emit_per_sm = emit_small_per_sm = c->emit_ctas_per_sm;   // tuning knob
    *small_grid = (uint32_t)(c->sm_count * emit_small_per_sm);
    return (uint64_t)c->sm_count * (uint64_t)emit_per_sm;
}

// mode 0: test + emit (orbit_meshlet_cull); mode 1: test only, record entries into `record_masks` (orbit_meshlet_test)
struct MainPassOutputs { const OrbitCullInfo* cull; void* draw_command_buffer; void* task_payloads; };   // fused LATE + MAIN

static int meshlet_stage(orbit_ctx* c, const OrbitCullInfo* cull, const OrbitSceneBuffers* scene, const orbit_hiz* hiz,
                         const void* meshlet_dispatch_buffer, uint64_t capacity_records, void* draw_command_buffer,
                         uint64_t capacity_draws, void* task_payloads, void* record_masks, void* stream,
                         const MainPassOutputs* fused_main = nullptr) {
    const bool test_only = record_masks != nullptr;
    if (!c || !meshlet_dispatch_buffer || (!test_only && !draw_command_buffer)) return ORBIT_ERR_INVALID_ARGUMENT;
    if (((uintptr_t)meshlet_dispatch_buffer & 3u) || ((uintptr_t)draw_command_buffer & 3u) || ((uintptr_t)task_payloads & 3u) ||
        ((uintptr_t)record_masks & 15u)) return ORBIT_ERR_INVALID_ARGUMENT;
    if (capacity_records > 0xFFFFFFFFull) capacity_records = 0xFFFFFFFFull;
    int rc = check_cull(cull, scene, hiz, true);
    if (rc != ORBIT_OK) return rc;
    // The record count lives on the device (the reference's dispatch_indirect); scratch and grid are sized for
    // the dispatch buffer's capacity and the kernel clamps the device-side count to it.
    const uint64_t max_records = capacity_records;
    GUARD(c);
    if (!test_only) {
        rc = ensure_record_scratch(c, max_records);
        if (rc != ORBIT_OK) return rc;
    }
    if (fused_main) {
        rc = ensure_main_masks(c, max_records);
        if (rc != ORBIT_OK) return rc;
    }
    MeshletCullParams p{};
    p.hiz = hiz_device(hiz);
    p.dispatch_words = (const uint32_t*)meshlet_dispatch_buffer;
    p.meshlets = (const uint4*)scene->meshlets;
    p.entities = (const float4*)scene->entities;
    p.materials = (const uint8_t*)scene->materials;
    p.meshlet_visibility = scene->meshlet_visibility;
    p.draw_words = (uint32_t*)draw_command_buffer;
    p.task_payloads = (uint32_t*)task_payloads;
    p.overflow_flag = &c->status_dev->draw_overflow;
    if (!test_only) {
        p.draw_masks = c->draw_masks;
        p.cmd_side = c->cmd_side;
        p.draw_total = c->counters + 4;     // [4],[5]
        p.chunk_parity = c->counters + 6;   // [6] word A, [7] word B
        p.chunk_counts = c->chunk_counts;
    } else {
        // the survivor counters of a test-only call are never read: they go to a second set of scratch words, so that
        // they cannot leak into a later orbit_meshlet_cull / orbit_draws_from_masks of this context
        p.draw_masks = (uint4*)record_masks;
        p.cmd_side = nullptr;               // entries carry flag 1: whoever emits reads the meshlet itself
        p.draw_total = c->counters + 10;    // [10],[11]
        p.chunk_parity = c->counters + 12;  // [12],[13]
        p.chunk_counts = c->chunk_counts + 2 * 2048;
    }
    if (fused_main) {
        p.main_masks = c->main_masks;
        p.main_chunk_counts = c->chunk_counts + 4 * 2048;
        p.main_chunk_parity = c->counters + 22;   // [22] word A, [23] word B
        p.main_draw_total = c->counters + 20;     // [20],[21]
        p.main_alpha_mode_flags = fused_main->cull->alpha_mode_flags;
    }
    p.capacity_records = max_records;
    p.capacity_draws = capacity_draws;
    p.scan.trace = next_trace(c);
    p.trace_emit = next_trace(c);
    set_cull(p, cull);
    // test kernel: persistent warps, cyclic tiles, no inter-CTA dependency -> one full wave of CTAs
    int& occ_slot = c->mc_occupancy[meshlet_cull_variant_index(*cull)];
    if (occ_slot <= 0) occ_slot = meshlet_cull_max_ctas_per_sm(p);
    const int occ = occ_slot;
    int per_sm = c->mc_ctas_per_sm;
    if (per_sm <= 0) per_sm = occ > 0 ? occ : 1;
    const uint64_t grid = (uint64_t)c->sm_count * (uint64_t)per_sm;
    uint32_t emit_small_grid;
    const uint64_t emit_grid = emit_grids(c, max_records, &emit_small_grid);
    p.emit_small_grid = emit_small_grid;
    const bool skip_emit = test_only || c->debug_skip == 1;
    const bool pair = fused_main && !skip_emit;      // both lists leave in one emit launch
    CK(launch_meshlet_cull(p, c->debug_skip == 2 ? 0 : (int)grid, (skip_emit || pair) ? 0 : (int)emit_grid, (cudaStream_t)stream));
    c->launches += test_only ? 1 : 2;   // test kernel (+ emit kernel)
    if (pair) {
        // the MAIN list: the ordinary emit code over the second set of record entries / chunk counts; its entries carry
        // flag 1, so the command words are read from the meshlets (the survivors of a steady frame: a few MB)
        MeshletCullParams m = p;
        m.cull = *fused_main->cull;
        m.draw_masks = c->main_masks; m.cmd_side = nullptr;
        m.chunk_counts = p.main_chunk_counts; m.chunk_parity = p.main_chunk_parity; m.draw_total = p.main_draw_total;
        m.draw_words = (uint32_t*)fused_main->draw_command_buffer;
        m.task_payloads = (uint32_t*)fused_main->task_payloads;
        m.main_masks = nullptr;
        m.trace_emit = next_trace(c);
        CK(launch_meshlet_emit_pair(p, m, (int)emit_grid, (cudaStream_t)stream));
    }
    return ORBIT_OK;
}

int orbit_meshlet_cull_late_main(orbit_ctx* c, const OrbitCullInfo* late, const OrbitCullInfo* main_pass, const OrbitSceneBuffers* scene,
                                 const orbit_hiz* hiz, const void* late_dispatch_buffer, uint64_t capacity_records,
                                 void* late_draw_command_buffer, void* main_draw_command_buffer, uint64_t capacity_draws,
                                 void* late_task_payloads, void* main_task_payloads, void* stream) {
    if (!main_draw_command_buffer || ((uintptr_t)main_draw_command_buffer & 3u) || ((uintptr_t)main_task_payloads & 3u) ||
        main_draw_command_buffer == late_draw_command_buffer) return ORBIT_ERR_INVALID_ARGUMENT;
    if (!orbit_cull_pair_compatible(late, main_pass)) return ORBIT_ERR_INVALID_ARGUMENT;
    const MainPassOutputs mo{main_pass, main_draw_command_buffer, main_task_payloads};
    return meshlet_stage(c, late, scene, hiz, late_dispatch_buffer, capacity_records, late_draw_command_buffer, capacity_draws,
                         late_task_payloads, nullptr, stream, &mo);
}

int orbit_meshlet_cull(orbit_ctx* c, const OrbitCullInfo* cull, const OrbitSceneBuffers* scene, const orbit_hiz* hiz,
                       const void* meshlet_dispatch_buffer, uint64_t capacity_records, void* draw_command_buffer,
                       uint64_t capacity_draws, void* task_payloads, void* stream) {
    return meshlet_stage(c, cull, scene, hiz, meshlet_dispatch_buffer, capacity_records, draw_command_buffer, capacity_draws, task_payloads,
                         nullptr, stream);
}

int orbit_meshlet_test(orbit_ctx* c, const OrbitCullInfo* cull, const OrbitSceneBuffers* scene, const orbit_hiz* hiz,
                       const void* meshlet_dispatch_buffer, uint64_t capacity_records, void* record_masks, void* stream) {
    if (!record_masks) return ORBIT_ERR_INVALID_ARGUMENT;
    return meshlet_stage(c, cull, scene, hiz, meshlet_dispatch_buffer, capacity_records, nullptr, 0, nullptr, record_masks, stream);
}

int orbit_record_masks_put(orbit_ctx* c, const void* src_record_masks, const void* meshlet_dispatch_buffer, uint64_t capacity_records,
                           void* dst_region, uint32_t* dst_count, void* stream) {
    if (!c || !src_record_masks || !meshlet_dispatch_buffer || !dst_region || !dst_count) return ORBIT_ERR_INVALID_ARGUMENT;
    if ((((uintptr_t)src_record_masks | (uintptr_t)dst_region) & 15u) || (((uintptr_t)meshlet_dispatch_buffer | (uintptr_t)dst_count) & 3u)) return ORBIT_ERR_INVALID_ARGUMENT;
    GUARD(c);
    CK(launch_record_masks_put((const uint4*)src_record_masks, (const uint32_t*)meshlet_dispatch_buffer, (uint4*)dst_region, dst_count,
                               capacity_records, c->sm_count * 8, (cudaStream_t)stream));
    c->launches += 1;
    return ORBIT_OK;
}

int orbit_draws_from_masks(orbit_ctx* c, const OrbitSceneBuffers* scene, const void* record_masks, uint64_t region_stride_records,
                           const uint32_t* region_counts, uint32_t n_regions, void* draw_command_buffer, uint64_t capacity_draws, void* stream) {
    if (!c || !scene || !scene->meshlets || !record_masks || !region_counts || n_regions == 0u || n_regions > 16u || !draw_command_buffer) return ORBIT_ERR_INVALID_ARGUMENT;
    if (((uintptr_t)record_masks & 15u) || ((uintptr_t)draw_command_buffer & 3u) || ((uintptr_t)scene->meshlets & 15u)) return ORBIT_ERR_INVALID_ARGUMENT;
    if (region_stride_records > 0xFFFFFFFFull) return ORBIT_ERR_INVALID_ARGUMENT;
    GUARD(c);
    MeshletCullParams p{};
    p.meshlets = (const uint4*)scene->meshlets;
    p.draw_words = (uint32_t*)draw_command_buffer;
    p.overflow_flag = &c->status_dev->draw_overflow;
    p.draw_masks = (uint4*)record_masks;      // read only on this path
    p.cmd_side = nullptr;
    p.draw_total = c->counters + 4;
    p.chunk_parity = c->counters + 6;
    p.chunk_counts = c->chunk_counts;
    p.capacity_records = 0xFFFFFFFFull;
    p.capacity_draws = capacity_draws;
    p.dispatch_words = c->counters + 16;      // a 3-word dispatch header written by the recount kernel
    p.region_counts = region_counts; p.region_stride = region_stride_records; p.n_regions = n_regions;
    p.trace_emit = next_trace(c);
    if (c->emit_occupancy <= 0) c->emit_occupancy = meshlet_emit_max_ctas_per_sm();
    int emit_per_sm = c->emit_occupancy > 0 ? c->emit_occupancy : 1;
    if (emit_per_sm > 4) emit_per_sm = 4;
    p.emit_small_grid = (uint32_t)(c->sm_count * (emit_per_sm < 2 ? emit_per_sm : 2));
    CK(launch_draws_from_masks(p, c->counters + 16, c->sm_count * 4, c->sm_count * emit_per_sm, (cudaStream_t)stream));
    c->launches += 2;
    return ORBIT_OK;
}

// ---- batched pass-0 views ---------------------------------------------------------------------------------
// one output buffer per view: present, 4-byte aligned, none shared with another view
static int check_view_buffers(const void* const* buffers, uint32_t n_views) {
    if (!buffers) return ORBIT_ERR_INVALID_ARGUMENT;
    for (uint32_t v = 0; v < n_views; ++v) {
        if (!buffers[v] || ((uintptr_t)buffers[v] & 3u)) return ORBIT_ERR_INVALID_ARGUMENT;
        for (uint32_t u = 0; u < v; ++u) if (buffers[u] == buffers[v]) return ORBIT_ERR_INVALID_ARGUMENT;
    }
    return ORBIT_OK;
}

// Checks shared by both stages: the view count, every view's CullInfo (pass 0, one projection type, check_cull), and one
// output buffer per view — present, 4-byte aligned, none shared with another view.
static int check_views(const OrbitCullInfo* culls, uint32_t n_views, const OrbitSceneBuffers* scene, const void* const* buffers,
                       bool meshlet_stage) {
    if (!culls || !buffers || n_views == 0u || n_views > ORBIT_MAX_BATCH_VIEWS) return ORBIT_ERR_INVALID_ARGUMENT;
    for (uint32_t v = 0; v < n_views; ++v) {
        int rc = check_cull(&culls[v], scene, nullptr, meshlet_stage);
        if (rc != ORBIT_OK) return rc;
        if (culls[v].occlusion_pass != 0u || culls[v].projection_type != culls[0].projection_type) return ORBIT_ERR_INVALID_ARGUMENT;
    }
    return check_view_buffers(buffers, n_views);
}

int orbit_entity_cull_views(orbit_ctx* c, const OrbitCullInfo* culls, uint32_t n_views, const OrbitSceneBuffers* scene,
                            void* const* dispatch_buffers, uint64_t capacity_records, void* stream) {
    if (!c) return ORBIT_ERR_INVALID_ARGUMENT;
    int rc = check_views(culls, n_views, scene, (const void* const*)dispatch_buffers, false);
    if (rc != ORBIT_OK) return rc;
    uint32_t begin, end;
    rc = draw_range(scene, &begin, &end);
    if (rc != ORBIT_OK) return rc;
    const uint32_t n = end - begin;
    GUARD(c);
    rc = ensure_status(c, (size_t)n_views * ((n + 255u) / 256u + 1u), (cudaStream_t)stream);   // one descriptor block per view
    if (rc != ORBIT_OK) return rc;
    EntityViewsParams pv{};
    pv.n_views = n_views;
    for (uint32_t v = 0; v < n_views; ++v) pv.view[v] = entity_params(c, &culls[v], scene, nullptr, dispatch_buffers[v], capacity_records, begin, end);
    pv.view[0].scan = next_scan(c);
    CK(launch_entity_cull_views(pv, n, entity_views_coresident_ctas(c, 0u), (cudaStream_t)stream));
    c->launches += 1;
    return ORBIT_OK;
}

// The meshlet stage of both batched forms, after their own checks: view v reads scenes[v] (per_view_scene) or scenes[0], and
// the pyramid hizs[v] (pass 2 with meshlet occlusion; NULL otherwise).
static int meshlet_views_stage(orbit_ctx* c, const OrbitCullInfo* culls, uint32_t n_views, const OrbitSceneBuffers* scenes, bool per_view_scene,
                               const orbit_hiz* const* hizs, const void* const* dispatch_buffers, uint64_t capacity_records,
                               void* const* draw_command_buffers, uint64_t capacity_draws, void* const* task_payloads, void* stream) {
    int rc = check_view_buffers((const void* const*)draw_command_buffers, n_views);
    if (rc != ORBIT_OK) return rc;
    for (uint32_t v = 0; task_payloads && v < n_views; ++v) {
        if ((uintptr_t)task_payloads[v] & 3u) return ORBIT_ERR_INVALID_ARGUMENT;
        for (uint32_t u = 0; u < v; ++u) if (task_payloads[v] && task_payloads[u] == task_payloads[v]) return ORBIT_ERR_INVALID_ARGUMENT;
    }
    if (capacity_records > 0xFFFFFFFFull) capacity_records = 0xFFFFFFFFull;
    GUARD(c);
    if (hizs && !c->views_pass2_configured) {   // the batched pass-2 test kernels' shared-memory opt-in, on first use
        CK(meshlet_cull_configure_views_pass2());
        c->views_pass2_configured = true;
    }
    // draw masks + side words of view v live at records [v * capacity_records, (v + 1) * capacity_records) of the grown scratch
    rc = ensure_record_scratch(c, (uint64_t)n_views * capacity_records);
    if (rc != ORBIT_OK) return rc;
    if (!c->view_counters) {   // first batched call: the counter block, zeroed in stream order ahead of the kernels
        CK(cudaMalloc(&c->view_counters, kViewCounterWords * sizeof(uint32_t)));
        CK(cudaMemsetAsync(c->view_counters, 0, kViewCounterWords * sizeof(uint32_t), (cudaStream_t)stream));
    }
    // emit: a row of CTAs per view. Every row gets the single-view grid, so a long list is walked by as many CTAs as a
    // single-view call gives it and the rows of short lists leave the machine to it (the lists of one batch differ by up to
    // four orders of magnitude: C5 cameras 1.4 k .. 9.4 M draws; rows of emit_grid / n_views CTAs made the 16-camera batch
    // 1.5x slower than separate calls, tools/bench_views.py). Short lists are emitted by small_grid / n_views CTAs of their
    // row, so a batch of short lists keeps the single-view number of working CTAs; the others leave at once.
    uint32_t small_grid;
    const uint64_t emit_grid = emit_grids(c, capacity_records, &small_grid);
    const uint32_t emit_per_view = (uint32_t)emit_grid;
    const uint32_t small_per_view = (small_grid + n_views - 1u) / n_views;
    MeshletViewsParams pv{};
    pv.n_views = n_views;
    for (uint32_t v = 0; v < n_views; ++v) {
        MeshletCullParams& p = pv.view[v];
        const OrbitSceneBuffers* scene = per_view_scene ? &scenes[v] : scenes;
        set_cull(p, &culls[v]);
        p.hiz = hiz_device(hizs ? hizs[v] : nullptr);
        p.dispatch_words = (const uint32_t*)dispatch_buffers[v];
        p.meshlets = (const uint4*)scene->meshlets;
        p.entities = (const float4*)scene->entities;
        p.materials = (const uint8_t*)scene->materials;
        p.meshlet_visibility = scene->meshlet_visibility;
        p.draw_words = (uint32_t*)draw_command_buffers[v];
        p.task_payloads = task_payloads ? (uint32_t*)task_payloads[v] : nullptr;
        p.overflow_flag = &c->status_dev->draw_overflow;
        p.draw_masks = c->draw_masks + (size_t)v * capacity_records;
        p.cmd_side = c->cmd_side + (size_t)v * capacity_records * 32u;
        p.chunk_counts = c->view_counters + v * kViewChunkWords;
        p.draw_total = c->view_counters + ORBIT_MAX_BATCH_VIEWS * kViewChunkWords + 4u * v;   // [0],[1]
        p.chunk_parity = p.draw_total + 2;                                                   // [2] word A, [3] word B
        p.capacity_records = capacity_records;
        p.capacity_draws = capacity_draws;
        p.emit_small_grid = small_per_view;
    }
    pv.view[0].scan.trace = next_trace(c);
    pv.view[0].trace_emit = next_trace(c);
    int& occ_slot = c->views_occupancy[meshlet_cull_variant_index(culls[0])];
    if (occ_slot <= 0) occ_slot = meshlet_cull_views_max_ctas_per_sm(culls[0]);
    int per_sm = c->mc_ctas_per_sm;
    if (per_sm <= 0) per_sm = occ_slot > 0 ? occ_slot : 1;
    CK(launch_meshlet_cull_views(pv, c->sm_count * per_sm, (int)emit_per_view, (cudaStream_t)stream));
    c->launches += 2;
    return ORBIT_OK;
}

int orbit_meshlet_cull_views(orbit_ctx* c, const OrbitCullInfo* culls, uint32_t n_views, const OrbitSceneBuffers* scene,
                             const void* const* dispatch_buffers, uint64_t capacity_records, void* const* draw_command_buffers,
                             uint64_t capacity_draws, void* const* task_payloads, void* stream) {
    if (!c) return ORBIT_ERR_INVALID_ARGUMENT;
    int rc = check_views(culls, n_views, scene, dispatch_buffers, true);
    if (rc != ORBIT_OK) return rc;
    return meshlet_views_stage(c, culls, n_views, scene, false, nullptr, dispatch_buffers, capacity_records, draw_command_buffers,
                               capacity_draws, task_payloads, stream);
}

// ---- batched two-pass occlusion views ----------------------------------------------------------------------
// Checks shared by both stages: view count; one pass (1 or 2), one projection type and one meshlet-occlusion setting for all
// views; check_cull per view; scenes[v] equal to scenes[0] except for the two visibility pointers, which no two views share (the
// entity stage's entity bits, the meshlet stage's meshlet words when meshlet occlusion is on); pass 2: one distinct pyramid per
// view, all of one geometry; one distinct, aligned output buffer per view.
static int check_views_occlusion(const OrbitCullInfo* culls, uint32_t n_views, const OrbitSceneBuffers* scenes, const orbit_hiz* const* hizs,
                                 const void* const* buffers, bool meshlet_stage) {
    if (!culls || !scenes || n_views == 0u || n_views > ORBIT_MAX_BATCH_VIEWS) return ORBIT_ERR_INVALID_ARGUMENT;
    const uint32_t pass = culls[0].occlusion_pass;
    const bool mocc = culls[0].meshlet_visibility_buffer != ORBIT_NO_BUFFER;
    if (pass != 1u && pass != 2u) return ORBIT_ERR_INVALID_ARGUMENT;
    if (pass == 2u && !hizs) return ORBIT_ERR_INVALID_ARGUMENT;
    for (uint32_t v = 0; v < n_views; ++v) {
        const OrbitCullInfo& ci = culls[v];
        if (ci.occlusion_pass != pass || ci.projection_type != culls[0].projection_type) return ORBIT_ERR_INVALID_ARGUMENT;
        if ((ci.meshlet_visibility_buffer != ORBIT_NO_BUFFER) != mocc) return ORBIT_ERR_INVALID_ARGUMENT;
        const orbit_hiz* h = pass == 2u ? hizs[v] : nullptr;
        if (pass == 2u) {
            if (!h || h->info.width != hizs[0]->info.width || h->info.height != hizs[0]->info.height || h->info.levels != hizs[0]->info.levels)
                return ORBIT_ERR_INVALID_ARGUMENT;
            for (uint32_t u = 0; u < v; ++u) if (hizs[u]->info.texels == h->info.texels) return ORBIT_ERR_INVALID_ARGUMENT;
        }
        int rc = check_cull(&ci, &scenes[v], h, meshlet_stage);
        if (rc != ORBIT_OK) return rc;
        OrbitSceneBuffers same = scenes[v];
        same.entity_visibility = scenes[0].entity_visibility; same.meshlet_visibility = scenes[0].meshlet_visibility;
        if (std::memcmp(&same, &scenes[0], sizeof(same)) != 0) return ORBIT_ERR_INVALID_ARGUMENT;
        for (uint32_t u = 0; u < v; ++u) {
            if (!meshlet_stage && scenes[u].entity_visibility == scenes[v].entity_visibility) return ORBIT_ERR_INVALID_ARGUMENT;
            if (meshlet_stage && mocc && scenes[u].meshlet_visibility == scenes[v].meshlet_visibility) return ORBIT_ERR_INVALID_ARGUMENT;
        }
    }
    return check_view_buffers(buffers, n_views);
}

int orbit_entity_cull_views_occlusion(orbit_ctx* c, const OrbitCullInfo* culls, uint32_t n_views, const OrbitSceneBuffers* scenes,
                                      const orbit_hiz* const* hizs, void* const* dispatch_buffers, uint64_t capacity_records, void* stream) {
    if (!c) return ORBIT_ERR_INVALID_ARGUMENT;
    int rc = check_views_occlusion(culls, n_views, scenes, hizs, (const void* const*)dispatch_buffers, false);
    if (rc != ORBIT_OK) return rc;
    uint32_t begin, end;
    rc = draw_range(&scenes[0], &begin, &end);
    if (rc != ORBIT_OK) return rc;
    const uint32_t n = end - begin, pass = culls[0].occlusion_pass;
    GUARD(c);
    rc = ensure_status(c, (size_t)n_views * ((n + 255u) / 256u + 1u), (cudaStream_t)stream);   // one descriptor block per view
    if (rc != ORBIT_OK) return rc;
    EntityViewsParams pv{};
    pv.n_views = n_views;
    for (uint32_t v = 0; v < n_views; ++v)
        pv.view[v] = entity_params(c, &culls[v], &scenes[v], pass == 2u ? hizs[v] : nullptr, dispatch_buffers[v], capacity_records, begin, end);
    pv.view[0].scan = next_scan(c);
    CK(launch_entity_cull_views(pv, n, entity_views_coresident_ctas(c, pass), (cudaStream_t)stream));
    c->launches += 1;
    return ORBIT_OK;
}

int orbit_meshlet_cull_views_occlusion(orbit_ctx* c, const OrbitCullInfo* culls, uint32_t n_views, const OrbitSceneBuffers* scenes,
                                       const orbit_hiz* const* hizs, const void* const* dispatch_buffers, uint64_t capacity_records,
                                       void* const* draw_command_buffers, uint64_t capacity_draws, void* const* task_payloads, void* stream) {
    if (!c) return ORBIT_ERR_INVALID_ARGUMENT;
    int rc = check_views_occlusion(culls, n_views, scenes, hizs, dispatch_buffers, true);
    if (rc != ORBIT_OK) return rc;
    const bool with_hiz = culls[0].occlusion_pass == 2u && culls[0].meshlet_visibility_buffer != ORBIT_NO_BUFFER;
    return meshlet_views_stage(c, culls, n_views, scenes, true, with_hiz ? hizs : nullptr, dispatch_buffers, capacity_records,
                               draw_command_buffers, capacity_draws, task_payloads, stream);
}

// ---- clustered lights ------------------------------------------------------------------------------------
int orbit_light_cluster(orbit_ctx* c, const OrbitClusterParams* params, const float* depth, const void* lights,
                        void* tile_masks, void* depth_bounds, void* unique_clusters, void* offset_count_image,
                        void* light_index_list, uint64_t capacity_indices, void* stream) {
    if (!c || !params || !depth || !tile_masks || !depth_bounds || !unique_clusters || !offset_count_image || !light_index_list)
        return ORBIT_ERR_INVALID_ARGUMENT;
    const OrbitClusterCullInfo& ci = params->info;
    const uint64_t cx = ci.cluster_count[0], cy = ci.cluster_count[1], cz = ci.cluster_count[2];
    if (cx == 0 || cy == 0 || cz == 0 || cx * cy * cz > 0x7FFFFFFFull || ci.tile_size_px == 0) return ORBIT_ERR_INVALID_ARGUMENT;
    if (ci.screen_size[0] == 0 || ci.screen_size[1] == 0) return ORBIT_ERR_INVALID_ARGUMENT;
    // every pixel must map to a tile inside the grid (cluster.rs:41-43 derives counts with div_ceil)
    if ((ci.screen_size[0] + ci.tile_size_px - 1u) / ci.tile_size_px > cx || (ci.screen_size[1] + ci.tile_size_px - 1u) / ci.tile_size_px > cy)
        return ORBIT_ERR_INVALID_ARGUMENT;
    const uint32_t L = ci.global_light_count;
    if (L != 0 && (!lights || ((uintptr_t)lights & 15u))) return ORBIT_ERR_INVALID_ARGUMENT;
    cudaStream_t s = (cudaStream_t)stream;
    const uint64_t clusters = cx * cy * cz;
    GUARD(c);
    const uint64_t hit_words = light_hits_words_needed(clusters, L);
    const bool light_parallel = L != 0u && hit_words * 4u <= c->light_hits_budget;
    int rc = light_parallel ? ensure_light_hits(c, hit_words) : ensure_lights(c, L);
    if (rc != ORBIT_OK) return rc;
    rc = ensure_status(c, (size_t)clusters + 1u, s);   // light culling scans one tile per active cluster
    if (rc != ORBIT_OK) return rc;
    ClusterParams p{};
    p.info = ci; p.z_scale = params->z_scale; p.z_bias = params->z_bias;
    p.depth = depth; p.lights = (const uint8_t*)lights; p.light_view = c->light_view;
    p.tile_masks = (uint32_t*)tile_masks; p.depth_bounds = (uint32_t*)depth_bounds;
    p.unique_clusters = (uint32_t*)unique_clusters; p.offset_count_image = (uint32_t*)offset_count_image;
    p.light_index_words = (uint32_t*)light_index_list; p.overflow_flag = &c->status_dev->light_index_overflow;
    p.capacity_indices = capacity_indices;
    // scratch of the light-parallel path: [boxes: 8 words per cluster][bit matrix][block counts][hit totals: 1 word per cluster]
    p.cluster_boxes = light_parallel ? reinterpret_cast<float4*>(c->light_hits) : nullptr;
    p.cluster_totals = light_parallel ? c->light_hits + clusters * (8u + (uint64_t)light_hits_blocks(L) * 17u) : nullptr;
    // fill_buffer(.., 0) of masks and bounds: cluster.rs:447-450; inactive image texels are zeroed (unspecified in the reference)
    CK(cudaMemsetAsync(tile_masks, 0, cx * cy * 4u, s));
    CK(cudaMemsetAsync(depth_bounds, 0, clusters * 8u, s));
    CK(cudaMemsetAsync(offset_count_image, 0, clusters * 8u, s));
    const uint64_t warps = (uint64_t)((ci.screen_size[0] + 31u) / 32u) * ((ci.screen_size[1] + 3u) / 4u);
    uint64_t grid = (warps + 7u) / 8u;
    const uint64_t cap_grid = (uint64_t)c->sm_count * 8u;
    if (grid > cap_grid) grid = cap_grid;
    CK(launch_mark_active(p, (int)grid, s));
    p.scan = next_scan(c);
    CK(launch_compact_clusters(p, s));
    if (light_parallel) {
        const uint32_t wpc = light_hits_blocks(L) * 16u;   // row stride of the bit matrix (64-byte aligned rows)
        uint32_t* const hit_rows = c->light_hits + clusters * 8u;
        uint32_t* const block_counts = hit_rows + clusters * wpc;
        CK(launch_light_hits(p, hit_rows, block_counts, wpc, (uint32_t)clusters, s));
        uint64_t lgrid = (clusters + 31u) / 32u;     // a warp per active cluster, 32 per CTA, persistent over tiles
        const uint64_t lcap = (uint64_t)c->sm_count * 2u;
        if (lgrid > lcap) lgrid = lcap;
        CK(launch_light_lists(p, hit_rows, block_counts, wpc, (int)lgrid, s));
        c->launches += 4;
    } else {
        CK(launch_light_view(p, s));
        p.scan = next_scan(c);
        uint64_t lgrid = clusters;                   // one CTA per active cluster, persistent: at most 2 x 1024 threads per SM
        const uint64_t lcap = (uint64_t)c->sm_count * 2u;
        if (lgrid > lcap) lgrid = lcap;
        CK(launch_light_culling(p, (int)lgrid, s));
        c->launches += (L ? 4 : 3);
    }
    return ORBIT_OK;
}

int orbit_draws_scatter(orbit_ctx* c, const void* src, uint64_t src_capacity_draws, void* dst, uint32_t dst_first, uint32_t total_count,
                        uint64_t dst_capacity_draws, void* stream) {
    if (!c || !src || !dst) return ORBIT_ERR_INVALID_ARGUMENT;
    GUARD(c);
    CK(launch_draws_scatter((const uint32_t*)src, src_capacity_draws, (uint32_t*)dst, dst_first, total_count, dst_capacity_draws,
                            c->sm_count * 16, (cudaStream_t)stream, nullptr, 0u, 0u));
    c->launches += 1;
    return ORBIT_OK;
}

int orbit_draws_scatter_ranked(orbit_ctx* c, const void* src, uint64_t src_capacity_draws, void* dst, const uint32_t* rank_counts, uint32_t rank, uint32_t world,
                               uint64_t dst_capacity_draws, void* stream) {
    if (!c || !src || !dst || !rank_counts || world == 0u || rank >= world) return ORBIT_ERR_INVALID_ARGUMENT;
    GUARD(c);
    CK(launch_draws_scatter((const uint32_t*)src, src_capacity_draws, (uint32_t*)dst, 0u, 0u, dst_capacity_draws, c->sm_count * 16, (cudaStream_t)stream,
                            rank_counts, rank, world));
    c->launches += 1;
    return ORBIT_OK;
}

int orbit_scene_update(orbit_ctx* c, const OrbitSceneUpdate* u, void* stream) {
    if (!c || !u) return ORBIT_ERR_INVALID_ARGUMENT;
    if (!u->entity_draws) return ORBIT_ERR_INVALID_ARGUMENT;
    GUARD(c);
    if (u->n_entities == 0u) {   // empty scene: only the count header is produced
        CK(cudaMemsetAsync(u->entity_draws, 0, 4, (cudaStream_t)stream));
        return ORBIT_OK;
    }
    if (!u->transforms || !u->mesh_slots || !u->visibility_offsets || !u->mesh_infos || !u->visibility_cursor || !u->entity_data)
        return ORBIT_ERR_INVALID_ARGUMENT;
    if (((uintptr_t)u->transforms | (uintptr_t)u->entity_data) & 15u) return ORBIT_ERR_INVALID_ARGUMENT;
    const size_t tiles = ((size_t)u->n_entities + 255u) / 256u;
    int rc = ensure_tile_sums(c, tiles);
    if (rc != ORBIT_OK) return rc;
    SceneUpdateParams p{};
    p.transforms = (const uint8_t*)u->transforms; p.mesh_slots = u->mesh_slots; p.visibility_offsets = u->visibility_offsets;
    p.mesh_infos = (const uint8_t*)u->mesh_infos; p.visibility_cursor = u->visibility_cursor;
    p.cursor_snapshot = c->counters + 8; p.tile_sums = c->tile_sums;
    p.entity_data = (float4*)u->entity_data; p.entity_draw_words = (uint32_t*)u->entity_draws;
    p.overflow_flag = &c->status_dev->visibility_overflow;
    p.n_entities = u->n_entities; p.visibility_capacity_words = u->visibility_capacity_words;
    CK(launch_scene_update(p, (cudaStream_t)stream));
    c->launches += 2;
    return ORBIT_OK;
}

int orbit_meshlet_bounds(orbit_ctx* c, const void* vertices, uint32_t vertex_stride, const uint32_t* meshlet_data, void* meshlets,
                         uint32_t n_meshlets, void* stream) {
    if (!c || !vertices || !meshlet_data || !meshlets || vertex_stride < 12u || (vertex_stride & 3u)) return ORBIT_ERR_INVALID_ARGUMENT;
    if (((uintptr_t)vertices & 3u) || ((uintptr_t)meshlet_data & 3u) || ((uintptr_t)meshlets & 15u)) return ORBIT_ERR_INVALID_ARGUMENT;
    if (n_meshlets == 0u) return ORBIT_OK;
    GUARD(c);
    MeshletBoundsParams p{};
    p.vertices = (const uint8_t*)vertices; p.vertex_stride = vertex_stride; p.meshlet_data = meshlet_data;
    p.meshlets = (uint8_t*)meshlets; p.n_meshlets = n_meshlets; p.error_flag = &c->status_dev->asset_error;
    uint64_t grid = ((uint64_t)n_meshlets + 3u) / 4u;
    const uint64_t cap = (uint64_t)c->sm_count * 16u;
    if (grid > cap) grid = cap;
    CK(launch_meshlet_bounds(p, (int)grid, (cudaStream_t)stream));
    c->launches += 1;
    return ORBIT_OK;
}

int orbit_mesh_bounds(orbit_ctx* c, const void* vertices, uint32_t vertex_stride, const uint32_t* vertex_ranges, void* mesh_infos,
                      uint32_t n_meshes, void* stream) {
    if (!c || !vertices || !vertex_ranges || !mesh_infos || vertex_stride < 12u || (vertex_stride & 3u)) return ORBIT_ERR_INVALID_ARGUMENT;
    if (((uintptr_t)vertices & 3u) || ((uintptr_t)vertex_ranges & 3u) || ((uintptr_t)mesh_infos & 15u)) return ORBIT_ERR_INVALID_ARGUMENT;
    if (n_meshes == 0u) return ORBIT_OK;
    GUARD(c);
    MeshBoundsParams p{};
    p.vertices = (const uint8_t*)vertices; p.vertex_stride = vertex_stride; p.vertex_ranges = vertex_ranges;
    p.mesh_infos = (uint8_t*)mesh_infos; p.n_meshes = n_meshes;
    uint64_t grid = n_meshes;
    const uint64_t cap = (uint64_t)c->sm_count * 8u;
    if (grid > cap) grid = cap;
    CK(launch_mesh_bounds(p, (int)grid, (cudaStream_t)stream));
    c->launches += 1;
    return ORBIT_OK;
}

int orbit_peer_alloc(orbit_ctx* c, uint64_t bytes, void** out_ptr, void* out_handle) {
    if (!c || !out_ptr || !out_handle || bytes == 0) return ORBIT_ERR_INVALID_ARGUMENT;
    GUARD(c);
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) { g_last_cuda_error = (int)e; return e == cudaErrorMemoryAllocation ? ORBIT_ERR_OUT_OF_MEMORY : ORBIT_ERR_CUDA; }
    cudaIpcMemHandle_t h;
    e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { g_last_cuda_error = (int)e; cudaFree(p); return ORBIT_ERR_CUDA; }
    static_assert(sizeof(h) == ORBIT_IPC_HANDLE_BYTES, "cudaIpcMemHandle_t is 64 bytes");
    std::memcpy(out_handle, &h, sizeof(h));
    *out_ptr = p;
    return ORBIT_OK;
}

int orbit_peer_open(orbit_ctx* c, const void* handle, void** out_ptr) {
    if (!c || !handle || !out_ptr) return ORBIT_ERR_INVALID_ARGUMENT;
    GUARD(c);
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, sizeof(h));
    CK(cudaIpcOpenMemHandle(out_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return ORBIT_OK;
}

int orbit_peer_close(orbit_ctx* c, void* mapped_ptr) {
    if (!c || !mapped_ptr) return ORBIT_ERR_INVALID_ARGUMENT;
    GUARD(c);
    CK(cudaIpcCloseMemHandle(mapped_ptr));
    return ORBIT_OK;
}

void orbit_peer_free(orbit_ctx* c, void* ptr) {
    if (!c || !ptr) return;
    DeviceGuard guard(c->device);
    cudaFree(ptr);
}

int orbit_device_copy(void* dst, const void* src, uint64_t bytes, void* stream) {
    if (!dst || !src) return ORBIT_ERR_INVALID_ARGUMENT;
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return ORBIT_OK;
}

}  // extern "C"

namespace orbit {
// Copies src's commands into dst at command index dst_first (peer-mapped dst allowed). The 28-byte commands start
// 4 bytes into both buffers and dst_first shifts the destination further, so source and destination are not
// mutually 16-byte aligned: the body issues ALIGNED 16-byte stores to the destination (what matters over NVLink),
// each assembled from four 4-byte loads of the local source; up to 3 head and 3 tail words go out as 4-byte stores.
// rank_counts != nullptr: dst_first and total_count come from the device (the all-gathered per-rank survivor counts):
// dst_first = sum of the counts of ranks below `rank`, total = sum over all `world` ranks — no host round trip.
// A count header may exceed its buffer's capacity after an overflow (the emit kernel stores the exact survivor count and
// drops the commands beyond capacity): every count read here — the source's own and the other ranks' — is clamped to
// src_capacity (the ranks of a sharded view use equal capacities), so nothing is read past a source buffer and the
// rank-major list has no gaps.
__global__ void __launch_bounds__(256) draws_scatter_kernel(const uint32_t* __restrict__ src, uint64_t src_capacity, uint32_t* __restrict__ dst,
                                                            uint32_t dst_first, uint32_t total_count, uint64_t dst_capacity,
                                                            const uint32_t* __restrict__ rank_counts, uint32_t rank, uint32_t world) {
    if (rank_counts) {
        uint32_t first = 0u, total = 0u;
        for (uint32_t r = 0; r < world; ++r) { const uint32_t c = (uint32_t)min((uint64_t)__ldcg(rank_counts + r), src_capacity); if (r < rank) first += c; total += c; }
        dst_first = first; total_count = total;
    }
    const uint32_t n = __ldcg(src);
    uint64_t m = min((uint64_t)n, src_capacity);
    if ((uint64_t)dst_first >= dst_capacity) m = 0; else if ((uint64_t)dst_first + m > dst_capacity) m = dst_capacity - dst_first;
    const uint64_t words = m * 7u;
    const uint32_t* s = src + 1;
    uint32_t* d = dst + 1u + (uint64_t)dst_first * 7u;
    const uint64_t gtid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, gsize = (uint64_t)gridDim.x * blockDim.x;
    // head: words until d + head is 16-byte aligned
    uint64_t head = ((16u - ((uintptr_t)d & 15u)) & 15u) >> 2;
    if (head > words) head = words;
    const uint64_t body4 = (words - head) >> 2;           // number of aligned uint4 stores
    if (gtid < head) d[gtid] = __ldcg(s + gtid);
    uint4* d4 = reinterpret_cast<uint4*>(d + head);
    const uint32_t* sb = s + head;
    // four independent 16-byte stores per thread and iteration: remote (NVLink) stores need many of them in flight
    uint64_t i = gtid;
    for (; i + 3u * gsize < body4; i += 4u * gsize) {
        uint4 v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t* q = sb + 4u * (i + (uint64_t)k * gsize);
            v[k] = make_uint4(__ldcg(q), __ldcg(q + 1), __ldcg(q + 2), __ldcg(q + 3));
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) __stcg(d4 + i + (uint64_t)k * gsize, v[k]);
    }
    for (; i < body4; i += gsize) {
        const uint32_t a = __ldcg(sb + 4u * i), b = __ldcg(sb + 4u * i + 1u), c = __ldcg(sb + 4u * i + 2u), e = __ldcg(sb + 4u * i + 3u);
        __stcg(d4 + i, make_uint4(a, b, c, e));
    }
    const uint64_t done = head + 4u * body4;
    if (gtid < words - done) d[done + gtid] = __ldcg(s + done + gtid);
    if (blockIdx.x == 0 && threadIdx.x == 0 && total_count != 0xFFFFFFFFu) dst[0] = total_count;
}
cudaError_t launch_draws_scatter(const uint32_t* src, uint64_t src_capacity, uint32_t* dst, uint32_t dst_first, uint32_t total_count,
                                 uint64_t dst_capacity, int grid, cudaStream_t s, const uint32_t* rank_counts, uint32_t rank, uint32_t world) {
    draws_scatter_kernel<<<grid, 256, 0, s>>>(src, src_capacity, dst, dst_first, total_count, dst_capacity, rank_counts, rank, world);
    return cudaGetLastError();
}
}  // namespace orbit

// ---- peer put / wait: one-sided transfers with a completion flag (no collective) ---------------------------------------
// orbit_peer_put: up to 16 transfers in one launch (blockIdx.y = transfer). A transfer copies `bytes` (multiple of 16, both
// ends 16-byte aligned) from local memory to `dst` — usually another GPU's memory mapped with orbit_peer_open, so the stores
// travel over NVLink — and, once every CTA of the transfer has issued and fenced its stores (the last one to count itself
// out knows), writes `flag_value` to `dst_flag` on the receiving GPU. orbit_peer_wait makes the stream wait until n local
// flag words all hold `flag_value` (a one-warp kernel polling with ld.acquire.sys). Flags only ever take the values the
// callers pass, so a monotonically increasing value per use needs no reset. The wait is bounded (~2 s): a peer that never
// arrives sets OrbitStatus::peer_timeout instead of hanging the GPU.
namespace orbit {
struct PeerPutParams { const uint4* src[16]; uint4* dst[16]; uint64_t n16[16]; uint32_t* flag[16]; uint32_t flag_value; uint32_t* done; };

__global__ void __launch_bounds__(256) peer_put_kernel(const __grid_constant__ PeerPutParams p) {
    const uint32_t t = blockIdx.y;
    const uint4* __restrict__ src = p.src[t];
    uint4* __restrict__ dst = p.dst[t];
    const uint64_t n = p.n16[t], gsize = (uint64_t)gridDim.x * blockDim.x;
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + 3u * gsize < n; i += 4u * gsize) {                       // four independent 16-byte stores in flight
        uint4 v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = __ldcg(src + i + (uint64_t)k * gsize);
#pragma unroll
        for (int k = 0; k < 4; ++k) __stcg(dst + i + (uint64_t)k * gsize, v[k]);
    }
    for (; i < n; i += gsize) __stcg(dst + i, __ldcg(src + i));
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int prev = atomicAdd(p.done + t, 1u);
        if (prev + 1u == gridDim.x) {
            p.done[t] = 0u;
            __threadfence_system();
            if (p.flag[t] != nullptr) asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p.flag[t]), "r"(p.flag_value) : "memory");
        }
    }
}

__global__ void __launch_bounds__(32) peer_wait_kernel(const uint32_t* flags, uint32_t n, uint32_t stride, uint32_t value, uint32_t* timeout_flag) {
    const uint32_t lane = threadIdx.x;
    bool ok = lane >= n;
    for (uint32_t spin = 0; spin < (1u << 22) && !__all_sync(0xFFFFFFFFu, ok); ++spin) {
        if (!ok) {
            uint32_t v;
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flags + (size_t)lane * stride) : "memory");
            ok = v == value;
            if (!ok) __nanosleep(200);
        }
    }
    if (!__all_sync(0xFFFFFFFFu, ok) && lane == 0) *timeout_flag = 1u;
    __threadfence_system();
}
}  // namespace orbit

extern "C" {
int orbit_peer_put(orbit_ctx* c, const OrbitPeerPut* puts, uint32_t n_puts, uint32_t flag_value, void* stream) {
    if (!c || !puts || n_puts == 0u || n_puts > 16u) return ORBIT_ERR_INVALID_ARGUMENT;
    orbit::PeerPutParams p{};
    uint64_t largest = 0u;
    for (uint32_t i = 0; i < n_puts; ++i) {
        if ((!puts[i].src || !puts[i].dst) && puts[i].bytes) return ORBIT_ERR_INVALID_ARGUMENT;
        if ((((uintptr_t)puts[i].src | (uintptr_t)puts[i].dst | puts[i].bytes) & 15u) || ((uintptr_t)puts[i].dst_flag & 3u)) return ORBIT_ERR_INVALID_ARGUMENT;
        p.src[i] = (const uint4*)puts[i].src; p.dst[i] = (uint4*)puts[i].dst; p.n16[i] = puts[i].bytes / 16u; p.flag[i] = puts[i].dst_flag;
        if (p.n16[i] > largest) largest = p.n16[i];
    }
    p.flag_value = flag_value;
    p.done = c->counters + 24;                 // [24..39]: CTAs that have finished, per transfer (self-resetting)
    GUARD(c);
    uint64_t gx = (largest + 1023u) / 1024u;   // four 16-byte stores per thread
    const uint64_t cap = (uint64_t)c->sm_count * 8u / n_puts;
    if (gx > cap) gx = cap;
    if (gx == 0u) gx = 1u;
    orbit::peer_put_kernel<<<dim3((unsigned)gx, n_puts), 256, 0, (cudaStream_t)stream>>>(p);
    CK(cudaGetLastError());
    c->launches += 1;
    return ORBIT_OK;
}

int orbit_peer_wait(orbit_ctx* c, const uint32_t* flags, uint32_t n_flags, uint32_t stride_words, uint32_t flag_value, void* stream) {
    if (!c || !flags || n_flags == 0u || n_flags > 32u || stride_words == 0u || ((uintptr_t)flags & 3u)) return ORBIT_ERR_INVALID_ARGUMENT;
    GUARD(c);
    orbit::peer_wait_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(flags, n_flags, stride_words, flag_value, &c->status_dev->peer_timeout);
    CK(cudaGetLastError());
    c->launches += 1;
    return ORBIT_OK;
}
}  // extern "C"
