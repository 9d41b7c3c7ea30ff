// frame_driver.cpp — compiled host side of one culled frame, above the C ABI (include/orbit_cuda.h).
//
// The reference's host is compiled code (Rust: SceneData::update_scene, scene.rs:404-492, then the depth-prepass
// culling passes of forward.rs:266-403 recorded every frame). This is its stand-in for end-to-end measurements: a
// software-pipelined frame loop with HOST inputs and outputs — per step: pinned-host Transforms + depth buffer ->
// device, orbit_scene_update, EARLY entity+meshlet cull, Hi-Z build, LATE entity+meshlet cull, MAIN entity+meshlet cull
// (forward.rs:518-548: pass 1 again with the bits the late pass wrote), the three survivor counts and lists -> pinned host — with `lookahead` steps enqueued ahead of the one being read back, each on
// its own copy of the scene/view buffers. Three streams: copy-in, compute, copy-out. No kernels here; every GPU
// operation is a C-ABI stage call or a cudaMemcpyAsync. Built into liborbit_host.so by orbit_b200/build.py.
#include <cuda_runtime.h>

#include <chrono>
#include <cstdint>
#include <cstring>
#include <deque>

#include "orbit_cuda.h"

extern "C" {

// Everything one in-flight step needs (one per scene copy). Device pointers unless noted.
typedef struct OrbitHostFrame {
    OrbitSceneUpdate update;            // transforms / entity buffers of this copy
    OrbitCullInfo cull_early, cull_late;
    OrbitSceneBuffers scene_early, scene_late;
    orbit_hiz* hiz;
    float* depth;                       // W x H f32
    void *early_dispatch, *early_draws, *late_dispatch, *late_draws, *main_dispatch, *main_draws;
    uint64_t capacity_records, capacity_draws;
    uint32_t width, height;
} OrbitHostFrame;

typedef struct OrbitHostFrameIO {
    const void* h_transforms;           // pinned host, n_entities x 48 B
    const float* h_depth;               // pinned host, W x H f32
    uint32_t* h_counts;                 // pinned host, 3 words (early, late, main)
    void* h_early_draws;                // pinned host, 28 B x capacity
    void* h_late_draws;
    void* h_main_draws;
    uint32_t depth_resident;            // != 0: the depth buffer already lives on the device (what Vulkan interop gives): not copied
    uint32_t reserved;
    uint64_t h2d_bytes_per_step;        // out
    uint64_t d2h_bytes_last_step;       // out
    double ms_per_step;                 // out: host wall clock over `steps`, everything drained
} OrbitHostFrameIO;

// sizeof probes for the ctypes mirrors (orbit_b200/layouts.py: HostFrame, HostFrameIO)
uint32_t orbit_host_sizeof_frame(void) { return (uint32_t)sizeof(OrbitHostFrame); }
uint32_t orbit_host_sizeof_io(void) { return (uint32_t)sizeof(OrbitHostFrameIO); }

// Pinned host staging memory for the loop's inputs. write_combined != 0: cudaHostAllocWriteCombined — the CPU only ever
// writes these buffers and the copy engines read them without snooping the CPU caches, which is what limits the aggregate
// host-to-device rate when several GPUs pull their inputs at once.
void* orbit_host_pinned_alloc(uint64_t bytes, int write_combined) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, write_combined ? cudaHostAllocWriteCombined : cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
void orbit_host_pinned_free(void* p) { if (p) cudaFreeHost(p); }

#define CU_OK(x) do { if ((x) != cudaSuccess) return ORBIT_ERR_CUDA; } while (0)
#define OR_OK(x) do { int rc_ = (x); if (rc_ != ORBIT_OK) return rc_; } while (0)

int orbit_host_frame_loop(orbit_ctx* ctx, const OrbitHostFrame* frames, uint32_t n_frames, OrbitHostFrameIO* io,
                          uint32_t steps, uint32_t lookahead) {
    if (!ctx || !frames || !io || n_frames == 0 || lookahead + 2 > n_frames) return ORBIT_ERR_INVALID_ARGUMENT;
    cudaStream_t s_in, s_comp, s_out;
    CU_OK(cudaStreamCreateWithFlags(&s_in, cudaStreamNonBlocking));
    CU_OK(cudaStreamCreateWithFlags(&s_comp, cudaStreamNonBlocking));
    CU_OK(cudaStreamCreateWithFlags(&s_out, cudaStreamNonBlocking));
    cudaEvent_t ev_in[16], ev_done[16], ev_free[16];
    if (n_frames > 16) return ORBIT_ERR_INVALID_ARGUMENT;
    for (uint32_t i = 0; i < n_frames; ++i) {
        CU_OK(cudaEventCreateWithFlags(&ev_in[i], cudaEventDisableTiming));
        CU_OK(cudaEventCreateWithFlags(&ev_done[i], cudaEventDisableTiming));
        CU_OK(cudaEventCreateWithFlags(&ev_free[i], cudaEventDisableTiming));
        CU_OK(cudaEventRecord(ev_free[i], s_out));
    }
    const size_t transform_bytes = (size_t)frames[0].update.n_entities * sizeof(OrbitTransform);
    const size_t depth_bytes = (size_t)frames[0].width * frames[0].height * sizeof(float);
    io->h2d_bytes_per_step = transform_bytes + (io->depth_resident ? 0 : depth_bytes);

    auto enqueue = [&](uint32_t step) -> int {
        const uint32_t k = step % n_frames;
        const OrbitHostFrame& f = frames[k];
        CU_OK(cudaStreamWaitEvent(s_in, ev_free[k], 0));          // this copy's previous outputs have been read back
        CU_OK(cudaMemcpyAsync((void*)f.update.transforms, io->h_transforms, transform_bytes, cudaMemcpyHostToDevice, s_in));
        if (!io->depth_resident) CU_OK(cudaMemcpyAsync(f.depth, io->h_depth, depth_bytes, cudaMemcpyHostToDevice, s_in));
        CU_OK(cudaEventRecord(ev_in[k], s_in));
        CU_OK(cudaStreamWaitEvent(s_comp, ev_in[k], 0));
        OR_OK(orbit_scene_update(ctx, &f.update, s_comp));
        OR_OK(orbit_entity_cull(ctx, &f.cull_early, &f.scene_early, nullptr, f.early_dispatch, f.capacity_records, s_comp));
        OR_OK(orbit_meshlet_cull(ctx, &f.cull_early, &f.scene_early, nullptr, f.early_dispatch, f.capacity_records, f.early_draws,
                                 f.capacity_draws, nullptr, s_comp));
        // Hi-Z build + LATE entity stage in one call (the entity kernel's pyramid-independent work runs under the build)
        if (orbit_cull_pair_compatible(&f.cull_late, &f.cull_early)) {
            // LATE + MAIN (= pass 1 again, the EARLY CullInfo) fused: one entity kernel, one test kernel, an emit kernel per list
            OR_OK(orbit_hiz_build_entity_cull_late(ctx, f.hiz, f.depth, f.width, f.height, &f.cull_late, &f.cull_early, &f.scene_late,
                                                   f.late_dispatch, f.main_dispatch, f.capacity_records, s_comp));
            OR_OK(orbit_meshlet_cull_late_main(ctx, &f.cull_late, &f.cull_early, &f.scene_late, f.hiz, f.late_dispatch, f.capacity_records,
                                               f.late_draws, f.main_draws, f.capacity_draws, nullptr, nullptr, s_comp));
        } else {
            OR_OK(orbit_hiz_build_entity_cull_late(ctx, f.hiz, f.depth, f.width, f.height, &f.cull_late, nullptr, &f.scene_late,
                                                   f.late_dispatch, nullptr, f.capacity_records, s_comp));
            OR_OK(orbit_meshlet_cull(ctx, &f.cull_late, &f.scene_late, f.hiz, f.late_dispatch, f.capacity_records, f.late_draws,
                                     f.capacity_draws, nullptr, s_comp));
            OR_OK(orbit_entity_cull(ctx, &f.cull_early, &f.scene_early, nullptr, f.main_dispatch, f.capacity_records, s_comp));   // MAIN = pass 1 again
            OR_OK(orbit_meshlet_cull(ctx, &f.cull_early, &f.scene_early, nullptr, f.main_dispatch, f.capacity_records, f.main_draws,
                                     f.capacity_draws, nullptr, s_comp));
        }
        CU_OK(cudaEventRecord(ev_done[k], s_comp));
        return ORBIT_OK;
    };
    auto readback = [&](uint32_t step) -> int {
        const uint32_t k = step % n_frames;
        const OrbitHostFrame& f = frames[k];
        CU_OK(cudaStreamWaitEvent(s_out, ev_done[k], 0));
        CU_OK(cudaMemcpyAsync(io->h_counts, f.early_draws, 4, cudaMemcpyDeviceToHost, s_out));
        CU_OK(cudaMemcpyAsync(io->h_counts + 1, f.late_draws, 4, cudaMemcpyDeviceToHost, s_out));
        CU_OK(cudaMemcpyAsync(io->h_counts + 2, f.main_draws, 4, cudaMemcpyDeviceToHost, s_out));
        CU_OK(cudaStreamSynchronize(s_out));
        uint64_t ne = io->h_counts[0], nl = io->h_counts[1], nm = io->h_counts[2];
        if (ne > f.capacity_draws) ne = f.capacity_draws;
        if (nl > f.capacity_draws) nl = f.capacity_draws;
        if (nm > f.capacity_draws) nm = f.capacity_draws;
        if (nm) CU_OK(cudaMemcpyAsync(io->h_main_draws, (const char*)f.main_draws + 4, 28 * nm, cudaMemcpyDeviceToHost, s_out));
        if (ne) CU_OK(cudaMemcpyAsync(io->h_early_draws, (const char*)f.early_draws + 4, 28 * ne, cudaMemcpyDeviceToHost, s_out));
        if (nl) CU_OK(cudaMemcpyAsync(io->h_late_draws, (const char*)f.late_draws + 4, 28 * nl, cudaMemcpyDeviceToHost, s_out));
        CU_OK(cudaEventRecord(ev_free[k], s_out));
        io->d2h_bytes_last_step = 12 + 28 * (ne + nl + nm);
        return ORBIT_OK;
    };

    CU_OK(cudaDeviceSynchronize());
    const auto t0 = std::chrono::steady_clock::now();
    uint32_t issued = 0;
    for (; issued < lookahead && issued < steps; ++issued) OR_OK(enqueue(issued));
    for (uint32_t i = 0; i < steps; ++i) {
        if (issued < steps) { OR_OK(enqueue(issued)); ++issued; }
        OR_OK(readback(i));
    }
    CU_OK(cudaDeviceSynchronize());
    io->ms_per_step = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count() / (steps ? steps : 1);
    for (uint32_t i = 0; i < n_frames; ++i) { cudaEventDestroy(ev_in[i]); cudaEventDestroy(ev_done[i]); cudaEventDestroy(ev_free[i]); }
    cudaStreamDestroy(s_in); cudaStreamDestroy(s_comp); cudaStreamDestroy(s_out);
    return ORBIT_OK;
}

}  // extern "C"
