// Host-side helpers shared by the C-ABI translation units: grow-only device scratch buffers
// for the host-pointer (Level-1 / end-to-end) entry points and the global lock that
// serialises them. Device-pointer (Level-2) entry points never touch these.
#pragma once
#include "common.cuh"
#include "launch_count.h"
#include "../../include/b200av1.h"
#include <mutex>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

namespace b200 {

struct Scratch {
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t n) {
        if (n <= cap) return 0;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = n + (n >> 2) + 4096;
        B200_CUDA_OK(cudaMalloc(&p, want));
        cap = want;
        return 0;
    }
    // host -> device (async on stream 0)
    int upload(const void *src, size_t n) {
        if (reserve(n)) return -1;
        if (n) B200_CUDA_OK(cudaMemcpyAsync(p, src, n, cudaMemcpyHostToDevice, 0));
        return 0;
    }
    int download(void *dst, size_t n) {
        if (n) B200_CUDA_OK(cudaMemcpyAsync(dst, p, n, cudaMemcpyDeviceToHost, 0));
        return 0;
    }
};

std::mutex &host_lock();

// row-range forms of the frame-wide sweeps (a band of a frame job, frame.cu; the b200_*_frame entry points pass the whole range)
int lf_frame_rows(int bdmax, const B200LfFrame *f, int ya4, int yb4, cudaStream_t stream);
// band-sliced intra stage (intra.cu): the records of one band (first: the done map is set up from done_init / zeroed
// first, also when the band has no records), and the edge rows the band below reads (intra.scratch header -> band y1)
int intra_band(int bdmax, const B200IntraFrame *f, const B200IntraTx *d_tx, int n, bool first, cudaStream_t stream);
int intra_edge_backup(int bdmax, const B200IntraFrame *f, int y1, void *edge, cudaStream_t stream);
int cdef_frame_rows(int bdmax, const B200CdefFrame *f, int t0, int t1, cudaStream_t stream);
int lr_frame_rows(int bdmax, const B200LrFrame *f, int r0, int r1, cudaStream_t stream);

[[noreturn]] inline void die(const char *what) {
    fprintf(stderr, "b200av1: %s failed: %s\n", what, b200_last_error());
    abort();
}

// copy a w x h rectangle of `px`-byte pixels between a strided (possibly negative stride, bytes)
// picture and a dense buffer
inline void pack_rect(void *dense, const void *pic, ptrdiff_t stride, int w, int h, size_t px) {
    for (int y = 0; y < h; y++)
        memcpy((uint8_t *)dense + (size_t)y * w * px, (const uint8_t *)pic + (ptrdiff_t)y * stride, (size_t)w * px);
}
inline void unpack_rect(void *pic, ptrdiff_t stride, const void *dense, int w, int h, size_t px) {
    for (int y = 0; y < h; y++)
        memcpy((uint8_t *)pic + (ptrdiff_t)y * stride, (const uint8_t *)dense + (size_t)y * w * px, (size_t)w * px);
}

}  // namespace b200

#ifndef B200_EMU
#include <map>
// A side stream + fork/join events per (caller stream, slot): lets a stage that is latency bound on few CTAs run
// beside the next stage instead of in front of it. fork(): side waits for everything enqueued on `main` so far;
// join(): `main` waits for everything enqueued on the side stream.
struct SideStream {
    cudaStream_t side = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    bool fork(cudaStream_t main) {
        return cudaEventRecord(ev_fork, main) == cudaSuccess && cudaStreamWaitEvent(side, ev_fork, 0) == cudaSuccess;
    }
    bool join(cudaStream_t main) {
        return cudaEventRecord(ev_join, side) == cudaSuccess && cudaStreamWaitEvent(main, ev_join, 0) == cudaSuccess;
    }
};
inline SideStream *side_stream_for(cudaStream_t main, int slot)
{
    static std::map<std::pair<cudaStream_t, int>, SideStream> pool;
    static std::mutex mu;
    std::lock_guard<std::mutex> lk(mu);
    auto key = std::make_pair(main, slot);
    auto it = pool.find(key);
    if (it != pool.end()) return &it->second;
    SideStream s;
    if (cudaStreamCreateWithFlags(&s.side, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&s.ev_fork, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&s.ev_join, cudaEventDisableTiming) != cudaSuccess) return nullptr;
    return &(pool[key] = s);
}
#endif
