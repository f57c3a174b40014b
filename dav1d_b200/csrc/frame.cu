// Whole-frame job: sequences the batched kernels of one frame on a stream (include/b200av1.h,
// B200FrameJob). The device-side counterpart of dav1d's per-frame task graph
// (TILE_RECONSTRUCTION -> DEBLOCK_COLS -> DEBLOCK_ROWS -> CDEF -> LOOP_RESTORATION,
// reference src/thread_task.c:699-854) with whole-frame stages instead of superblock rows.
#include "host_util.h"

extern "C" {

// the stages before intra reconstruction; *fg_side is set when the film grain preparation was forked to a side stream
static int frame_phase_recon(const B200FrameJob *j, void *stream, void **fg_side)
{
    int r;
    const int bd = j->bitdepth_max;
    *fg_side = nullptr;
#ifndef B200_EMU
    // film grain LUT preparation: one CTA, latency bound, depends only on the frame header -> side stream. The
    // scratch is reused frame after frame on this stream, hence the fork (after everything enqueued so far).
    SideStream *fs = nullptr;
    if (j->run_fg && (fs = side_stream_for((cudaStream_t)stream, 0)) && fs->fork((cudaStream_t)stream)) {
        if ((r = b200_fg_prep(bd, &j->fg, fs->side))) return r;
        *fg_side = fs;
    }
#endif
    if (j->n_expand > 0) {
        B200_CUDA_OK(cudaMemsetAsync(j->d_coef, 0, j->coef_bytes, (cudaStream_t)stream));
        if ((r = b200_coef_expand(bd, j->d_expand, j->n_expand, j->d_ccoef, j->d_coef, stream))) return r;
    }
    if ((r = b200_mc_batch(bd, &j->mc, j->d_pred, j->n_pred, stream))) return r;
    if ((r = b200_mc_scaled_batch(bd, &j->mc, j->d_scaled, j->n_scaled, stream))) return r;
    if ((r = b200_mc_warp_batch(bd, &j->mc, j->d_warp, j->n_warp, stream))) return r;
    if ((r = b200_mc_comp_fused_batch(bd, &j->mc, j->d_cfused, j->n_cfused, stream))) return r;
    if ((r = b200_mc_comp_fused_batch(bd, &j->mc, j->d_cfused2, j->n_cfused2, stream))) return r;
    if ((r = b200_mc_comp_batch(bd, &j->mc, j->d_comp, j->n_comp, stream))) return r;
    if ((r = b200_mc_comp_batch(bd, &j->mc, j->d_comp2, j->n_comp2, stream))) return r;
    if ((r = b200_mc_blend_batch(bd, &j->mc, j->d_blend, j->n_blend, stream))) return r;
    if ((r = b200_mc_blend_batch(bd, &j->mc, j->d_blend2, j->n_blend2, stream))) return r;
    if ((r = b200_itx_add_frame(bd, (const void *const *)j->d_itx, j->n_itx, j->d_coef, j->mc.dst, j->itx_stride,
                                j->zero_coefs, stream)))
        return r;
    return 0;
}

static int frame_phase_post(const B200FrameJob *j, void *stream, void *fg_side)
{
    int r;
    const int bd = j->bitdepth_max;
    if (j->run_lf && (r = b200_lf_frame(bd, &j->lf, stream))) return r;
    if (j->run_cdef && (r = b200_cdef_frame(bd, &j->cdef, stream))) return r;
    if (j->run_resize) {                     // super-resolution: CDEF output (and the deblocked picture LR reads) upscaled
        if ((r = b200_resize_frame(bd, &j->resize[0], stream))) return r;
        if ((r = b200_resize_frame(bd, &j->resize[1], stream))) return r;
    }
    if (j->run_lr && (r = b200_lr_frame(bd, &j->lr, stream))) return r;
    if (j->run_fg) {
#ifndef B200_EMU
        if (fg_side && !((SideStream *)fg_side)->join((cudaStream_t)stream)) { b200_set_error("b200_frame_run: stream join failed"); return -1; }
#endif
        if (!fg_side && (r = b200_fg_prep(bd, &j->fg, stream))) return r;
        if ((r = b200_fg_apply(bd, &j->fg, stream))) return r;
    }
    return 0;
}

int b200_frame_run(const B200FrameJob *j, void *stream)
{
    int r;
    void *fg_side;
    if ((r = frame_phase_recon(j, stream, &fg_side))) return r;
    if (j->n_intra > 0 && (r = b200_intra_frame(j->bitdepth_max, &j->intra, j->d_intra, j->n_intra, stream))) return r;
    return frame_phase_post(j, stream, fg_side);
}

int b200_frame_run_batch(const B200FrameJob *const *jobs, int n, void *stream)
{
    if (n <= 0) return 0;
    if (n > 256) { b200_set_error("b200_frame_run_batch: too many jobs"); return -2; }
    int r;
    void *fg_side[256];
    B200IntraFrame frames[256];
    const B200IntraTx *tx[256];
    int32_t ntx[256];
    for (int i = 0; i < n; i++) {
        if (jobs[i]->bitdepth_max != jobs[0]->bitdepth_max) { b200_set_error("b200_frame_run_batch: mixed bit depths"); return -2; }
        if (jobs[i]->run_fg) { b200_set_error("b200_frame_run_batch: film grain jobs must be run one by one"); return -2; }
        if ((r = frame_phase_recon(jobs[i], stream, &fg_side[i]))) return r;
        frames[i] = jobs[i]->intra; tx[i] = jobs[i]->d_intra; ntx[i] = jobs[i]->n_intra;
    }
    if ((r = b200_intra_frames(jobs[0]->bitdepth_max, frames, tx, ntx, n, stream))) return r;
    for (int i = 0; i < n; i++)
        if ((r = frame_phase_post(jobs[i], stream, fg_side[i]))) return r;
    return 0;
}

// ---- band-sliced job (include/b200av1.h, B200FrameBand) --------------------------------------------------------
static int job_luma_h(const B200FrameJob *j) { return j->lr.h > 0 ? j->lr.h : j->lf.h4 * 4; }

int b200_band_progress(const B200FrameJob *j, int y1, int last, int plane)
{
    const int ssv = plane ? j->lf.ss_ver : 0;
    const int ph = (job_luma_h(j) + ssv) >> ssv;
    if (last) return ph;
    int p;
    if (j->run_lr)        p = ssv ? (y1 >> 1) - 36 : (y1 <= 64 ? 0 : y1 - 40);   // the last tile row that could run (see b200_frame_run_band)
    else if (j->run_cdef) p = (y1 - 32) >> ssv;
    else if (j->run_lf)   p = ssv ? (y1 >> 1) - 4 : y1 - 8;        // a row edge at y1 still changes up to 6 (chroma: 2) rows above it
    else                  p = y1 >> ssv;
    return p < 0 ? 0 : (p > ph ? ph : p);
}

int b200_frame_run_band(const B200FrameJob *j, const B200FrameBand *b, void *stream)
{
    return b200_frame_run_band_phase(j, b, B200_BAND_RECON | B200_BAND_POST, stream);
}

int b200_frame_run_band_phase(const B200FrameJob *j, const B200FrameBand *b, int phases, void *stream)
{
    int r;
    const bool do_recon = phases & B200_BAND_RECON, do_post = phases & B200_BAND_POST;
    const int bd = j->bitdepth_max;
    const int H = job_luma_h(j);
    if ((b->y0 & 63) || b->y0 < 0 || b->y1 <= b->y0 || (!b->last && (b->y1 & 63)) || (b->last && b->y1 < H)) {
        b200_set_error("b200_frame_run_band: band [%d, %d) must be 64-row aligned (last band: down to the picture height %d)", b->y0, b->y1, H);
        return -2;
    }
    const bool first = b->y0 == 0;
    // intra records: the band's own range of d_intra, in a topological order of the dependencies inside the band (those on
    // the bands above are met); a record on the band's first row reads its top edge from the rows the band above saved
    if (j->n_intra > 0) {
        if (b->intra[0] < 0 || b->intra[1] < 0 || b->intra[1] > j->n_intra - b->intra[0]) {
            b200_set_error("b200_frame_run_band: intra records [%d, +%d) outside [0, %d)", b->intra[0], b->intra[1], j->n_intra);
            return -2;
        }
        if (j->intra.sb && !(first && b->last)) { b200_set_error("b200_frame_run_band: the superblock-granular intra schedule is not band-sliced (one band, or b200_frame_run)"); return -2; }
        if (!first && b->intra[1] > 0 && !b->edge_top) { b200_set_error("b200_frame_run_band: band [%d, %d) has intra records but no edge_top", b->y0, b->y1); return -2; }
        if (!b->last && !b->edge_bottom) { b200_set_error("b200_frame_run_band: band [%d, %d) of a job with intra records has no edge_bottom", b->y0, b->y1); return -2; }
    }
    if (j->run_resize) { b200_set_error("b200_frame_run_band: the super-resolution stage is not band-sliced (b200_frame_run)"); return -2; }
    // (the grain LUTs belong to the post phase: its stream forks the preparation beside the first band and joins it before
    // the last band's application)
#ifndef B200_EMU
    bool fg_forked = false;
    if (do_post && first && j->run_fg) {       // grain LUTs depend on the frame header only
        SideStream *fs = side_stream_for((cudaStream_t)stream, 0);
        if (fs && fs->fork((cudaStream_t)stream)) { if ((r = b200_fg_prep(bd, &j->fg, fs->side))) return r; fg_forked = true; }
    }
    if (do_post && first && j->run_fg && !fg_forked && (r = b200_fg_prep(bd, &j->fg, stream))) return r;
#else
    if (do_post && first && j->run_fg && (r = b200_fg_prep(bd, &j->fg, stream))) return r;
#endif
    if (do_recon) {
    if (first && j->n_expand > 0) B200_CUDA_OK(cudaMemsetAsync(j->d_coef, 0, j->coef_bytes, (cudaStream_t)stream));
#define SUB(ptr, rng) ((ptr) ? (ptr) + (rng)[0] : (ptr)), ((ptr) ? (rng)[1] : 0)
    if (j->n_expand > 0 && (r = b200_coef_expand(bd, SUB(j->d_expand, b->expand), j->d_ccoef, j->d_coef, stream))) return r;
    if ((r = b200_mc_batch(bd, &j->mc, SUB(j->d_pred, b->pred), stream))) return r;
    if ((r = b200_mc_scaled_batch(bd, &j->mc, SUB(j->d_scaled, b->scaled), stream))) return r;
    if ((r = b200_mc_warp_batch(bd, &j->mc, SUB(j->d_warp, b->warp), stream))) return r;
    if ((r = b200_mc_comp_fused_batch(bd, &j->mc, SUB(j->d_cfused, b->cfused), stream))) return r;
    if ((r = b200_mc_comp_fused_batch(bd, &j->mc, SUB(j->d_cfused2, b->cfused2), stream))) return r;
    if ((r = b200_mc_comp_batch(bd, &j->mc, SUB(j->d_comp, b->comp), stream))) return r;
    if ((r = b200_mc_comp_batch(bd, &j->mc, SUB(j->d_comp2, b->comp2), stream))) return r;
    if ((r = b200_mc_blend_batch(bd, &j->mc, SUB(j->d_blend, b->blend), stream))) return r;
    if ((r = b200_mc_blend_batch(bd, &j->mc, SUB(j->d_blend2, b->blend2), stream))) return r;
#undef SUB
    const void *itx_p[B200_N_RECT_TX_SIZES];
    int32_t itx_n[B200_N_RECT_TX_SIZES];
    for (int t = 0; t < B200_N_RECT_TX_SIZES; t++) {
        itx_p[t] = j->d_itx[t] ? j->d_itx[t] + b->itx[t][0] : nullptr;
        itx_n[t] = j->d_itx[t] ? b->itx[t][1] : 0;
    }
    if ((r = b200_itx_add_frame(bd, itx_p, itx_n, j->d_coef, j->mc.dst, j->itx_stride, j->zero_coefs, stream))) return r;
    if (j->n_intra > 0) {
        if ((r = b200::intra_band(bd, &j->intra, j->d_intra + b->intra[0], b->intra[1], first, (cudaStream_t)stream))) return r;
        // the band's last rows, before its post filters change them: the top edge of the band below (launch + ticket reset)
        if (!b->last && (r = b200::intra_edge_backup(bd, &j->intra, b->y1, b->edge_bottom, (cudaStream_t)stream))) return r;
    }
    }
    if (!do_post) return 0;
    // sweeps: what this band's reconstruction makes final. Deblock: the band's own rows (a row-edge filter at y1 will still
    // change rows >= y1 - 6). CDEF tile rows (32 luma rows, reading 2 more on each side): those ending at or above y1 - 32.
    // Loop restoration tile rows (32 rows inside the 64-row stripes that end at 64 k - 8, reading CDEF output up to 3 rows
    // further inside the stripe and 2 deblocked rows beyond it): luma tile rows ending at or above y1 - 40, a subsampled
    // chroma stripe (one tile) once it ends at or above (y1 - 32) / 2 - 12.
    const cudaStream_t st = (cudaStream_t)stream;
    if (j->run_lf && (r = b200::lf_frame_rows(bd, &j->lf, b->y0 >> 2, b->last ? j->lf.h4 : b->y1 >> 2, st))) return r;
    const int big = 1 << 28;
    if (j->run_cdef && (r = b200::cdef_frame_rows(bd, &j->cdef, b->y0 ? (b->y0 >> 5) - 1 : 0, b->last ? big : (b->y1 >> 5) - 1, st))) return r;
    // (the top stripe is 8 rows shorter and its first tile row spans rows 0 .. 31: it needs CDEF rows up to 34, i.e. the band below)
    const int lr0 = b->y0 > 64 ? 2 * (b->y0 >> 6) - 1 : 0, lr1 = b->last ? big : (b->y1 > 64 ? 2 * (b->y1 >> 6) - 1 : 0);
    if (j->run_lr && (r = b200::lr_frame_rows(bd, &j->lr, lr0, lr1, st))) return r;
    if (b->last && j->run_fg) {
#ifndef B200_EMU
        SideStream *fs = side_stream_for(st, 0);
        if (fs && !fs->join(st)) { b200_set_error("b200_frame_run_band: stream join failed"); return -1; }
#endif
        if ((r = b200_fg_apply(bd, &j->fg, stream))) return r;
    }
    return 0;
}

// ---- cross-GPU exchange primitives -------------------------------------------------------------------------------
#ifndef B200_EMU
namespace {
__global__ void flag_signal_kernel(uint32_t *flag, uint32_t value)
{
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(flag), "r"(value) : "memory");
}
__global__ void flag_wait_kernel(const uint32_t *flag, uint32_t value)
{
    uint32_t v;
    for (;;) {
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if ((int32_t)(v - value) >= 0) break;
        __nanosleep(200);
    }
}
__global__ void flag_signal_rel_kernel(uint32_t *flag, const uint32_t *base, int sub, int shift, int add)
{
    const uint32_t value = ((*(volatile const uint32_t *)base - (uint32_t)sub) << shift) + (uint32_t)add;
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(flag), "r"(value) : "memory");
}
__global__ void flag_wait_rel_kernel(const uint32_t *flag, const uint32_t *base, int sub, int shift, int add)
{
    const uint32_t value = ((*(volatile const uint32_t *)base - (uint32_t)sub) << shift) + (uint32_t)add;
    uint32_t v;
    for (;;) {
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if ((int32_t)(v - value) >= 0) break;
        __nanosleep(200);
    }
}
struct PutArgs { B200PutRange r[3]; B200PutFlag f[2]; int n_ranges, n_flags; uint32_t *counter; };
constexpr int kPutThreads = 256;
__global__ void __launch_bounds__(kPutThreads) put_rows_kernel(const __grid_constant__ PutArgs a)
{
    const int tid = blockIdx.x * kPutThreads + threadIdx.x, nt = gridDim.x * kPutThreads;
    for (int k = 0; k < a.n_ranges; k++) {
        const unsigned char *src = (const unsigned char *)a.r[k].src;
        unsigned char *d0 = (unsigned char *)a.r[k].dst[0], *d1 = (unsigned char *)a.r[k].dst[1];
        const size_t n = a.r[k].bytes;
        // head up to the first 16-byte boundary, 16-byte body, tail (src and dst share their alignment modulo 16)
        size_t head = (16 - ((uintptr_t)src & 15)) & 15;
        if (head > n) head = n;
        const size_t body = (n - head) >> 4;
        for (size_t i = tid; i < head; i += nt) { const unsigned char v = src[i]; if (d0) d0[i] = v; if (d1) d1[i] = v; }
        const uint4 *s4 = (const uint4 *)(src + head);
        uint4 *p0 = d0 ? (uint4 *)(d0 + head) : nullptr, *p1 = d1 ? (uint4 *)(d1 + head) : nullptr;
        for (size_t i = tid; i < body; i += nt) { const uint4 v = s4[i]; if (p0) p0[i] = v; if (p1) p1[i] = v; }
        for (size_t i = head + (body << 4) + tid; i < n; i += nt) { const unsigned char v = src[i]; if (d0) d0[i] = v; if (d1) d1[i] = v; }
    }
    // publish: every thread's stores -> system-scope fence -> CTA barrier -> one count per CTA; the last CTA raises the flags
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned done = atomicAdd(a.counter, 1u) + 1;
        if (done == gridDim.x) {
            *a.counter = 0;                       // ready for the next launch on this stream
            __threadfence_system();
            for (int k = 0; k < a.n_flags; k++) {
                const B200PutFlag &f = a.f[k];
                const uint32_t value = f.base ? ((*(volatile const uint32_t *)f.base - (uint32_t)f.sub) << f.shift) + (uint32_t)f.add : (uint32_t)f.add;
                asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(f.flag), "r"(value) : "memory");
            }
        }
    }
}
// cuStreamWaitValue32 through the runtime's driver entry point (no link-time dependency on libcuda)
typedef int (*WaitValue32Fn)(cudaStream_t, unsigned long long, uint32_t, unsigned);
WaitValue32Fn wait_value_fn()
{
    static WaitValue32Fn fn = [] {
        void *p = nullptr;
        // Default: a polling kernel. cuStreamWaitValue32 parks the stream's whole hardware work queue on the semaphore: any
        // other stream that shares the queue (the copy stream that still has to deliver the rows the peer is waiting for)
        // stops too, which deadlocked two ranks waiting for each other (gop_probe, round 2). A polling kernel only
        // occupies one thread; kernels of other streams keep being dispatched. B200_WAIT_VALUE=1 selects the memory op.
        if (!getenv("B200_WAIT_VALUE")) return (WaitValue32Fn) nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuStreamWaitValue32", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
        cudaGetLastError();
        return (WaitValue32Fn)p;
    }();
    return fn;
}
}
#endif

int b200_ipc_export(void *dev_ptr, uint8_t handle[B200_IPC_HANDLE_BYTES])
{
#ifndef B200_EMU
    static_assert(sizeof(cudaIpcMemHandle_t) == B200_IPC_HANDLE_BYTES, "ipc handle size");
    cudaIpcMemHandle_t h;
    B200_CUDA_OK(cudaIpcGetMemHandle(&h, dev_ptr));
    memcpy(handle, &h, sizeof(h));
    return 0;
#else
    (void)dev_ptr; (void)handle;
    b200_set_error("b200_ipc_export: no peer memory on the host emulator");
    return -1;
#endif
}

void *b200_ipc_open(const uint8_t handle[B200_IPC_HANDLE_BYTES])
{
#ifndef B200_EMU
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    void *p = nullptr;
    const cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { b200_set_error("b200_ipc_open: %s", cudaGetErrorString(e)); return nullptr; }
    return p;
#else
    (void)handle;
    b200_set_error("b200_ipc_open: no peer memory on the host emulator");
    return nullptr;
#endif
}

int b200_ipc_close(void *p)
{
#ifndef B200_EMU
    if (p) B200_CUDA_OK(cudaIpcCloseMemHandle(p));
#else
    (void)p;
#endif
    return 0;
}

int b200_copy_async(void *dst, const void *src, size_t bytes, void *stream)
{
    if (bytes) B200_CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, (cudaStream_t)stream));
    return 0;
}

int b200_put_rows(const B200PutRange *ranges, int n_ranges, const B200PutFlag *flags, int n_flags, uint32_t *counter, void *stream)
{
    if (n_ranges < 0 || n_ranges > 3 || n_flags < 0 || n_flags > 2 || !counter) { b200_set_error("b200_put_rows: bad arguments"); return -2; }
#ifndef B200_EMU
    PutArgs a;
    memset(&a, 0, sizeof(a));
    size_t total = 0;
    for (int k = 0; k < n_ranges; k++) {
        a.r[k] = ranges[k]; total += ranges[k].bytes;
        for (int d = 0; d < 2; d++)
            if (ranges[k].dst[d] && (((uintptr_t)ranges[k].dst[d] ^ (uintptr_t)ranges[k].src) & 15)) { b200_set_error("b200_put_rows: src / dst alignment differs"); return -2; }
    }
    for (int k = 0; k < n_flags; k++) a.f[k] = flags[k];
    a.n_ranges = n_ranges; a.n_flags = n_flags; a.counter = counter;
    // enough CTAs to keep the NVLink stores of one band flowing, few enough to leave the SMs to the reconstruction
    const int grid = (int)(total >> 16) < 1 ? 1 : (int)(total >> 16) > 32 ? 32 : (int)(total >> 16);
    put_rows_kernel<<<grid, kPutThreads, 0, (cudaStream_t)stream>>>(a);
    b200_count_launch();
    B200_CUDA_OK(cudaGetLastError());
#else
    (void)stream; (void)counter;
    for (int k = 0; k < n_ranges; k++)
        for (int d = 0; d < 2; d++)
            if (ranges[k].dst[d]) memcpy(ranges[k].dst[d], ranges[k].src, ranges[k].bytes);
    for (int k = 0; k < n_flags; k++)
        *flags[k].flag = flags[k].base ? ((*flags[k].base - (uint32_t)flags[k].sub) << flags[k].shift) + (uint32_t)flags[k].add : (uint32_t)flags[k].add;
#endif
    return 0;
}

int b200_flag_signal(uint32_t *flag, uint32_t value, void *stream)
{
#ifndef B200_EMU
    flag_signal_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(flag, value);
    b200_count_launch();
    B200_CUDA_OK(cudaGetLastError());
#else
    (void)stream;
    *flag = value;
#endif
    return 0;
}

int b200_flag_wait_geq(const uint32_t *flag, uint32_t value, void *stream)
{
#ifndef B200_EMU
    if (WaitValue32Fn fn = wait_value_fn()) {
        const int rc = fn((cudaStream_t)stream, (unsigned long long)(uintptr_t)flag, value, 1 /* CU_STREAM_WAIT_VALUE_GEQ */);
        if (rc == 0) return 0;
        b200_set_error("b200_flag_wait_geq: cuStreamWaitValue32 -> %d", rc);
        return -1;
    }
    flag_wait_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(flag, value);
    b200_count_launch();
    B200_CUDA_OK(cudaGetLastError());
#else
    (void)stream;
    if ((int32_t)(*flag - value) < 0) { b200_set_error("b200_flag_wait_geq: flag %u < %u (the emulator executes in program order)", *flag, value); return -1; }
#endif
    return 0;
}

int b200_flag_signal_rel(uint32_t *flag, const uint32_t *base, int32_t sub, int32_t shift, int32_t add, void *stream)
{
#ifndef B200_EMU
    flag_signal_rel_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(flag, base, sub, shift, add);
    b200_count_launch();
    B200_CUDA_OK(cudaGetLastError());
#else
    (void)stream;
    *flag = ((*base - (uint32_t)sub) << shift) + (uint32_t)add;
#endif
    return 0;
}

int b200_flag_wait_geq_rel(const uint32_t *flag, const uint32_t *base, int32_t sub, int32_t shift, int32_t add, void *stream)
{
#ifndef B200_EMU
    flag_wait_rel_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(flag, base, sub, shift, add);
    b200_count_launch();
    B200_CUDA_OK(cudaGetLastError());
#else
    (void)stream;
    const uint32_t value = ((*base - (uint32_t)sub) << shift) + (uint32_t)add;
    if ((int32_t)(*flag - value) < 0) { b200_set_error("b200_flag_wait_geq_rel: flag %u < %u (the emulator executes in program order)", *flag, value); return -1; }
#endif
    return 0;
}

int b200_graph_begin(void *stream)
{
#ifndef B200_EMU
    B200_CUDA_OK(cudaStreamBeginCapture((cudaStream_t)stream, cudaStreamCaptureModeRelaxed));
    return 0;
#else
    (void)stream;
    b200_set_error("b200_graph_begin: no graphs on the host emulator");
    return -1;
#endif
}

void *b200_graph_end(void *stream)
{
#ifndef B200_EMU
    cudaGraph_t g = nullptr;
    cudaError_t e = cudaStreamEndCapture((cudaStream_t)stream, &g);
    if (e != cudaSuccess || !g) { b200_set_error("b200_graph_end: cudaStreamEndCapture -> %s", cudaGetErrorString(e)); cudaGetLastError(); return nullptr; }
    cudaGraphExec_t x = nullptr;
    e = cudaGraphInstantiate(&x, g, 0);
    cudaGraphDestroy(g);
    if (e != cudaSuccess) { b200_set_error("b200_graph_end: cudaGraphInstantiate -> %s", cudaGetErrorString(e)); cudaGetLastError(); return nullptr; }
    return (void *)x;
#else
    (void)stream;
    return nullptr;
#endif
}

int b200_graph_launch(void *graph_exec, void *stream)
{
#ifndef B200_EMU
    B200_CUDA_OK(cudaGraphLaunch((cudaGraphExec_t)graph_exec, (cudaStream_t)stream));
    return 0;
#else
    (void)graph_exec; (void)stream;
    return -1;
#endif
}

void b200_graph_destroy(void *graph_exec)
{
#ifndef B200_EMU
    if (graph_exec) cudaGraphExecDestroy((cudaGraphExec_t)graph_exec);
#else
    (void)graph_exec;
#endif
}

void *b200_event_create(void)
{
#ifndef B200_EMU
    cudaEvent_t e = nullptr;
    const cudaError_t r = cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    if (r != cudaSuccess) { b200_set_error("b200_event_create: %s", cudaGetErrorString(r)); return nullptr; }
    return (void *)e;
#else
    return (void *)(uintptr_t)1;
#endif
}
void b200_event_destroy(void *ev)
{
#ifndef B200_EMU
    if (ev) cudaEventDestroy((cudaEvent_t)ev);
#else
    (void)ev;
#endif
}
int b200_event_record(void *ev, void *stream)
{
#ifndef B200_EMU
    B200_CUDA_OK(cudaEventRecord((cudaEvent_t)ev, (cudaStream_t)stream));
#else
    (void)ev; (void)stream;
#endif
    return 0;
}
int b200_stream_wait_event(void *stream, void *ev)
{
#ifndef B200_EMU
    B200_CUDA_OK(cudaStreamWaitEvent((cudaStream_t)stream, (cudaEvent_t)ev, 0));
#else
    (void)ev; (void)stream;
#endif
    return 0;
}

int b200_struct_size(int which)
{
    switch (which) {
    case 0: return sizeof(B200McFrame); case 1: return sizeof(B200McBlock); case 2: return sizeof(B200CompBlock);
    case 3: return sizeof(B200BlendBlock); case 4: return sizeof(B200WarpBlock); case 5: return sizeof(B200ItxBlock);
    case 6: return sizeof(B200LfFrame); case 7: return sizeof(B200CdefFrame); case 8: return sizeof(B200LrFrame);
    case 9: return sizeof(B200FrameJob); case 10: return sizeof(B200Av1Filter); case 11: return sizeof(B200Av1Restoration);
    case 12: return sizeof(B200FgFrame); case 13: return sizeof(B200FilmGrainData);
    case 14: return sizeof(B200IntraTx); case 15: return sizeof(B200IntraFrame); case 16: return sizeof(B200McScaledBlock); case 17: return sizeof(B200CoefBlock); case 18: return sizeof(B200IntraSb); case 19: return sizeof(B200CompFusedBlock); case 20: return sizeof(B200FrameBand); case 21: return sizeof(B200ResizeFrame);
    }
    return -1;
}

int b200_frame_submit_host(const B200FrameJob *job, const B200Xfer *up, int n_up, const B200Xfer *down, int n_down,
                           void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    for (int i = 0; i < n_up; i++)
        if (up[i].bytes) B200_CUDA_OK(cudaMemcpyAsync(up[i].dev, up[i].host, up[i].bytes, cudaMemcpyHostToDevice, st));
    int r = b200_frame_run(job, stream);
    if (r) return r;
    for (int i = 0; i < n_down; i++)
        if (down[i].bytes) B200_CUDA_OK(cudaMemcpyAsync(down[i].host, down[i].dev, down[i].bytes, cudaMemcpyDeviceToHost, st));
    return 0;
}

int b200_frame_submit_host_batch(const B200FrameJob *const *jobs, int n_jobs, const B200Xfer *up, int n_up,
                                 const B200Xfer *down, int n_down, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    for (int i = 0; i < n_up; i++)
        if (up[i].bytes) B200_CUDA_OK(cudaMemcpyAsync(up[i].dev, up[i].host, up[i].bytes, cudaMemcpyHostToDevice, st));
    int r = b200_frame_run_batch(jobs, n_jobs, stream);
    if (r) return r;
    for (int i = 0; i < n_down; i++)
        if (down[i].bytes) B200_CUDA_OK(cudaMemcpyAsync(down[i].host, down[i].dev, down[i].bytes, cudaMemcpyDeviceToHost, st));
    return 0;
}

int b200_frame_wait(void *stream)
{
    B200_CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
    return 0;
}

int b200_frame_run_host(const B200FrameJob *job, const B200Xfer *up, int n_up, const B200Xfer *down, int n_down,
                        void *stream)
{
    int r = b200_frame_submit_host(job, up, n_up, down, n_down, stream);
    return r ? r : b200_frame_wait(stream);
}

}  // extern "C"
