// Intra reconstruction of a whole frame (dav1d_recon_b_intra, reference src/recon_tmpl.c:1176-1555, with
// dav1d_prepare_intra_edges, reference src/ipred_prepare_tmpl.c:75-204, run on the device).
//
// Intra prediction reads the *reconstructed* pixels left of / above the block, so transform blocks form a
// dependency graph (left, top, top-left, and — when the bitstream order made them available — top-right and
// bottom-left neighbours; CFL chroma additionally needs its luma block). The kernel is a dataflow machine:
//   * a persistent grid; each CTA repeatedly takes the next record (atomic ticket). Records are in a
//     topological order, so everything a record waits for has already been taken by a running CTA;
//   * the CTA polls the per-4x4 "done" map of the cells its edge pixels come from, then gathers the edge array
//     into shared memory with L1-bypassing loads (the rules of dav1d_prepare_intra_edges: replication past the
//     tile end, default values without neighbours, Z2 corner smoothing);
//   * predicts (ipred_body.cuh) into a shared-memory tile, adds the inverse transform (itx_body.cuh) there, writes
//     the finished block to the picture with row-contiguous stores, fences, publishes its cells;
//   * the next ticket, the next record and an L2 prefetch of its coefficients are issued while the current block is
//     in flight, so that only [poll -> edge loads -> predict -> transform -> store -> fence] is on the dependency chain.
// Three more record kinds ride on the same machine (frames that mix prediction types, reference src/recon_tmpl.c:1201-1223,
// 1601-1626, 1737-1777): B200_INTRA_MODE_PAL writes a palette block from its 8 colours + packed index map,
// B200_INTRA_MODE_II blends an intra predictor over a whole inter block into the inter prediction that an earlier launch
// left in the picture (inter-intra), and B200_INTRA_MODE_RESID adds a transform block's residual to such a block in place.
// The done map therefore has three states per 4x4 cell: 0 = not written, 2 = predicted (PAL / II with residual records to
// come), 1 = final. Neighbours wait for 1, a RESID record waits for 2 on its own cells. In frames with inter blocks the map
// starts from `done_init` (every cell that no intra record covers is already final when the kernel starts).
// Integer, bit-exact with the reference C path.
#include "ipred_body.cuh"
#include "itx_body.cuh"
#include "launch_count.h"

namespace b200 {

// scratch layout: [header: 256 B][done maps of the three planes, one byte per 4x4 cell]
// The header holds the ticket counter and the band the next launch reconstructs. A band-sliced job (b200_frame_run_band)
// launches the kernel once per band; the edge-backup kernel of band k-1 resets the ticket and points `edge` at the row
// of each plane just above band k, saved before that row was deblocked (dav1d's f->ipred_edge, reference
// src/recon_tmpl.c:2111-2135). Records on the band's first row take their top edge from there. All zero (the state
// b200_intra_frames starts from): no band, every edge comes from the picture.
struct IntraHdr {
    int ticket;
    int band_y;                 // luma row where the band starts (its first chroma row: band_y >> ss_ver)
    const void *edge;           // NULL, or the Y, U and V rows above band_y, each `stride[p]` samples long, back to back
};
struct IntraScratch {
    size_t done_off[3], total;
};
static inline IntraScratch intra_scratch_layout(const B200IntraFrame *f)
{
    IntraScratch L;
    size_t o = 256;
    for (int p = 0; p < 3; p++) { L.done_off[p] = o; o += ((size_t)f->w4[p] * f->h4[p] + 255) & ~(size_t)255; }
    L.total = o;
    return L;
}
// CTAs per launch: a frame's wavefront is a few dozen blocks wide; a modest grid leaves room for other frames'
// kernels (other streams) to run beside this one
constexpr int kIntraGrid = 148;

// what the kernels read of a B200IntraFrame (same member names; keeps 24 frames per launch inside the parameter space)
struct IntraFrameDev {
    void *pic;
    int32_t stride[3];
    int32_t ss_hor, ss_ver;
    int32_t w4[3], h4[3];
    void *d_coef;
    int32_t zero_coefs;
    uint32_t plane_off[3];
    int32_t n_sb, sb_w, sb_h;
    const B200IntraSb *sb;
    const uint8_t *mask, *pal;
};
struct IntraParams {
    IntraFrameDev f;
    const B200IntraTx *tx;
    int n;
    uint8_t *scratch;       // [ticket counter: 256 B][done maps]; superblock mode: one flag per superblock at done_off[0]
    uint32_t done_off[3];
};
// several independent frames per launch (blockIdx.y = frame): frames are the parallel axis of intra decoding and
// one launch is not limited by the number of hardware work queues the way one stream per frame is
constexpr int kIntraMaxBatch = 24;
struct IntraBatch { IntraParams p[kIntraMaxBatch]; };
static_assert(sizeof(IntraBatch) <= 4080, "kernel parameter space (4 KB with the trailing int)");

B200_DEV int ld_cell(const uint8_t *p) { return *(const volatile uint8_t *)p; }
// the row above a block: the picture's, or the saved edge row when the block starts the band (its row above belongs to
// the previous band, whose post filters may already be rewriting it). The header is read only on the first row of a
// 64-luma-row superblock row (bands start there): nothing stays live across the loop.
template <class pixel, class Frame>
B200_DEV const pixel *top_row(const Frame &f, const uint8_t *scratch, const pixel *dst, int pl, int x4, int y4)
{
    const int ssv = pl ? f.ss_ver : 0;
    if (!((y4 * 4) & (63 >> ssv))) {
        const IntraHdr *const hdr = (const IntraHdr *)scratch;
        const void *const edge = hdr->edge;
        if (edge && (y4 * 4) << ssv == hdr->band_y)
            return (const pixel *)edge + (pl ? f.stride[0] + (pl - 1) * f.stride[1] : 0) + x4 * 4;
    }
    return dst - f.stride[pl];
}
// a dependency that never arrives (records not in a topological order) must not hang the GPU: fail the launch
B200_DEV void intra_stuck() {
#ifndef B200_EMU
    __trap();
#else
    abort();
#endif
}

template <bool HBD> B200_DEV int ld_px(const typename Bd<HBD>::pixel *p) {
#ifdef B200_EMU
    return *p;
#else
    return __ldcg(p);          // L2 only: another SM wrote it, this SM's L1 may hold a stale line
#endif
}

B200_DEV void prefetch_l2(const void *p) {
#ifndef B200_EMU
    asm volatile("prefetch.global.L2 [%0];" :: "l"(p));
#else
    (void)p;
#endif
}

// Intra block copy: one sample of mc[FILTER_2D_BILINEAR] (put_bilin_c, reference src/mc_tmpl.c:434-490) read from the picture
// being reconstructed, source coordinates clamped to the plane area like emu_edge (mc(), src/recon_tmpl.c:956-977 with
// w = f->bw * 4 >> ss_hor, h = f->bh * 4 >> ss_ver). L2 loads: other SMs wrote the source.
template <bool HBD, class Frame>
__device__ __forceinline__ int ibc_sample(const Frame &f, const B200IntraTx &r, const int pl, const int xx, const int yy,
                                          const int bitdepth, const int bdmax)
{
    typedef typename Bd<HBD>::pixel pixel;
    const int st = f.stride[pl], pw = f.w4[pl] * 4, ph = f.h4[pl] * 4;
    const int mx = r.cfl_w_pad, my = r.cfl_h_pad;
    const int sx = (int)(r.luma_off & 0xffff) + xx, sy = (int)(r.luma_off >> 16) + yy;
    // the plane starts where this block's row 0 / column 0 is, minus its own position
    const pixel *const plane = (const pixel *)f.pic + r.dst_off - ((ptrdiff_t)r.y4 * 4 * st + r.x4 * 4);
    const int x0 = iclip(sx, 0, pw - 1), x1 = iclip(sx + 1, 0, pw - 1), y0 = iclip(sy, 0, ph - 1), y1 = iclip(sy + 1, 0, ph - 1);
    const int ib = bitdepth == 12 ? 2 : 4;                       // intermediate_bits
    const int a = ld_px<HBD>(plane + (ptrdiff_t)y0 * st + x0);
    if (!mx && !my) return a;
    if (mx && !my) {
        const int b = ld_px<HBD>(plane + (ptrdiff_t)y0 * st + x1);
        const int px = (16 * a + mx * (b - a) + ((1 << (4 - ib)) >> 1)) >> (4 - ib);
        return iclip((px + ((1 << ib) >> 1)) >> ib, 0, bdmax);
    }
    const int c = ld_px<HBD>(plane + (ptrdiff_t)y1 * st + x0);
    if (!mx) return iclip((16 * a + my * (c - a) + 8) >> 4, 0, bdmax);
    const int b = ld_px<HBD>(plane + (ptrdiff_t)y0 * st + x1), d = ld_px<HBD>(plane + (ptrdiff_t)y1 * st + x1);
    const int m0 = (16 * a + mx * (b - a) + ((1 << (4 - ib)) >> 1)) >> (4 - ib);
    const int m1 = (16 * c + mx * (d - c) + ((1 << (4 - ib)) >> 1)) >> (4 - ib);
    return iclip((16 * m0 + my * (m1 - m0) + ((1 << (4 + ib)) >> 1)) >> (4 + ib), 0, bdmax);
}

template <bool HBD>
#ifndef B200_POLL_NS0
#define B200_POLL_NS0 32
#define B200_POLL_NSMAX 256
#endif
#ifndef B200_INTRA_MINB
#define B200_INTRA_MINB 5
#endif
__global__ void __launch_bounds__(kIpT, B200_INTRA_MINB) intra_frame_kernel(const __grid_constant__ IntraBatch B, const int bdmax)
{
    const IntraParams &P = B.p[blockIdx.y];
    typedef typename Bd<HBD>::pixel pixel;
    typedef typename Bd<HBD>::coef coef;
    constexpr int kRecWords = sizeof(B200IntraTx) / 4;
    __shared__ IpShared S;
    __shared__ int s_itx[ItxGeom<64, 64>::NB * ItxGeom<64, 64>::SLOT];
    __shared__ pixel s_px[64 * 64];                 // the block being reconstructed (pitch = its width)
    __shared__ int16_t s_ac[32 * 32];
    __shared__ coef s_cf[32 * 32];                  // this block's coefficients, fetched while waiting
    __shared__ B200ItxBlock s_blk;
    __shared__ int s_ticket, s_next;
    __shared__ uint32_t s_rec[kRecWords];
    const int tid = threadIdx.x;
    const IntraFrameDev &f = P.f;
    const int bitdepth = 32 - __clz(bdmax);
    int *const tl = S.edge + 128;

    if (tid == 0) s_ticket = atomicAdd(((int *)P.scratch), 1);
    __syncthreads();
    if (tid < kRecWords && s_ticket < P.n) s_rec[tid] = ((const uint32_t *)&P.tx[s_ticket])[tid];
    __syncthreads();

    for (;;) {
        const int ti = s_ticket;
        if (ti >= P.n) break;
        B200IntraTx r;
#pragma unroll
        for (int k = 0; k < kRecWords; k++) ((uint32_t *)&r)[k] = s_rec[k];
        int nxt = 0;
        if (tid == 0) nxt = atomicAdd(((int *)P.scratch), 1);          // consumed at the end of this iteration
        const int pl = r.plane, st = f.stride[pl];
        const int tw = c_tx_w4[r.tx], th = c_tx_h4[r.tx];              // 4-sample units
        const int w = tw * 4, h = th * 4;
        const int x = r.x4, y = r.y4, xe = r.xend4, ye = r.yend4;
        const bool have_left = r.flags & B200_INTRA_HAVE_LEFT, have_top = r.flags & B200_INTRA_HAVE_TOP;
        const bool have_tr = have_top && x + tw < xe && (r.flags & B200_INTRA_TOP_HAS_RIGHT);
        const bool have_bl = have_left && y + th < ye && (r.flags & B200_INTRA_LEFT_HAS_BOTTOM);
        const bool is_cfl = r.mode == B200_INTRA_MODE_CFL && r.cfl_alpha != 0;
        const bool is_ii = r.mode == B200_INTRA_MODE_II, is_resid = r.mode == B200_INTRA_MODE_RESID, is_pal = r.mode == B200_INTRA_MODE_PAL;
        const bool is_ibc = r.mode == B200_INTRA_MODE_IBC;
        const uint8_t *const dmap = (P.scratch + P.done_off[pl]);
        const int mw = f.w4[pl];
        // coefficients: loads issued before the wait, parked in shared memory after it (off the dependency chain)
        const int ncf = imin(w, 32) * imin(h, 32);
        coef *const gcf = (coef *)f.d_coef + r.coef_off;
        coef creg[1024 / kIpT];
        if (r.eob >= 0) {
#pragma unroll
            for (int k = 0; k < 1024 / kIpT; k++) { const int i = tid + k * kIpT; creg[k] = i < ncf ? gcf[i] : (coef)0; }
        }

        // ---- wait for the neighbours whose pixels the edge array reads
        {
            // a residual-only record waits for its own cells to be "predicted" (2), everything else for final neighbours (1)
            const bool no_edges = is_resid || is_ibc;
            const int n_left = no_edges ? 0 : have_left ? imin(th, ye - y) + (have_bl ? imin(th, ye - y - th) : 0) : 0;
            const int n_top = no_edges ? 0 : have_top ? imin(tw, xe - x) + (have_tr ? imin(tw, xe - x - tw) : 0) : 0;
            const int n_tl = !no_edges && have_left && have_top;
            // intra block copy: every cell of the source rectangle (one sample more where the bilinear phase is not 0)
            int n_src = 0, sc_x0 = 0, sc_y0 = 0, sc_w = 1;
            if (is_ibc) {
                const int sx = r.luma_off & 0xffff, sy = r.luma_off >> 16;
                sc_x0 = imin(sx >> 2, mw - 1); sc_y0 = imin(sy >> 2, f.h4[pl] - 1);
                sc_w = imin((sx + w - 1 + (r.cfl_w_pad != 0)) >> 2, mw - 1) - sc_x0 + 1;
                n_src = sc_w * (imin((sy + h - 1 + (r.cfl_h_pad != 0)) >> 2, f.h4[pl] - 1) - sc_y0 + 1);
            }
            const int self_w = imin(tw, mw - x), n_self = is_resid ? self_w * imin(th, f.h4[pl] - y) : 0;
            const int want = is_resid ? 2 : 1;
            int n_luma = 0, lw4 = 0, lx4 = 0, ly4 = 0;
            if (is_cfl) {
                lx4 = x << f.ss_hor; ly4 = y << f.ss_ver;
                lw4 = imin((tw - r.cfl_w_pad) << f.ss_hor, f.w4[0] - lx4);
                const int lh4 = imin((th - r.cfl_h_pad) << f.ss_ver, f.h4[0] - ly4);
                n_luma = lw4 * lh4;
            }
            // only warp 0 polls (the other warps park at the barrier and cost no issue slots)
            if (tid < 32) {
                for (int c = tid; c < n_left + n_top + n_tl + n_luma + n_self + n_src; c += 32) {
                    const uint8_t *cell;
                    if (c >= n_left + n_top + n_tl + n_luma + n_self) { const int k = c - n_left - n_top - n_tl - n_luma - n_self; cell = dmap + (sc_y0 + k / sc_w) * mw + sc_x0 + k % sc_w; }
                    else if (c >= n_left + n_top + n_tl + n_luma) { const int k = c - n_left - n_top - n_tl - n_luma; cell = dmap + (y + k / self_w) * mw + x + k % self_w; }
                    else if (c < n_left) cell = dmap + (y + c) * mw + x - 1;
                    else if (c < n_left + n_top) cell = dmap + (y - 1) * mw + x + (c - n_left);
                    else if (c < n_left + n_top + n_tl) cell = dmap + (y - 1) * mw + x - 1;
                    else { const int k = c - n_left - n_top - n_tl; cell = (P.scratch + P.done_off[0]) + (ly4 + k / lw4) * f.w4[0] + lx4 + k % lw4; }
                    unsigned ns = B200_POLL_NS0, spins = 0;
                    while (ld_cell(cell) != want) {
                        __nanosleep(ns); if (ns < B200_POLL_NSMAX) ns += ns >> 1;
                        if (++spins > (1u << 23)) intra_stuck();      // seconds: records are not in a valid order
                    }
                }
                __threadfence();          // acquire side, by the polling warp only (the barrier below publishes it)
            }
            if (tid == 0) s_next = nxt;
            if (r.eob >= 0) {
#pragma unroll
                for (int k = 0; k < 1024 / kIpT; k++) { const int i = tid + k * kIpT; if (i < ncf) s_cf[i] = creg[k]; }
            }
            __syncthreads();
        }

        pixel *const dst = (pixel *)f.pic + r.dst_off;
        // ---- dav1d_prepare_intra_edges: mode conversion (:97-120)
        int mode = r.mode, angle = r.angle;
        if (is_ii) { mode = r.angle; angle = 0; }                              // inter-intra: the predictor is in `angle`
        if (is_resid || is_pal || is_ibc) mode = 0;
        if (mode == B200_INTRA_MODE_CFL) mode = 0;                             // DC_PRED (:1446, :1373)
        if (mode >= 1 && mode <= 8) {                                          // VERT_PRED .. VERT_LEFT_PRED
            const int base = mode == 1 ? 90 : mode == 2 ? 180 : mode == 3 ? 45 : mode == 4 ? 135 : mode == 5 ? 113
                           : mode == 6 ? 157 : mode == 7 ? 203 : 67;
            angle = base + 3 * angle;
            if (angle <= 90) mode = angle < 90 && have_top ? B200_Z1_PRED : B200_VERT_PRED;
            else if (angle < 180) mode = B200_Z2_PRED;
            else mode = angle > 180 && have_left ? B200_Z3_PRED : B200_HOR_PRED;
        } else if (mode == 0) {
            mode = have_left ? (have_top ? B200_DC_PRED : B200_LEFT_DC_PRED) : (have_top ? B200_TOP_DC_PRED : B200_DC_128_PRED);
        } else if (mode == 12) {
            mode = have_left ? (have_top ? B200_PAETH_PRED : B200_HOR_PRED) : (have_top ? B200_VERT_PRED : B200_DC_128_PRED);
        }
        // ---- edge gather (every part is filled; the predictors read only what the reference fills)
        {
            const pixel *const top = top_row(f, P.scratch, dst, pl, x, y);
            const int half = (1 << bitdepth) >> 1;
            const int lpx = imin(h, (ye - y) << 2), lpx2 = imin(h, (ye - y - th) << 2);
            const int tpx = imin(w, (xe - x) << 2), tpx2 = imin(w, (xe - x - tw) << 2);
            const int left_fill = have_top ? ld_px<HBD>(top) : half + 1;
            const int top_fill = have_left ? ld_px<HBD>(dst - 1) : half - 1;
            for (int i = tid; i < 2 * h; i += kIpT) {                           // tl[-(1+i)]: left, then bottom-left
                int v;
                if (i < h) v = have_left ? ld_px<HBD>(dst + (ptrdiff_t)imin(i, lpx - 1) * st - 1) : left_fill;
                else if (have_bl) v = ld_px<HBD>(dst + (ptrdiff_t)(h + imin(i - h, lpx2 - 1)) * st - 1);
                else v = have_left ? ld_px<HBD>(dst + (ptrdiff_t)(lpx - 1) * st - 1) : left_fill;
                tl[-(1 + i)] = v;
            }
            for (int i = tid; i < 2 * w; i += kIpT) {                           // tl[1+i]: top, then top-right
                int v;
                if (i < w) v = have_top ? ld_px<HBD>(top + imin(i, tpx - 1)) : top_fill;
                else if (have_tr) v = ld_px<HBD>(top + w + imin(i - w, tpx2 - 1));
                else v = have_top ? ld_px<HBD>(top + tpx - 1) : top_fill;
                tl[1 + i] = v;
            }
            if (tid == 0)
                tl[0] = have_left ? (have_top ? ld_px<HBD>(top - 1) : ld_px<HBD>(dst - 1)) : (have_top ? ld_px<HBD>(top) : half);
            // CFL: the (sub-sampled, padded) luma block -> s_ac (mean removed below)
            int part = 0;
            if (is_cfl) {
                const pixel *ypx = (const pixel *)f.pic + r.luma_off;
                const int ssh = f.ss_hor, ssv = f.ss_ver, ys = f.stride[0];
                for (int i = tid; i < w * h; i += kIpT) {
                    const int yy = i / w, xx = i - yy * w;
                    const int sy = imin(yy, h - 4 * r.cfl_h_pad - 1), sx = imin(xx, w - 4 * r.cfl_w_pad - 1);
                    const pixel *p = ypx + (ptrdiff_t)(sy << ssv) * ys + (sx << ssh);
                    int sacc = ld_px<HBD>(p);
                    if (ssh) sacc += ld_px<HBD>(p + 1);
                    if (ssv) { sacc += ld_px<HBD>(p + ys); if (ssh) sacc += ld_px<HBD>(p + ys + 1); }
                    sacc <<= 1 + !ssv + !ssh;
                    s_ac[i] = (int16_t)sacc;
                    part += sacc;
                }
                S.tile[tid] = part;
            }
            __syncthreads();
            if (tid == 0 && mode == B200_Z2_PRED && tw + th >= 6 && (r.angle_flags & 1024))
                tl[0] = ((tl[-1] + tl[1]) * 5 + tl[0] * 6 + 8) >> 4;
            if (is_cfl && tid == 0) {
                const int log2sz = (__ffs(w) - 1) + (__ffs(h) - 1);
                int sum = (1 << log2sz) >> 1;
                for (int i = 0; i < kIpT; i++) sum += S.tile[i];
                S.dc = sum >> log2sz;
            }
            __syncthreads();
        }
        // the next record (its ticket has arrived by now): loads issued here, consumed at the end of the iteration
        uint32_t next_word = 0;
        const int nti = s_next;
        if (tid < kRecWords && nti < P.n) next_word = ((const uint32_t *)&P.tx[nti])[tid];

        // ---- predict into the shared tile
        if (is_resid) {
            // residual only: the tile is what the inter-intra record of this block left in the picture (another SM wrote it)
            for (int i = tid; i < w * h; i += kIpT) { const int yy = i / w, xx = i - yy * w; s_px[i] = (pixel)ld_px<HBD>(dst + (ptrdiff_t)yy * st + xx); }
        } else if (is_pal) {
            // palette: 8 colours, then the index map (two 4-bit indices per byte, low nibble first)
            const pixel *const colours = (const pixel *)(f.pal + r.luma_off);
            const uint8_t *const idx = f.pal + r.luma_off + 8 * sizeof(pixel);
            for (int i = tid; i < w * h; i += kIpT) s_px[i] = colours[(idx[i >> 1] >> ((i & 1) * 4)) & 7];
        } else if (is_ibc) {
            for (int i = tid; i < w * h; i += kIpT) s_px[i] = (pixel)ibc_sample<HBD>(f, r, pl, i % w, i / w, bitdepth, bdmax);
        } else if (is_cfl) {
            const int dc = S.dc;
            for (int i = tid; i < w * h; i += kIpT) s_ac[i] = (int16_t)(s_ac[i] - dc);
            __syncthreads();
            ipred_cfl_pred_body<HBD>(S, s_px, w, w, h, mode, r.cfl_alpha, s_ac, bdmax);
        } else {
            const int a = (mode == B200_FILTER_PRED ? r.angle : angle) | r.angle_flags;
            ipred_pred_body<HBD>(S, s_px, w, w, h, mode, a, r.max_w, r.max_h, bdmax);
        }
        __syncthreads();
        if (is_ii) {
            // inter-intra: blend the intra prediction into the inter prediction already in the picture (earlier launch),
            // dst = (inter * (64 - m) + intra * m + 32) >> 6 (dsp->mc.blend, reference src/mc_tmpl.c:683-694)
            const uint8_t *const msk = f.mask + r.luma_off;
            for (int i = tid; i < w * h; i += kIpT) {
                const int yy = i / w, xx = i - yy * w, m = msk[i];
                s_px[i] = (pixel)(((int)dst[(ptrdiff_t)yy * st + xx] * (64 - m) + (int)s_px[i] * m + 32) >> 6);
            }
            __syncthreads();
        }

        // ---- residual, added in the shared tile
        if (r.eob >= 0) {
            if (tid == 0) { s_blk.dst_off = 0; s_blk.coef_off = 0; s_blk.eob = r.eob; s_blk.txtp = r.txtp; s_blk.plane = 0; }
            __syncthreads();
            switch (r.tx) {
#define X(TX, W, H, SH) case TX: itx_add_body<W, H, TX, SH, HBD, true>(0, s_itx, &s_blk, 1, s_cf, s_px, W, W, W, bdmax, 0); break;
            B200_ITX_SIZES(X)
#undef X
            }
            __syncthreads();
            if (f.zero_coefs)
                for (int i = tid; i < ncf; i += kIpT) gcf[i] = 0;
        }
        // ---- write the block, publish
        for (int i = tid; i < w * h; i += kIpT) {
            const int yy = i / w, xx = i - yy * w;
            dst[(ptrdiff_t)yy * st + xx] = s_px[i];
        }
        // one device-scope fence per block: the barrier orders every thread's stores before thread 0's fence (causality
        // through bar.sync, fences are cumulative), the warp barrier orders the fence before the flag stores of warp 0
        __syncthreads();
        if (tid < 32) {
            if (tid == 0) __threadfence();
            __syncwarp();
            uint8_t *const dm = (P.scratch + P.done_off[pl]);
            const int cw = imin(tw, mw - x), chh = imin(th, f.h4[pl] - y);
            const uint8_t state = (is_ii || is_pal || is_ibc) && r.cfl_alpha ? 2 : 1;   // 2: predicted, the block's residual records follow
            for (int c = tid; c < cw * chh; c += 32) *(volatile uint8_t *)(dm + (y + c / cw) * mw + x + c % cw) = state;
        }
        // ---- hand over to the next record
        if (tid < kRecWords) s_rec[tid] = next_word;
        if (tid == 0) s_ticket = nti;
        if (tid == 1 && nti < P.n) {                     // word 1 of the record = coef_off: warm L2 with its coefficients
            const char *cf = (const char *)((const coef *)f.d_coef + next_word);
            for (int k = 0; k < 8; k++) prefetch_l2(cf + k * 256);
        }
        __syncthreads();
    }
}


// ---- warp-per-block dataflow (round 2) -----------------------------------------------------------------------
// The same machine with a WARP as the unit instead of a CTA: every warp of the persistent grid takes tickets on its own,
// polls the done map, gathers its edges, predicts, transforms and publishes without a single CTA barrier. ncu on the
// CTA-per-block kernel (profiles/r01_intra_sb_v5.md) showed half of all stall samples in bar.sync — one warp ran the
// transform while three waited — and instruction-cache misses from 48 K inlined instructions. Here the independent
// blocks of a wavefront run side by side inside a CTA (4 warps = 4 blocks), only __syncwarp separates the phases of a
// block, and the 1-D transforms are out-of-line (one copy per length, shared by the row and the column pass and by all
// block shapes). The flags are written after a device-scope fence and read with volatile loads + fence, pixels of
// neighbours are read through L2 (ld.cg): the same publication protocol as before.
constexpr int kIwWarps = 4;
template <bool HBD> struct IwShared {
    typedef typename Bd<HBD>::pixel pixel;
    typedef typename Bd<HBD>::coef coef;
    IpShared S;                       // edge array, scratch of the directional / filter predictors
    union {                           // first the transform tile (ItxGeom: SH rows of pitch W + 1, at most 32 x 65) while the residual
        int itx[32 * 65];             // is computed, then (the residual sits in `resid`) the prediction of the block (pitch = its width)
        pixel px[64 * 64];
    } u;
    int16_t resid[64 * 64];           // the block's residual, transformed while the warp still waits for its neighbours
    coef cf[32 * 32];
    int16_t ac[32 * 32];
};

template <bool HBD>
__global__ void __launch_bounds__(kIwWarps * 32) intra_warp_kernel(const __grid_constant__ IntraBatch B, const int bdmax)
{
    const IntraParams &P = B.p[blockIdx.y];
    typedef typename Bd<HBD>::pixel pixel;
    typedef typename Bd<HBD>::coef coef;
    typedef IpWarp G;
#ifdef B200_EMU
    IwShared<HBD> *const all = (IwShared<HBD> *)B200_EMU_DYN_SMEM;
#else
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    IwShared<HBD> *const all = (IwShared<HBD> *)dyn_smem;
#endif
    IwShared<HBD> &W = all[threadIdx.x >> 5];
    IpShared &S = W.S;
    pixel *const s_px = W.u.px;
    int16_t *const s_ac = W.ac;
    coef *const s_cf = W.cf;
    const int lane = threadIdx.x & 31;
    const IntraFrameDev &f = P.f;
    const int bitdepth = 32 - __clz(bdmax);
    int *const tl = S.edge + 128;

    for (;;) {
        int ti = 0;
        if (lane == 0) ti = atomicAdd(((int *)P.scratch), 1);
        ti = __shfl_sync(0xffffffffu, ti, 0);
        if (ti >= P.n) break;
        const B200IntraTx r = P.tx[ti];
        const int pl = r.plane, st = f.stride[pl];
        const int tw = c_tx_w4[r.tx], th = c_tx_h4[r.tx];              // 4-sample units
        const int w = tw * 4, h = th * 4;
        const int x = r.x4, y = r.y4, xe = r.xend4, ye = r.yend4;
        const bool have_left = r.flags & B200_INTRA_HAVE_LEFT, have_top = r.flags & B200_INTRA_HAVE_TOP;
        const bool have_tr = have_top && x + tw < xe && (r.flags & B200_INTRA_TOP_HAS_RIGHT);
        const bool have_bl = have_left && y + th < ye && (r.flags & B200_INTRA_LEFT_HAS_BOTTOM);
        const bool is_cfl = r.mode == B200_INTRA_MODE_CFL && r.cfl_alpha != 0;
        const bool is_ii = r.mode == B200_INTRA_MODE_II, is_resid = r.mode == B200_INTRA_MODE_RESID, is_pal = r.mode == B200_INTRA_MODE_PAL;
        const bool is_ibc = r.mode == B200_INTRA_MODE_IBC;
        uint8_t *const dmap = (P.scratch + P.done_off[pl]);
        const int mw = f.w4[pl];
        const int ncf = imin(w, 32) * imin(h, 32);
        coef *const gcf = (coef *)f.d_coef + r.coef_off;
        // The residual does not depend on the neighbours: inverse transform NOW, into an int16 tile, off the dependency chain
        // (the chain of a frame is ~1000 blocks deep; what stays on it is poll -> edge loads -> predict -> add -> store -> publish)
        if (r.eob >= 0) {
            for (int i = lane; i < ncf; i += 32) s_cf[i] = gcf[i];
            __syncwarp();
            switch (r.tx) {
#define X(TX, TW, TH, SH) case TX: itx_add_warp<TW, TH, TX, SH, HBD>(W.u.itx, s_cf, (pixel *)nullptr, TW, r.eob, r.txtp, bdmax, W.resid); break;
            B200_ITX_SIZES(X)
#undef X
            }
            if (f.zero_coefs)
                for (int i = lane; i < ncf; i += 32) gcf[i] = 0;
            __syncwarp();
        }

        // ---- wait for the neighbours whose pixels the edge array reads
        {
            const bool no_edges = is_resid || is_ibc;
            const int n_left = no_edges ? 0 : have_left ? imin(th, ye - y) + (have_bl ? imin(th, ye - y - th) : 0) : 0;
            const int n_top = no_edges ? 0 : have_top ? imin(tw, xe - x) + (have_tr ? imin(tw, xe - x - tw) : 0) : 0;
            const int n_tl = !no_edges && have_left && have_top;
            // intra block copy: every cell of the source rectangle (one sample more where the bilinear phase is not 0)
            int n_src = 0, sc_x0 = 0, sc_y0 = 0, sc_w = 1;
            if (is_ibc) {
                const int sx = r.luma_off & 0xffff, sy = r.luma_off >> 16;
                sc_x0 = imin(sx >> 2, mw - 1); sc_y0 = imin(sy >> 2, f.h4[pl] - 1);
                sc_w = imin((sx + w - 1 + (r.cfl_w_pad != 0)) >> 2, mw - 1) - sc_x0 + 1;
                n_src = sc_w * (imin((sy + h - 1 + (r.cfl_h_pad != 0)) >> 2, f.h4[pl] - 1) - sc_y0 + 1);
            }
            const int self_w = imin(tw, mw - x), n_self = is_resid ? self_w * imin(th, f.h4[pl] - y) : 0;
            const int want = is_resid ? 2 : 1;       // a residual-only record waits for its own cells to be "predicted" (2)
            int n_luma = 0, lw4 = 0, lx4 = 0, ly4 = 0;
            if (is_cfl) {
                lx4 = x << f.ss_hor; ly4 = y << f.ss_ver;
                lw4 = imin((tw - r.cfl_w_pad) << f.ss_hor, f.w4[0] - lx4);
                const int lh4 = imin((th - r.cfl_h_pad) << f.ss_ver, f.h4[0] - ly4);
                n_luma = lw4 * lh4;
            }
            for (int c = lane; c < n_left + n_top + n_tl + n_luma + n_self + n_src; c += 32) {
                const uint8_t *cell;
                if (c >= n_left + n_top + n_tl + n_luma + n_self) { const int k = c - n_left - n_top - n_tl - n_luma - n_self; cell = dmap + (sc_y0 + k / sc_w) * mw + sc_x0 + k % sc_w; }
                else if (c >= n_left + n_top + n_tl + n_luma) { const int k = c - n_left - n_top - n_tl - n_luma; cell = dmap + (y + k / self_w) * mw + x + k % self_w; }
                else if (c < n_left) cell = dmap + (y + c) * mw + x - 1;
                else if (c < n_left + n_top) cell = dmap + (y - 1) * mw + x + (c - n_left);
                else if (c < n_left + n_top + n_tl) cell = dmap + (y - 1) * mw + x - 1;
                else { const int k = c - n_left - n_top - n_tl; cell = (P.scratch + P.done_off[0]) + (ly4 + k / lw4) * f.w4[0] + lx4 + k % lw4; }
                unsigned ns = B200_POLL_NS0, spins = 0;
                while (ld_cell(cell) != want) {
                    __nanosleep(ns); if (ns < B200_POLL_NSMAX) ns += ns >> 1;
                    if (++spins > (1u << 23)) intra_stuck();      // seconds: records are not in a valid order
                }
            }
            __threadfence();              // acquire side
            __syncwarp();
        }

        pixel *const dst = (pixel *)f.pic + r.dst_off;
        // ---- dav1d_prepare_intra_edges: mode conversion (:97-120)
        int mode = r.mode, angle = r.angle;
        if (is_ii) { mode = r.angle; angle = 0; }                              // inter-intra: the predictor is in `angle`
        if (is_resid || is_pal || is_ibc) mode = 0;
        if (mode == B200_INTRA_MODE_CFL) mode = 0;                             // DC_PRED (:1446, :1373)
        if (mode >= 1 && mode <= 8) {                                          // VERT_PRED .. VERT_LEFT_PRED
            const int base = mode == 1 ? 90 : mode == 2 ? 180 : mode == 3 ? 45 : mode == 4 ? 135 : mode == 5 ? 113
                           : mode == 6 ? 157 : mode == 7 ? 203 : 67;
            angle = base + 3 * angle;
            if (angle <= 90) mode = angle < 90 && have_top ? B200_Z1_PRED : B200_VERT_PRED;
            else if (angle < 180) mode = B200_Z2_PRED;
            else mode = angle > 180 && have_left ? B200_Z3_PRED : B200_HOR_PRED;
        } else if (mode == 0) {
            mode = have_left ? (have_top ? B200_DC_PRED : B200_LEFT_DC_PRED) : (have_top ? B200_TOP_DC_PRED : B200_DC_128_PRED);
        } else if (mode == 12) {
            mode = have_left ? (have_top ? B200_PAETH_PRED : B200_HOR_PRED) : (have_top ? B200_VERT_PRED : B200_DC_128_PRED);
        }
        // ---- edge gather (every part is filled; the predictors read only what the reference fills)
        if (!is_resid && !is_pal && !is_ibc) {
            const pixel *const top = top_row(f, P.scratch, dst, pl, x, y);
            const int half = (1 << bitdepth) >> 1;
            const int lpx = imin(h, (ye - y) << 2), lpx2 = imin(h, (ye - y - th) << 2);
            const int tpx = imin(w, (xe - x) << 2), tpx2 = imin(w, (xe - x - tw) << 2);
            const int left_fill = have_top ? ld_px<HBD>(top) : half + 1;
            const int top_fill = have_left ? ld_px<HBD>(dst - 1) : half - 1;
            for (int i = lane; i < 2 * h; i += 32) {                            // tl[-(1+i)]: left, then bottom-left
                int v;
                if (i < h) v = have_left ? ld_px<HBD>(dst + (ptrdiff_t)imin(i, lpx - 1) * st - 1) : left_fill;
                else if (have_bl) v = ld_px<HBD>(dst + (ptrdiff_t)(h + imin(i - h, lpx2 - 1)) * st - 1);
                else v = have_left ? ld_px<HBD>(dst + (ptrdiff_t)(lpx - 1) * st - 1) : left_fill;
                tl[-(1 + i)] = v;
            }
            for (int i = lane; i < 2 * w; i += 32) {                            // tl[1+i]: top, then top-right
                int v;
                if (i < w) v = have_top ? ld_px<HBD>(top + imin(i, tpx - 1)) : top_fill;
                else if (have_tr) v = ld_px<HBD>(top + w + imin(i - w, tpx2 - 1));
                else v = have_top ? ld_px<HBD>(top + tpx - 1) : top_fill;
                tl[1 + i] = v;
            }
            if (lane == 0)
                tl[0] = have_left ? (have_top ? ld_px<HBD>(top - 1) : ld_px<HBD>(dst - 1)) : (have_top ? ld_px<HBD>(top) : half);
            // CFL: the (sub-sampled, padded) luma block -> s_ac, mean removed
            if (is_cfl) {
                const pixel *ypx = (const pixel *)f.pic + r.luma_off;
                const int ssh = f.ss_hor, ssv = f.ss_ver, ys = f.stride[0];
                int part = 0;
                for (int i = lane; i < w * h; i += 32) {
                    const int yy = i / w, xx = i - yy * w;
                    const int sy = imin(yy, h - 4 * r.cfl_h_pad - 1), sx = imin(xx, w - 4 * r.cfl_w_pad - 1);
                    const pixel *p = ypx + (ptrdiff_t)(sy << ssv) * ys + (sx << ssh);
                    int sacc = ld_px<HBD>(p);
                    if (ssh) sacc += ld_px<HBD>(p + 1);
                    if (ssv) { sacc += ld_px<HBD>(p + ys); if (ssh) sacc += ld_px<HBD>(p + ys + 1); }
                    sacc <<= 1 + !ssv + !ssh;
                    s_ac[i] = (int16_t)sacc;
                    part += sacc;
                }
#pragma unroll
                for (int o = 16; o; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
                const int log2sz = (__ffs(w) - 1) + (__ffs(h) - 1);
                const int dc = (part + ((1 << log2sz) >> 1)) >> log2sz;
                __syncwarp();
                for (int i = lane; i < w * h; i += 32) s_ac[i] = (int16_t)(s_ac[i] - dc);
            }
            __syncwarp();
            if (lane == 0 && mode == B200_Z2_PRED && tw + th >= 6 && (r.angle_flags & 1024))
                tl[0] = ((tl[-1] + tl[1]) * 5 + tl[0] * 6 + 8) >> 4;
            __syncwarp();
        }

        // ---- predict into the shared tile
        if (is_resid) {
            // residual only: the tile is what the inter-intra record of this block left in the picture (another SM wrote it)
            for (int i = lane; i < w * h; i += 32) { const int yy = i / w, xx = i - yy * w; s_px[i] = (pixel)ld_px<HBD>(dst + (ptrdiff_t)yy * st + xx); }
        } else if (is_pal) {
            // palette: 8 colours, then the index map (two 4-bit indices per byte, low nibble first)
            const pixel *const colours = (const pixel *)(f.pal + r.luma_off);
            const uint8_t *const idx = f.pal + r.luma_off + 8 * sizeof(pixel);
            for (int i = lane; i < w * h; i += 32) s_px[i] = colours[(idx[i >> 1] >> ((i & 1) * 4)) & 7];
        } else if (is_ibc) {
            for (int i = lane; i < w * h; i += 32) s_px[i] = (pixel)ibc_sample<HBD>(f, r, pl, i % w, i / w, bitdepth, bdmax);
        } else if (is_cfl) {
            ipred_cfl_pred_body<HBD, G>(S, s_px, w, w, h, mode, r.cfl_alpha, s_ac, bdmax);
        } else {
            const int a = (mode == B200_FILTER_PRED ? r.angle : angle) | r.angle_flags;
            ipred_pred_body<HBD, G>(S, s_px, w, w, h, mode, a, r.max_w, r.max_h, bdmax);
        }
        __syncwarp();
        if (is_ii) {
            // inter-intra: blend the intra prediction into the inter prediction already in the picture (earlier launch),
            // dst = (inter * (64 - m) + intra * m + 32) >> 6 (dsp->mc.blend, reference src/mc_tmpl.c:683-694)
            const uint8_t *const msk = f.mask + r.luma_off;
            for (int i = lane; i < w * h; i += 32) {
                const int yy = i / w, xx = i - yy * w, m = msk[i];
                s_px[i] = (pixel)(((int)dst[(ptrdiff_t)yy * st + xx] * (64 - m) + (int)s_px[i] * m + 32) >> 6);
            }
            __syncwarp();
        }

        // ---- prediction + residual -> picture, publish
        if (r.eob >= 0) {
            for (int i = lane; i < w * h; i += 32) {
                const int yy = i / w, xx = i - yy * w;
                dst[(ptrdiff_t)yy * st + xx] = (pixel)iclip((int)s_px[i] + W.resid[i], 0, bdmax);
            }
        } else {
            for (int i = lane; i < w * h; i += 32) {
                const int yy = i / w, xx = i - yy * w;
                dst[(ptrdiff_t)yy * st + xx] = s_px[i];
            }
        }
        __syncwarp();
        {
            const int cw = imin(tw, mw - x), chh = imin(th, f.h4[pl] - y);
            const uint8_t state = (is_ii || is_pal || is_ibc) && r.cfl_alpha ? 2 : 1;   // 2: predicted, the block's residual records follow
            if (lane < cw * chh || lane == 0) __threadfence();                  // the warp barrier above ordered every lane's stores before it
            for (int c = lane; c < cw * chh; c += 32) *(volatile uint8_t *)(dmap + (y + c / cw) * mw + x + c % cw) = state;
        }
        __syncwarp();
    }
}

// ---- superblock-granular variant -------------------------------------------------------------------------
// A CTA takes a whole 64x64 superblock (ticket order = wavefront order of superblocks) and reconstructs its
// transform blocks one after the other in decode order on a shared-memory canvas (superblock + the row above,
// reaching 64 samples into the top-right superblock, + the column to the left). Dependencies inside the
// superblock therefore cost a barrier instead of a global-memory flag round trip; only the four neighbouring
// superblocks (left, top-left, top, top-right) are waited for through global flags, and the picture is read /
// written once per superblock. The next record and its coefficients are fetched while the current block runs.
template <bool HBD>
#ifndef B200_INTRA_SB_MINB
#define B200_INTRA_SB_MINB 3
#endif
__global__ void __launch_bounds__(kIpT, B200_INTRA_SB_MINB) intra_sb_kernel(const __grid_constant__ IntraBatch B, const int bdmax)
{
    typedef typename Bd<HBD>::pixel pixel;
    typedef typename Bd<HBD>::coef coef;
    constexpr int kRecWords = sizeof(B200IntraTx) / 4;
    const IntraParams &P = B.p[blockIdx.y];
    __shared__ IpShared S;
    __shared__ int s_itx[ItxGeom<64, 64>::NB * ItxGeom<64, 64>::SLOT];
    __shared__ int16_t s_ac[32 * 32];
    __shared__ coef s_cf[32 * 32];
    __shared__ B200ItxBlock s_blk;
    __shared__ int s_ticket;
    __shared__ uint32_t s_rec[kRecWords];
#ifdef B200_EMU
    pixel *const canvas = (pixel *)B200_EMU_DYN_SMEM;
#else
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    pixel *const canvas = (pixel *)dyn_smem;
#endif
    const int tid = threadIdx.x;
    const IntraFrameDev &f = P.f;
    const int bitdepth = 32 - __clz(bdmax);
    int *const tl = S.edge + 128;
    // canvas geometry per plane: pitch cs, origin of the superblock's top-left sample at co + cs + 1
    int cs[3], co[3], sbw[3], sbh[3];
    {
        int o = 0;
        for (int p = 0; p < 3; p++) {
            sbw[p] = 64 >> (p ? f.ss_hor : 0); sbh[p] = 64 >> (p ? f.ss_ver : 0);
            cs[p] = 2 * sbw[p] + 2;                       // left column + 2 superblock widths (+1 pad: even pitch)
            co[p] = o; o += cs[p] * (sbh[p] + 1);
        }
    }

    for (;;) {
        __syncthreads();
        if (tid == 0) s_ticket = atomicAdd(((int *)P.scratch), 1);
        __syncthreads();
        const int si = s_ticket;
        if (si >= f.n_sb) break;
        const B200IntraSb sb = f.sb[si];
        const int sx = sb.sx, sy = sb.sy;
        // first record + its coefficients (exposed once per superblock)
        if (tid < kRecWords && sb.count) s_rec[tid] = ((const uint32_t *)&P.tx[sb.first])[tid];
        // ---- wait for the neighbouring superblocks, then load the halos
        if (tid < 4) {
            const int dx = tid == 3 ? 1 : tid == 2 ? 0 : -1, dy = tid == 0 ? 0 : -1;   // left, top-left, top, top-right
            const int nx = sx + dx, ny = sy + dy;
            if (nx >= 0 && nx < f.sb_w && ny >= 0) {
                const uint8_t *cell = (P.scratch + P.done_off[0]) + ny * f.sb_w + nx;
                unsigned ns = 64, spins = 0;
                while (!ld_cell(cell)) {
                    __nanosleep(ns); if (ns < 1024) ns += ns >> 1;
                    if (++spins > (1u << 22)) intra_stuck();
                }
            }
            __threadfence();
        }
        __syncthreads();
        for (int p = 0; p < 3; p++) {
            const pixel *pic = (const pixel *)f.pic + f.plane_off[p];
            const int st = f.stride[p], pw = f.w4[p] * 4;
            const int X0 = sx * sbw[p], Y0 = sy * sbh[p];
            pixel *cv = canvas + co[p];
            if (sy > 0)      // row above: x = X0-1 .. X0 + 2*sbw - 1, limited to the plane
                for (int i = tid; i < 2 * sbw[p] + 1; i += kIpT) {
                    const int x = X0 - 1 + i;
                    if (x >= 0 && x < pw) cv[i] = (pixel)ld_px<HBD>(pic + (ptrdiff_t)(Y0 - 1) * st + x);
                }
            if (sx > 0)      // column to the left
                for (int i = tid; i < sbh[p]; i += kIpT)
                    if (Y0 + i < f.h4[p] * 4) cv[(1 + i) * cs[p]] = (pixel)ld_px<HBD>(pic + (ptrdiff_t)(Y0 + i) * st + X0 - 1);
        }
        __syncthreads();

        // ---- the superblock's transform blocks, in decode order
        for (unsigned ri = 0; ri < sb.count; ri++) {
            B200IntraTx r;
#pragma unroll
            for (int k = 0; k < kRecWords; k++) ((uint32_t *)&r)[k] = s_rec[k];
            const int pl = r.plane;
            const int tw = c_tx_w4[r.tx], th = c_tx_h4[r.tx];
            const int w = tw * 4, h = th * 4;
            const int x = r.x4, y = r.y4, xe = r.xend4, ye = r.yend4;
            const bool have_left = r.flags & B200_INTRA_HAVE_LEFT, have_top = r.flags & B200_INTRA_HAVE_TOP;
            const bool have_tr = have_top && x + tw < xe && (r.flags & B200_INTRA_TOP_HAS_RIGHT);
            const bool have_bl = have_left && y + th < ye && (r.flags & B200_INTRA_LEFT_HAS_BOTTOM);
            const bool is_cfl = r.mode == B200_INTRA_MODE_CFL && r.cfl_alpha != 0;
            const int ncf = imin(w, 32) * imin(h, 32);
            coef *const gcf = (coef *)f.d_coef + r.coef_off;
            // this block's coefficients -> shared memory (for ri > 0 they were prefetched to L2 one block ago)
            if (r.eob >= 0)
                for (int i = tid; i < ncf; i += kIpT) s_cf[i] = gcf[i];
            // next record: load issued now, parked at the end of the iteration
            uint32_t next_word = 0;
            if (tid < kRecWords && ri + 1 < sb.count) next_word = ((const uint32_t *)&P.tx[sb.first + ri + 1])[tid];
            const int st = cs[pl];
            pixel *const dst = canvas + co[pl] + (1 + (y * 4 - sy * sbh[pl])) * st + 1 + (x * 4 - sx * sbw[pl]);

            int mode = r.mode, angle = r.angle;
            if (mode == B200_INTRA_MODE_CFL) mode = 0;
            if (mode >= 1 && mode <= 8) {
                const int base = mode == 1 ? 90 : mode == 2 ? 180 : mode == 3 ? 45 : mode == 4 ? 135 : mode == 5 ? 113
                               : mode == 6 ? 157 : mode == 7 ? 203 : 67;
                angle = base + 3 * angle;
                if (angle <= 90) mode = angle < 90 && have_top ? B200_Z1_PRED : B200_VERT_PRED;
                else if (angle < 180) mode = B200_Z2_PRED;
                else mode = angle > 180 && have_left ? B200_Z3_PRED : B200_HOR_PRED;
            } else if (mode == 0) {
                mode = have_left ? (have_top ? B200_DC_PRED : B200_LEFT_DC_PRED) : (have_top ? B200_TOP_DC_PRED : B200_DC_128_PRED);
            } else if (mode == 12) {
                mode = have_left ? (have_top ? B200_PAETH_PRED : B200_HOR_PRED) : (have_top ? B200_VERT_PRED : B200_DC_128_PRED);
            }
            {   // edge gather from the canvas (same rules as the global-memory kernel above)
                const pixel *const top = dst - st;
                const int half = (1 << bitdepth) >> 1;
                const int lpx = imin(h, (ye - y) << 2), lpx2 = imin(h, (ye - y - th) << 2);
                const int tpx = imin(w, (xe - x) << 2), tpx2 = imin(w, (xe - x - tw) << 2);
                const int left_fill = have_top ? (int)top[0] : half + 1;
                const int top_fill = have_left ? (int)dst[-1] : half - 1;
                for (int i = tid; i < 2 * h; i += kIpT) {
                    int v;
                    if (i < h) v = have_left ? (int)dst[(ptrdiff_t)imin(i, lpx - 1) * st - 1] : left_fill;
                    else if (have_bl) v = dst[(ptrdiff_t)(h + imin(i - h, lpx2 - 1)) * st - 1];
                    else v = have_left ? (int)dst[(ptrdiff_t)(lpx - 1) * st - 1] : left_fill;
                    tl[-(1 + i)] = v;
                }
                for (int i = tid; i < 2 * w; i += kIpT) {
                    int v;
                    if (i < w) v = have_top ? (int)top[imin(i, tpx - 1)] : top_fill;
                    else if (have_tr) v = top[w + imin(i - w, tpx2 - 1)];
                    else v = have_top ? (int)top[tpx - 1] : top_fill;
                    tl[1 + i] = v;
                }
                if (tid == 0)
                    tl[0] = have_left ? (have_top ? (int)top[-1] : (int)dst[-1]) : (have_top ? (int)top[0] : half);
                if (is_cfl) {
                    const int ssh = f.ss_hor, ssv = f.ss_ver, ys = cs[0];
                    // co-located luma block inside the luma canvas (:1346: position rounded down to even units)
                    const int lx = ((x << ssh) & ~ssh) * 4 - sx * 64, ly = ((y << ssv) & ~ssv) * 4 - sy * 64;
                    const pixel *ypx = canvas + co[0] + (1 + ly) * ys + 1 + lx;
                    int part = 0;
                    for (int i = tid; i < w * h; i += kIpT) {
                        const int yy = i / w, xx = i - yy * w;
                        const int syy = imin(yy, h - 4 * r.cfl_h_pad - 1), sxx = imin(xx, w - 4 * r.cfl_w_pad - 1);
                        const pixel *q = ypx + (ptrdiff_t)(syy << ssv) * ys + (sxx << ssh);
                        int sacc = q[0];
                        if (ssh) sacc += q[1];
                        if (ssv) { sacc += q[ys]; if (ssh) sacc += q[ys + 1]; }
                        sacc <<= 1 + !ssv + !ssh;
                        s_ac[i] = (int16_t)sacc;
                        part += sacc;
                    }
                    S.tile[tid] = part;
                }
                __syncthreads();
                if (tid == 0 && mode == B200_Z2_PRED && tw + th >= 6 && (r.angle_flags & 1024))
                    tl[0] = ((tl[-1] + tl[1]) * 5 + tl[0] * 6 + 8) >> 4;
                if (is_cfl && tid == 0) {
                    const int log2sz = (__ffs(w) - 1) + (__ffs(h) - 1);
                    int sum = (1 << log2sz) >> 1;
                    for (int i = 0; i < kIpT; i++) sum += S.tile[i];
                    S.dc = sum >> log2sz;
                }
                __syncthreads();
            }
            if (is_cfl) {
                const int dc = S.dc;
                for (int i = tid; i < w * h; i += kIpT) s_ac[i] = (int16_t)(s_ac[i] - dc);
                __syncthreads();
                ipred_cfl_pred_body<HBD>(S, dst, st, w, h, mode, r.cfl_alpha, s_ac, bdmax);
            } else {
                const int a = (mode == B200_FILTER_PRED ? r.angle : angle) | r.angle_flags;
                ipred_pred_body<HBD>(S, dst, st, w, h, mode, a, r.max_w, r.max_h, bdmax);
            }
            __syncthreads();
            if (r.eob >= 0) {
                if (tid == 0) { s_blk.dst_off = 0; s_blk.coef_off = 0; s_blk.eob = r.eob; s_blk.txtp = r.txtp; s_blk.plane = 0; }
                __syncthreads();
                switch (r.tx) {
#define X(TX, W, H, SH) case TX: itx_add_body<W, H, TX, SH, HBD, true>(0, s_itx, &s_blk, 1, s_cf, dst, st, st, st, bdmax, 0); break;
                B200_ITX_SIZES(X)
#undef X
                }
                if (f.zero_coefs)
                    for (int i = tid; i < ncf; i += kIpT) gcf[i] = 0;
            }
            __syncthreads();
            if (tid < kRecWords) s_rec[tid] = next_word;
            if (tid == 1 && ri + 1 < sb.count) {          // word 1 of the next record = coef_off: warm L2
                const char *cf = (const char *)((const coef *)f.d_coef + next_word);
                for (int k = 0; k < 8; k++) prefetch_l2(cf + k * 256);
            }
            __syncthreads();
        }

        // ---- write the superblock (the part inside the plane), publish
        for (int p = 0; p < 3; p++) {
            pixel *pic = (pixel *)f.pic + f.plane_off[p];
            const int st = f.stride[p];
            const int X0 = sx * sbw[p], Y0 = sy * sbh[p];
            const int ww = imin(sbw[p], f.w4[p] * 4 - X0), hh = imin(sbh[p], f.h4[p] * 4 - Y0);
            const pixel *cv = canvas + co[p] + cs[p] + 1;
            for (int i = tid; i < sbw[p] * hh; i += kIpT) {
                const int yy = i / sbw[p], xx = i - yy * sbw[p];
                if (xx < ww) pic[(ptrdiff_t)(Y0 + yy) * st + X0 + xx] = cv[yy * cs[p] + xx];
            }
        }
        __syncthreads();
        if (tid == 0) { __threadfence(); *(volatile uint8_t *)((P.scratch + P.done_off[0]) + sy * f.sb_w + sx) = 1; }
    }
}

// ---- band-sliced jobs: the rows band k+1 reads from above ---------------------------------------------------------
// Run at the end of band k's reconstruction, before its post filters: copies the last row of each plane of the band
// (luma y1 - 1, chroma (y1 >> ss_ver) - 1, `stride` samples each) into `edge`, then sets the header up for band k+1's
// launch (ticket 0, band row y1, edge). One CTA per plane.
struct EdgeBackupArgs {
    const unsigned char *src[3];
    uint32_t bytes[3], dst_off[3];
    unsigned char *edge;
    IntraHdr *hdr;
    int band_y;
};
constexpr int kEdgeThreads = 256;
__global__ void __launch_bounds__(kEdgeThreads) intra_edge_backup_kernel(const __grid_constant__ EdgeBackupArgs a)
{
    const int p = blockIdx.x;
    const unsigned char *const src = a.src[p];
    unsigned char *const dst = a.edge + a.dst_off[p];
    const uint32_t n = a.bytes[p];
    if (!(((uintptr_t)src | (uintptr_t)dst | n) & 3)) {
        for (uint32_t i = threadIdx.x; i < n >> 2; i += kEdgeThreads) ((uint32_t *)dst)[i] = ((const uint32_t *)src)[i];
    } else {
        for (uint32_t i = threadIdx.x; i < n; i += kEdgeThreads) dst[i] = src[i];
    }
    if (p == 0 && threadIdx.x == 0) { a.hdr->ticket = 0; a.hdr->band_y = a.band_y; a.hdr->edge = a.edge; }
}

int intra_edge_backup(int bdmax, const B200IntraFrame *f, int y1, void *edge, cudaStream_t stream)
{
    const size_t px = bdmax > 255 ? 2 : 1;
    EdgeBackupArgs a;
    memset(&a, 0, sizeof(a));
    uint32_t o = 0;
    for (int p = 0; p < 3; p++) {
        const int row = (p ? y1 >> f->ss_ver : y1) - 1;
        a.src[p] = (const unsigned char *)f->pic + (f->plane_off[p] + (size_t)row * f->stride[p]) * px;
        a.bytes[p] = (uint32_t)(f->stride[p] * px);
        a.dst_off[p] = o;
        o += a.bytes[p];
    }
    a.edge = (unsigned char *)edge;
    a.hdr = (IntraHdr *)f->scratch;
    a.band_y = y1;
    B200_LAUNCH(intra_edge_backup_kernel, dim3(3), dim3(kEdgeThreads), 0, stream, a);
    b200_count_launch();
    B200_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace b200

using namespace b200;

static int intra_frames_impl(int bdmax, const B200IntraFrame *frames, const B200IntraTx *const *d_tx, const int32_t *n_tx,
                             int n_frames, bool init, void *stream);

namespace b200 {
int intra_band(int bdmax, const B200IntraFrame *f, const B200IntraTx *d_tx, int n, bool first, cudaStream_t stream)
{
    if (n > 0) return intra_frames_impl(bdmax, f, &d_tx, &n, 1, first, stream);
    if (!first) return 0;
    // a first band without intra records still sets the done map up for the bands below it
    if (!f->scratch) { b200_set_error("b200_frame_run_band: no intra scratch"); return -2; }
    const IntraScratch L = intra_scratch_layout(f);
    if (f->done_init) B200_CUDA_OK(cudaMemcpyAsync(f->scratch, f->done_init, L.total, cudaMemcpyDeviceToDevice, stream));
    else B200_CUDA_OK(cudaMemsetAsync(f->scratch, 0, L.total, stream));
    return 0;
}
}  // namespace b200

extern "C" {

size_t b200_intra_scratch_bytes(const B200IntraFrame *f) { return intra_scratch_layout(f).total; }

static size_t intra_canvas_bytes(const B200IntraFrame *f, size_t px)
{
    size_t n = 0;
    for (int p = 0; p < 3; p++) {
        const int bw = 64 >> (p ? f->ss_hor : 0), bh = 64 >> (p ? f->ss_ver : 0);
        n += (size_t)(2 * bw + 2) * (bh + 1);
    }
    return (n * px + 15) & ~(size_t)15;
}

int b200_intra_frames(int bdmax, const B200IntraFrame *frames, const B200IntraTx *const *d_tx, const int32_t *n_tx,
                      int n_frames, void *stream)
{
    return intra_frames_impl(bdmax, frames, d_tx, n_tx, n_frames, true, stream);
}

}  // extern "C"

// init: set the scratch up (done map from done_init or zeroed, header zeroed) before the launch; false: a later band of a
// band-sliced job, whose done map holds the bands above and whose header the edge-backup kernel has set
static int intra_frames_impl(int bdmax, const B200IntraFrame *frames, const B200IntraTx *const *d_tx, const int32_t *n_tx,
                             int n_frames, bool init, void *stream)
{
    if (bdmax != 255 && bdmax != 1023 && bdmax != 4095) { b200_set_error("b200_intra_frames: bad bitdepth_max"); return -2; }
    const size_t px = bdmax > 255 ? 2 : 1;
    static const bool use_cta_kernel = getenv("B200_INTRA_CTA") != nullptr;      // round-1 CTA-per-block kernel (A/B measurements)
    for (int mode = 0; mode < 2; mode++)          // 0: per-transform-block dataflow, 1: superblock-granular
    for (int base = 0; base < n_frames; ) {
        IntraBatch B;
        memset(&B, 0, sizeof(B));
        int nb = 0, grid = 0, i = base;
        size_t dyn = 0;
        for (; i < n_frames && nb < kIntraMaxBatch; i++) {
            if (n_tx[i] <= 0) continue;
            const B200IntraFrame *f = &frames[i];
            if ((f->sb != nullptr) != (mode == 1)) continue;
            if (!f->scratch) { b200_set_error("b200_intra_frames: no scratch"); return -2; }
            if (mode == 1 && nb && (f->ss_hor != B.p[0].f.ss_hor || f->ss_ver != B.p[0].f.ss_ver)) break;   // one canvas layout per launch
            const IntraScratch L = intra_scratch_layout(f);
            IntraParams &P = B.p[nb++];
            P.f.pic = f->pic; P.f.ss_hor = f->ss_hor; P.f.ss_ver = f->ss_ver; P.f.d_coef = f->d_coef; P.f.zero_coefs = f->zero_coefs;
            for (int p = 0; p < 3; p++) { P.f.stride[p] = f->stride[p]; P.f.w4[p] = f->w4[p]; P.f.h4[p] = f->h4[p]; P.f.plane_off[p] = f->plane_off[p]; }
            P.f.n_sb = f->n_sb; P.f.sb_w = f->sb_w; P.f.sb_h = f->sb_h; P.f.sb = f->sb; P.f.mask = f->mask; P.f.pal = f->pal;
            P.tx = d_tx[i]; P.n = n_tx[i];
            uint8_t *base_p = (uint8_t *)f->scratch;
            P.scratch = base_p;
            for (int p = 0; p < 3; p++) P.done_off[p] = (uint32_t)L.done_off[p];
            if (!init)
                ;
            else if (!mode && f->done_init)
                B200_CUDA_OK(cudaMemcpyAsync(base_p, f->done_init, L.total, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
            else
                B200_CUDA_OK(cudaMemsetAsync(base_p, 0, mode ? 256 + (size_t)f->sb_w * f->sb_h : L.total, (cudaStream_t)stream));
            const int units = mode ? f->n_sb : n_tx[i];
            // warp-per-block kernel: two CTAs (8 blocks in flight) per SM fit its shared memory
            const int want = f->grid > 0 ? f->grid : (mode ? 16 : (use_cta_kernel ? kIntraGrid : 2 * kIntraGrid));
            grid = imax(grid, units < want ? units : want);
            if (mode) dyn = intra_canvas_bytes(f, px);
        }
        base = i;
        if (!nb) continue;
        if (mode == 0 && !use_cta_kernel) {
            // warp-per-block: a CTA carries kIwWarps blocks, so the same number of blocks in flight needs a quarter of the CTAs
            const size_t iw = kIwWarps * (bdmax > 255 ? sizeof(IwShared<true>) : sizeof(IwShared<false>));
#ifndef B200_EMU
            static bool iw_attr[2] = { false, false };
            if (!iw_attr[bdmax > 255]) {
                if (bdmax > 255) B200_CUDA_OK(cudaFuncSetAttribute(intra_warp_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)iw));
                else B200_CUDA_OK(cudaFuncSetAttribute(intra_warp_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)iw));
                iw_attr[bdmax > 255] = true;
            }
#endif
            if (bdmax > 255) { auto k = intra_warp_kernel<true>; B200_LAUNCH(k, dim3(grid, nb), dim3(kIwWarps * 32), iw, (cudaStream_t)stream, B, bdmax); }
            else { auto k = intra_warp_kernel<false>; B200_LAUNCH(k, dim3(grid, nb), dim3(kIwWarps * 32), iw, (cudaStream_t)stream, B, bdmax); }
        } else if (mode == 0) {
            if (bdmax > 255) { auto k = intra_frame_kernel<true>; B200_LAUNCH(k, dim3(grid, nb), dim3(kIpT), 0, (cudaStream_t)stream, B, bdmax); }
            else { auto k = intra_frame_kernel<false>; B200_LAUNCH(k, dim3(grid, nb), dim3(kIpT), 0, (cudaStream_t)stream, B, bdmax); }
        } else {
#ifndef B200_EMU
            static bool attr_set[2] = { false, false };
            if (!attr_set[bdmax > 255]) {
                if (bdmax > 255) B200_CUDA_OK(cudaFuncSetAttribute(intra_sb_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
                else B200_CUDA_OK(cudaFuncSetAttribute(intra_sb_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
                attr_set[bdmax > 255] = true;
            }
#endif
            if (bdmax > 255) { auto k = intra_sb_kernel<true>; B200_LAUNCH(k, dim3(grid, nb), dim3(kIpT), dyn, (cudaStream_t)stream, B, bdmax); }
            else { auto k = intra_sb_kernel<false>; B200_LAUNCH(k, dim3(grid, nb), dim3(kIpT), dyn, (cudaStream_t)stream, B, bdmax); }
        }
        b200_count_launch();
        B200_CUDA_OK(cudaGetLastError());
    }
    return 0;
}

extern "C" {

int b200_intra_frame(int bdmax, const B200IntraFrame *f, const B200IntraTx *d_tx, int n, void *stream)
{
    if (n <= 0) return 0;
    const int32_t nn = n;
    return b200_intra_frames(bdmax, f, &d_tx, &nn, 1, stream);
}

}  // extern "C"
