/*
 * b200av1.h — C ABI of the B200-native AV1 reconstruction / post-filter back end.
 *
 * Drop-in boundary for videolan/dav1d's block-reconstruction path (SURVEY.md §8b):
 *
 *   Level 1  b200_*_dsp_init_{8,16}bpc() fill tables of function pointers that have exactly
 *            the signatures of dav1d's Dav1dDSPContext members (reference src/internal.h:62-70;
 *            itx: src/itx.h:37-40,70-72). Each call ships its operands to HBM, launches the
 *            CUDA kernel and waits — correct but one block per launch; it is the semantic
 *            definition of the batched kernels and what the parity tests drive.
 *   Level 2  b200_*_batch() take arrays of block records already resident in HBM (device
 *            pointers) and process a whole frame's worth of work per launch; this is what
 *            a dav1d `f->bd_fn` record emitter (reference src/internal.h:247-262) feeds.
 *
 * Plain C: pointers, sizes, no C++/torch types. All functions return 0 on success and a
 * negative value on error (b200_last_error() gives the message) unless they mirror a
 * `void` dav1d signature. There is NO CPU fallback: without a CUDA device every entry
 * point fails.
 */
#ifndef B200AV1_H
#define B200AV1_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_API __attribute__((visibility("default")))

/* ---- library / context ------------------------------------------------------------- */
B200_API int b200_version(void);
B200_API const char *b200_last_error(void);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
B200_API uint64_t b200_launch_count(void);
/* programmatic dependent launch between the kernels of a frame job (default on; B200_NO_PDL=1 in the environment turns it
 * off): worth ~3 % on a single chain of whole-frame jobs, a loss when several chains of small launches share the GPU
 * (banded frames on two streams) — the frame pipeline switches it per configuration */
B200_API void b200_set_pdl(int on);

/* Device / pinned-host memory and streams for C hosts (a dav1d build has no other way to own HBM): thin
 * wrappers over cudaMalloc / cudaMallocHost / cudaStreamCreate. NULL on failure (b200_last_error() says why). */
B200_API void *b200_dev_alloc(size_t bytes);
B200_API void b200_dev_free(void *p);
B200_API void *b200_host_alloc(size_t bytes);      /* page-locked */
B200_API void b200_host_free(void *p);
B200_API void *b200_stream_create(void);
B200_API void b200_stream_destroy(void *stream);
B200_API int b200_dev_memset(void *p, int value, size_t bytes, void *stream);

/* enum RectTxfmSize / enum TxfmType numbering is dav1d's (reference src/levels.h:38-110) */
#define B200_N_RECT_TX_SIZES 19
#define B200_N_TX_TYPES_PLUS_LL 17
#define B200_WHT_WHT 16

/* ---- itx: Level 1 (replaces dav1d_itx_dsp_init_{8,16}bpc, reference src/itx_tmpl.c:220-311) */
/* typedefs mirror decl_itx_fn (reference src/itx.h:37-40) */
typedef void (*b200_itxfm_fn_8bpc)(uint8_t *dst, ptrdiff_t dst_stride, int16_t *coeff, int eob);
typedef void (*b200_itxfm_fn_16bpc)(uint16_t *dst, ptrdiff_t dst_stride, int32_t *coeff, int eob,
                                    int bitdepth_max);
/* same layout as Dav1dInvTxfmDSPContext (reference src/itx.h:70-72) */
typedef struct B200InvTxfmDSPContext8 {
    b200_itxfm_fn_8bpc itxfm_add[B200_N_RECT_TX_SIZES][B200_N_TX_TYPES_PLUS_LL];
} B200InvTxfmDSPContext8;
typedef struct B200InvTxfmDSPContext16 {
    b200_itxfm_fn_16bpc itxfm_add[B200_N_RECT_TX_SIZES][B200_N_TX_TYPES_PLUS_LL];
} B200InvTxfmDSPContext16;
B200_API void b200_itx_dsp_init_8bpc(B200InvTxfmDSPContext8 *c, int bpc);
B200_API void b200_itx_dsp_init_16bpc(B200InvTxfmDSPContext16 *c, int bpc);
/* non-table form of the same call (host pointers); bitdepth_max 255 selects 8 bpc */
B200_API int b200_inv_txfm_add(void *dst, ptrdiff_t dst_stride, void *coeff, int eob, int tx,
                               int txtp, int bitdepth_max);

/* ---- itx: Level 2 (batched, device-resident) ---------------------------------------- */
/* One transform block of a frame. All blocks of one b200_itx_add_batch call share `tx`.
 * dst_off: offset of the block's top-left pixel, in PIXELS, from the picture base pointer;
 * coef_off: offset in COEFFICIENTS into the coefficient stream. The block's coefficients are
 * min(w,32)*min(h,32) entries laid out as dav1d's decode_coefs writes them (x-frequency major:
 * coeff[y + x*min(h,32)], reference src/itx_tmpl.c:96-102), dequantised. */
typedef struct B200ItxBlock {
    uint32_t dst_off;
    uint32_t coef_off;
    int16_t eob;      /* as passed to itxfm_add (>= 0) */
    uint8_t txtp;     /* enum TxfmType, 16 = WHT_WHT */
    uint8_t plane;    /* index into stride_px[] */
} B200ItxBlock;

/* d_blocks/d_coef/d_pic are DEVICE pointers; stride_px[3] per-plane picture strides in pixels
 * (may be negative); stream is a cudaStream_t (NULL = default stream). The call is
 * asynchronous with respect to the host. If zero_coefs != 0 the consumed coefficients are
 * zeroed like dav1d's callee contract (reference src/itx_tmpl.c:108). */
B200_API int b200_itx_add_batch(int bitdepth_max, int tx, const B200ItxBlock *d_blocks, int n_blocks,
                                void *d_coef, void *d_pic, const int32_t stride_px[3],
                                int zero_coefs, void *stream);

/* All 19 transform sizes of a frame in one launch (d_blocks[tx] / n_blocks[tx] as above, sizes with
 * n_blocks[tx] <= 0 are skipped). Blocks of different sizes must not overlap in the picture. */
B200_API int b200_itx_add_frame(int bitdepth_max, const void *const d_blocks[19], const int32_t n_blocks[19],
                                void *d_coef, void *d_pic, const int32_t stride_px[3], int zero_coefs, void *stream);

/* Same work through HOST buffers (the end-to-end leg of bench.py): copies blocks, coefficients
 * and the picture to HBM, runs b200_itx_add_batch, copies the picture back, synchronises. */
B200_API int b200_itx_add_batch_host(int bitdepth_max, int tx, const B200ItxBlock *blocks, int n_blocks,
                                     void *coef, size_t coef_bytes, void *pic, size_t pic_bytes,
                                     const int32_t stride_px[3], int zero_coefs);

/* ==== mc (Dav1dMCDSPContext, reference src/mc.h:38-162, src/mc_tmpl.c) ================== */
/* horizontal upscaling of whole planes with dav1d's `resize` (reference src/mc_tmpl.c:918-944): per plane dst_w samples per row
 * from src_w, position step dx and start mx0 in 1/16384 sample units (f->resize_step / f->resize_start) */
typedef struct B200ResizeFrame {
    const void *src; void *dst;              /* device pictures */
    uint32_t src_plane_off[3], dst_plane_off[3];
    int32_t src_stride[3], dst_stride[3];    /* samples */
    int32_t src_w[3], dst_w[3], h[3];
    int32_t dx[3], mx0[3];
    int32_t n_planes, pad;
} B200ResizeFrame;
B200_API int b200_resize_frame(int bitdepth_max, const B200ResizeFrame *frame, void *stream);

#define B200_N_2D_FILTERS 10          /* enum Filter2d, reference src/levels.h:184-196 (9 = bilinear) */

/* ---- mc: Level 2 (batched, device-resident) ---- */
/* Shared geometry of one b200_mc_*_batch call. Reference pictures are 3-plane allocations;
 * ref_plane_off/ref_stride/ref_w/ref_h describe the planes (in pixels). Source coordinates that
 * fall outside [0,ref_w) x [0,ref_h) are clamped — exactly the replicate padding dav1d's
 * emu_edge builds for such blocks (reference src/recon_tmpl.c:960-977, src/mc_tmpl.c:868-916). */
typedef struct B200RefGeom {     /* a reference picture whose size is not the current frame's (scaled references) */
    uint32_t plane_off[3];
    int32_t stride[3];
    int32_t w[3], h[3];
} B200RefGeom;
typedef struct B200McFrame {
    const void *ref[8];          /* device base pointer per reference slot */
    uint32_t ref_plane_off[3];
    int32_t ref_stride[3];
    int32_t ref_w[3], ref_h[3];
    void *dst;                   /* device picture being reconstructed (dst_off includes the plane offset) */
    int32_t dst_stride[3];
    int16_t *tmp;                /* device int16 scratch: prep outputs / compound inputs */
    uint8_t *mask;               /* device uint8 scratch: w_mask outputs, mask / blend inputs */
    const void *px_tmp;          /* device pixel scratch: blend inputs (OBMC / inter-intra predictions); written by B200McBlock op 2 */
    uint32_t scaled_mask;        /* bit k: reference k has another size than the frame being decoded and its planes are described by
                                    ref_geom[k] instead of ref_plane_off / ref_stride / ref_w / ref_h. Only B200McScaledBlock records
                                    may name such a reference (reference src/recon_tmpl.c:991-1046, f->svc[refidx]). */
    uint32_t pad_geom;
    B200RefGeom ref_geom[8];
} B200McFrame;

/* one prediction block: dav1d's mc[filter2d] (op 0, "put") or mct[filter2d] (op 1, "prep") */
typedef struct B200McBlock {
    uint32_t dst_off;            /* put: pixel offset in dst (op 2: in px_tmp); prep: int16 offset in tmp (dense, pitch w) */
    int32_t src_x, src_y;        /* integer sample position of the block's top-left in the ref plane */
    uint8_t w, h;                /* w in {2,4,..,128}; 2 <= h <= 128 */
    uint8_t mx, my;              /* subpel phase 0..15 */
    uint8_t filter2d;
    uint8_t op;                  /* 0 put, 1 prep, 2 put into px_tmp (dst_off = pixel offset there, dense, pitch w) */
    uint8_t plane;
    uint8_t ref;
} B200McBlock;
B200_API int b200_mc_batch(int bitdepth_max, const B200McFrame *frame, const B200McBlock *d_blocks,
                           int n_blocks, void *stream);

/* compound combine of two prep outputs: avg / w_avg / mask / w_mask (reference src/mc_tmpl.c:628-781) */
enum { B200_COMP_AVG = 0, B200_COMP_W_AVG = 1, B200_COMP_MASK = 2, B200_COMP_W_MASK_444 = 3,
       B200_COMP_W_MASK_422 = 4, B200_COMP_W_MASK_420 = 5 };
typedef struct B200CompBlock {
    uint32_t dst_off;            /* pixel offset in dst */
    uint32_t tmp1_off, tmp2_off; /* int16 offsets in frame->tmp */
    uint32_t mask_off;           /* offset in frame->mask (mask: input; w_mask: output) */
    uint8_t w, h;
    uint8_t op;
    uint8_t param;               /* w_avg: weight 0..16; w_mask: sign */
    uint8_t plane;
    uint8_t pad[3];
} B200CompBlock;
B200_API int b200_mc_comp_batch(int bitdepth_max, const B200McFrame *frame, const B200CompBlock *d_blocks,
                                int n_blocks, void *stream);

/* Fused compound prediction: both mct[] predictions and avg / w_avg / mask / w_mask in one pass, the int16
 * intermediates never leave the SM (same arithmetic, bit-identical to prep + compound). `mask` / `w_mask` use
 * frame->mask at mask_off exactly like B200CompBlock (mask: input, pitch w; w_mask: output). */
typedef struct B200CompFusedBlock {
    uint32_t dst_off;            /* pixel offset in dst */
    uint32_t mask_off;
    int32_t src_x[2], src_y[2];  /* integer sample position of the block's top-left in each reference plane */
    uint8_t w, h;
    uint8_t mx[2], my[2];        /* subpel phases 0..15 */
    uint8_t ref[2];
    uint8_t filter2d, op, param, plane;
    uint8_t pad[4];
} B200CompFusedBlock;
B200_API int b200_mc_comp_fused_batch(int bitdepth_max, const B200McFrame *frame, const B200CompFusedBlock *d_blocks,
                                      int n_blocks, void *stream);

/* blend / blend_v / blend_h (reference src/mc_tmpl.c:683-722) */
enum { B200_BLEND = 0, B200_BLEND_V = 1, B200_BLEND_H = 2 };
typedef struct B200BlendBlock {
    uint32_t dst_off;            /* pixel offset in dst */
    uint32_t tmp_off;            /* pixel offset in frame->px_tmp (dense, pitch w) */
    uint32_t mask_off;           /* B200_BLEND only: offset in frame->mask */
    uint8_t w, h, op, plane;
} B200BlendBlock;
B200_API int b200_mc_blend_batch(int bitdepth_max, const B200McFrame *frame, const B200BlendBlock *d_blocks,
                                 int n_blocks, void *stream);

/* 8x8 affine warp: warp8x8 (op 0) / warp8x8t (op 1) (reference src/mc_tmpl.c:799-866) */
typedef struct B200WarpBlock {
    uint32_t dst_off;            /* op 0: pixel offset in dst; op 1: int16 offset in tmp */
    int32_t src_x, src_y;        /* position of the 8x8 block's top-left (row 0, col 0 of the 15x15 window is -3,-3) */
    int32_t mx, my;
    int16_t abcd[4];
    uint16_t tmp_stride;         /* op 1: pitch of tmp in int16 elements */
    uint8_t op, plane, ref, pad;
} B200WarpBlock;
B200_API int b200_mc_warp_batch(int bitdepth_max, const B200McFrame *frame, const B200WarpBlock *d_blocks,
                                int n_blocks, void *stream);

/* scaled references: mc_scaled[filter2d] (op 0) / mct_scaled[filter2d] (op 1) (reference src/mc_tmpl.c:189-244,
 * 307-358, 491-531, 588-626; caller src/recon_tmpl.c:991-1046). Positions advance by dx / dy 1/1024ths of a sample
 * per output column / row; src_x, src_y is the sample that (mx, my) = (0, 0) addresses. Source coordinates are
 * clamped to the reference plane (= emu_edge). */
typedef struct B200McScaledBlock {
    uint32_t dst_off;            /* put: pixel offset in dst; prep: int16 offset in tmp (dense, pitch w) */
    int32_t src_x, src_y;
    uint16_t mx, my;             /* 0 .. 1023 */
    uint16_t dx, dy;             /* 1 .. 2048 */
    uint8_t w, h;                /* 2 .. 128 */
    uint8_t filter2d, op, plane, ref;      /* op: 0 put, 1 prep (int16 into tmp), 2 put into px_tmp (pitch w) like B200McBlock */
    uint8_t pad[2];
} B200McScaledBlock;
B200_API int b200_mc_scaled_batch(int bitdepth_max, const B200McFrame *frame, const B200McScaledBlock *d_blocks,
                                  int n_blocks, void *stream);

/* ---- mc: Level 1 (host pointers, dav1d signatures; bitdepth_max appended like HIGHBD_DECL_SUFFIX) */
B200_API int b200_mc_put_scaled(void *dst, ptrdiff_t dst_stride, const void *src, ptrdiff_t src_stride, int w, int h,
                                int mx, int my, int dx, int dy, int filter2d, int bitdepth_max);
B200_API int b200_mc_prep_scaled(int16_t *tmp, const void *src, ptrdiff_t src_stride, int w, int h, int mx, int my,
                                 int dx, int dy, int filter2d, int bitdepth_max);
B200_API int b200_mc_put(void *dst, ptrdiff_t dst_stride, const void *src, ptrdiff_t src_stride,
                         int w, int h, int mx, int my, int filter2d, int bitdepth_max);
B200_API int b200_mc_prep(int16_t *tmp, const void *src, ptrdiff_t src_stride, int w, int h,
                          int mx, int my, int filter2d, int bitdepth_max);
B200_API int b200_mc_comp(void *dst, ptrdiff_t dst_stride, const int16_t *tmp1, const int16_t *tmp2,
                          int w, int h, int op, int param, uint8_t *mask, int bitdepth_max);
B200_API int b200_mc_blend(void *dst, ptrdiff_t dst_stride, const void *tmp, int w, int h, int op,
                           const uint8_t *mask, int bitdepth_max);
B200_API int b200_mc_warp8x8(int op, void *out, ptrdiff_t out_stride, const void *src, ptrdiff_t src_stride,
                             const int16_t *abcd, int mx, int my, int bitdepth_max);
B200_API int b200_mc_emu_edge(intptr_t bw, intptr_t bh, intptr_t iw, intptr_t ih, intptr_t x, intptr_t y,
                              void *dst, ptrdiff_t dst_stride, const void *ref, ptrdiff_t ref_stride,
                              int bitdepth_max);
B200_API int b200_mc_resize(void *dst, ptrdiff_t dst_stride, const void *src, ptrdiff_t src_stride,
                            int dst_w, int h, int src_w, int dx, int mx, int bitdepth_max);

/* same layout as Dav1dMCDSPContext (reference src/mc.h:146-162) */
typedef struct B200MCDSPContext {
    void *mc[B200_N_2D_FILTERS];
    void *mc_scaled[B200_N_2D_FILTERS];
    void *mct[B200_N_2D_FILTERS];
    void *mct_scaled[B200_N_2D_FILTERS];
    void *avg, *w_avg, *mask, *w_mask[3], *blend, *blend_v, *blend_h, *warp8x8, *warp8x8t, *emu_edge, *resize;
} B200MCDSPContext;
B200_API void b200_mc_dsp_init_8bpc(B200MCDSPContext *c);
B200_API void b200_mc_dsp_init_16bpc(B200MCDSPContext *c);

/* ==== loopfilter (Dav1dLoopFilterDSPContext, reference src/loopfilter.h:39-53) =========== */
/* byte-identical to dav1d's Av1FilterLUT / Av1Filter (reference src/lf_mask.h:36-57): a dav1d
 * record emitter ships f->lf.lim_lut and f->lf.mask[] (after the tile-edge fix-ups of
 * src/lf_apply_tmpl.c:331-401) and f->lf.level[] to HBM unchanged. */
typedef struct B200FilterLUT {
    uint8_t e[64];
    uint8_t i[64];
    uint64_t sharp[2];
} B200FilterLUT;
typedef struct B200Av1Filter {
    uint16_t filter_y[2 /* 0=col, 1=row */][32][3][2];
    uint16_t filter_uv[2 /* 0=col, 1=row */][32][2][2];
    int8_t cdef_idx[4];
    uint16_t noskip_mask[16][2];
} B200Av1Filter;

/* Level 2: deblock a whole picture in HBM (replaces dav1d_loopfilter_sbrow_cols/_rows for every
 * superblock row, reference src/lf_apply_tmpl.c:313-466): one sweep over all column edges of
 * all planes, then one over all row edges. */
typedef struct B200LfFrame {
    void *pic;                     /* device picture, 3 planes */
    uint32_t plane_off[3];         /* pixels */
    int32_t stride[3];             /* pixels */
    int32_t w4, h4;                /* f->w4, f->h4: picture size in luma 4-px units */
    int32_t sb128w;                /* f->sb128w */
    int32_t b4_stride;             /* f->b4_stride */
    int32_t ss_hor, ss_ver;        /* chroma subsampling */
    int32_t sb128;                 /* informational (walk order only matters on the CPU) */
    int32_t filter_y, filter_uv;   /* frame header: level_y[0]|level_y[1], level_u|level_v */
    const B200Av1Filter *mask;     /* device, sb128w * ceil(h4/32) entries */
    const uint8_t (*level)[4];     /* device, f->lf.level */
    B200FilterLUT lut;
} B200LfFrame;
B200_API int b200_lf_frame(int bitdepth_max, const B200LfFrame *frame, void *stream);

/* Level 1: loop_filter_sb[plane_class][dir] with host pointers (decl_loopfilter_sb_fn) */
B200_API int b200_loop_filter_sb(int plane_class, int dir, void *dst, ptrdiff_t stride, const uint32_t *mask,
                                 const uint8_t (*lvl)[4], ptrdiff_t lvl_stride, const B200FilterLUT *lut,
                                 int w, int bitdepth_max);
typedef struct B200LoopFilterDSPContext { void *loop_filter_sb[2][2]; } B200LoopFilterDSPContext;
B200_API void b200_loop_filter_dsp_init_8bpc(B200LoopFilterDSPContext *c);
B200_API void b200_loop_filter_dsp_init_16bpc(B200LoopFilterDSPContext *c);

/* ==== cdef (Dav1dCdefDSPContext, reference src/cdef.h:53-67) ============================= */
enum { B200_CDEF_HAVE_LEFT = 1, B200_CDEF_HAVE_RIGHT = 2, B200_CDEF_HAVE_TOP = 4, B200_CDEF_HAVE_BOTTOM = 8 };

/* Level 2: CDEF over a whole deblocked picture, OUT OF PLACE (src -> dst; every 8x8 of the
 * bw x bh area is written, unfiltered blocks are copied through). Replaces dav1d_cdef_brow for
 * every superblock row (reference src/cdef_apply_tmpl.c:97-308); CDEF only ever reads pre-CDEF
 * samples, which is what the reference's cdef_line / lr_bak backups emulate in place. */
typedef struct B200CdefFrame {
    const void *src;               /* device, deblocked picture */
    void *dst;                     /* device, same geometry */
    uint32_t plane_off[3];
    int32_t stride[3];
    int32_t bw, bh;                /* f->bw, f->bh (4-px units) */
    int32_t sb128w, ss_hor, ss_ver;
    int32_t damping;               /* frame_hdr->cdef.damping */
    int32_t y_strength[8], uv_strength[8];   /* frame_hdr->cdef.{y,uv}_strength */
    const B200Av1Filter *mask;     /* device: cdef_idx[] and noskip_mask[] are read */
} B200CdefFrame;
B200_API int b200_cdef_frame(int bitdepth_max, const B200CdefFrame *frame, void *stream);

/* Level 1 (host pointers): cdef.dir and cdef.fb[0..2] = 8x8 / 4x8 / 4x4 */
B200_API int b200_cdef_dir(const void *img, ptrdiff_t stride, unsigned *var, int bitdepth_max);
B200_API int b200_cdef_fb(void *dst, ptrdiff_t stride, const void *left, const void *top, const void *bottom,
                          int pri_strength, int sec_strength, int dir, int damping, int w, int h, int edges,
                          int bitdepth_max);
typedef struct B200CdefDSPContext { void *dir; void *fb[3]; } B200CdefDSPContext;
B200_API void b200_cdef_dsp_init_8bpc(B200CdefDSPContext *c);
B200_API void b200_cdef_dsp_init_16bpc(B200CdefDSPContext *c);

/* ==== looprestoration (Dav1dLoopRestorationDSPContext, reference src/looprestoration.h:49-75) == */
enum { B200_LR_HAVE_LEFT = 1, B200_LR_HAVE_RIGHT = 2, B200_LR_HAVE_TOP = 4, B200_LR_HAVE_BOTTOM = 8 };
/* byte-identical to dav1d's Av1RestorationUnit / Av1Restoration (reference src/lf_mask.h:42-62) */
typedef struct B200RestorationUnit {
    uint8_t type;                  /* 0 none, 2 Wiener, 3 + sgr_idx self-guided */
    int8_t filter_h[3], filter_v[3];
    int8_t sgr_weights[2];
} B200RestorationUnit;
typedef struct B200Av1Restoration { B200RestorationUnit lr[3][4]; } B200Av1Restoration;

/* Level 2: restore a whole picture, OUT OF PLACE. `cdef` is the picture after CDEF (rows inside a
 * 64-row stripe), `dbl` the picture after deblocking / before CDEF (the two rows above and below each
 * stripe boundary: what dav1d_copy_lpf saves, reference src/lf_apply_tmpl.c:40-174), `dst` receives the
 * restored picture (unrestored units are copied through). Replaces dav1d_lr_sbrow for every superblock
 * row (reference src/lr_apply_tmpl.c:36-202); the unit lookup in lr_mask[] is dav1d's. */
typedef struct B200LrFrame {
    const void *cdef, *dbl;
    void *dst;
    uint32_t plane_off[3];
    int32_t stride[3];
    int32_t w, h;                  /* picture size in luma pixels (f->sr_cur.p.p.w / h) */
    int32_t ss_hor, ss_ver, sb128, sr_sb128w;
    int32_t unit_size_log2[2];     /* frame_hdr->restoration.unit_size[y, uv] */
    int32_t restore_planes;        /* f->lf.restore_planes */
    const B200Av1Restoration *lr_mask;   /* device, f->lf.lr_mask */
} B200LrFrame;
B200_API int b200_lr_frame(int bitdepth_max, const B200LrFrame *frame, void *stream);

/* Level 1 (host pointers, decl_lr_filter_fn): kind 0 = wiener (7- and 5-tap), 1..3 = sgr 5x5 / 3x3 / mix.
 * `params` points at a LooprestorationParams (int16 filter[2][8] or {uint32 s0, s1; int16 w0, w1}). */
B200_API int b200_lr_filter(int kind, void *dst, ptrdiff_t stride, const void *left, const void *lpf, int w, int h,
                            const void *params, int edges, int bitdepth_max);
typedef struct B200LoopRestorationDSPContext { void *wiener[2]; void *sgr[3]; } B200LoopRestorationDSPContext;
B200_API void b200_loop_restoration_dsp_init_8bpc(B200LoopRestorationDSPContext *c, int bpc);
B200_API void b200_loop_restoration_dsp_init_16bpc(B200LoopRestorationDSPContext *c, int bpc);

/* ==== ipred (Dav1dIntraPredDSPContext, reference src/ipred.h:44-90) ======================= */
/* DSP-table mode indices (reference src/levels.h:112-136) */
enum { B200_DC_PRED = 0, B200_VERT_PRED = 1, B200_HOR_PRED = 2, B200_LEFT_DC_PRED = 3, B200_TOP_DC_PRED = 4,
       B200_DC_128_PRED = 5, B200_Z1_PRED = 6, B200_Z2_PRED = 7, B200_Z3_PRED = 8, B200_SMOOTH_PRED = 9,
       B200_SMOOTH_V_PRED = 10, B200_SMOOTH_H_PRED = 11, B200_PAETH_PRED = 12, B200_FILTER_PRED = 13 };
enum { B200_IPRED_OP_PRED = 0, B200_IPRED_OP_CFL_PRED = 1, B200_IPRED_OP_PAL_PRED = 2, B200_IPRED_OP_CFL_AC = 3 };

/* Level 2: independent intra blocks whose edge arrays are already assembled (what
 * dav1d_prepare_intra_edges produces, reference src/ipred_prepare_tmpl.c:75-204). */
typedef struct B200IpredFrame {
    void *dst;                     /* device picture */
    int32_t dst_stride[3];
    int32_t ss_hor, ss_ver;        /* for cfl_ac */
    const void *edge;              /* device pixel buffer holding every block's edge array / palette */
    int16_t *ac;                   /* device int16 buffer: cfl_ac outputs, cfl_pred inputs (dense, pitch w) */
    const uint8_t *pal_idx;        /* device palette index bytes (two 3-bit indices per byte) */
} B200IpredFrame;
typedef struct B200IpredBlock {
    uint32_t dst_off;              /* pixel offset in dst (cfl_ac: of the luma block in dst) */
    uint32_t edge_off;             /* pixel index of `topleft` inside edge (pal_pred: of pal[8]) */
    uint32_t ac_off;               /* int16 offset in ac (pal_pred: byte offset in pal_idx) */
    int32_t max_w, max_h;          /* Z2 only */
    int16_t angle;                 /* angle | flags (Z modes), filter index (FILTER), w_pad | h_pad << 8 (cfl_ac) */
    int8_t alpha;                  /* cfl_pred */
    uint8_t w, h, mode, op, plane;
} B200IpredBlock;
B200_API int b200_ipred_batch(int bitdepth_max, const B200IpredFrame *frame, const B200IpredBlock *d_blocks,
                              int n_blocks, void *stream);

/* Level 1 (host pointers) */
B200_API int b200_ipred(int mode, void *dst, ptrdiff_t stride, const void *topleft, int w, int h, int angle,
                        int max_w, int max_h, int bitdepth_max);
B200_API int b200_cfl_ac(int16_t *ac, const void *ypx, ptrdiff_t stride, int w_pad, int h_pad, int cw, int ch,
                         int ss_hor, int ss_ver, int bitdepth_max);
B200_API int b200_cfl_pred(int mode, void *dst, ptrdiff_t stride, const void *topleft, int w, int h,
                           const int16_t *ac, int alpha, int bitdepth_max);
B200_API int b200_pal_pred(void *dst, ptrdiff_t stride, const void *pal, const uint8_t *idx, int w, int h,
                           int bitdepth_max);
typedef struct B200IntraPredDSPContext {
    void *intra_pred[14];
    void *cfl_ac[3];               /* 420, 422, 444 */
    void *cfl_pred[6];
    void *pal_pred;
} B200IntraPredDSPContext;
B200_API void b200_intra_pred_dsp_init_8bpc(B200IntraPredDSPContext *c);
B200_API void b200_intra_pred_dsp_init_16bpc(B200IntraPredDSPContext *c);

/* ==== filmgrain (Dav1dFilmGrainDSPContext, reference src/filmgrain.h:46-80) ================ */
/* byte-identical to Dav1dFilmGrainData (reference include/dav1d/headers.h:315-333), 224 bytes */
typedef struct B200FilmGrainData {
    unsigned seed;
    int num_y_points;
    uint8_t y_points[14][2];
    int chroma_scaling_from_luma;
    int num_uv_points[2];
    uint8_t uv_points[2][10][2];
    int scaling_shift;
    int ar_coeff_lag;
    int8_t ar_coeffs_y[24];
    int8_t ar_coeffs_uv[2][25 + 3];
    uint64_t ar_coeff_shift;
    int grain_scale_shift;
    int uv_mult[2];
    int uv_luma_mult[2];
    int uv_offset[2];
    int overlap_flag;
    int clip_to_restricted_range;
} B200FilmGrainData;
#define B200_GRAIN_WIDTH 82
#define B200_GRAIN_HEIGHT 73
#define B200_FG_SCRATCH_BYTES (256 * 1024)

/* Level 2: grain synthesis + application for a whole picture, out of place (in -> out), like
 * dav1d_apply_grain (reference src/fg_apply_tmpl.c:100-240): one small kernel builds the three grain
 * LUTs (LFSR + Gaussian table + AR filter run as a skewed wavefront), the scaling LUTs and the
 * per-32x32-block offsets in `scratch` (device, >= B200_FG_SCRATCH_BYTES), then one sweep applies the
 * noise to all planes. */
typedef struct B200FgFrame {
    const void *in;
    void *out;
    uint32_t plane_off[3];
    int32_t stride[3];
    int32_t w, h, ss_hor, ss_ver;
    int32_t is_id;                 /* seq_hdr->mtrx == DAV1D_MC_IDENTITY */
    B200FilmGrainData data;
    void *scratch;
} B200FgFrame;
B200_API int b200_fg_apply_frame(int bitdepth_max, const B200FgFrame *frame, void *stream);
/* the two halves of the above: prep touches only frame->data / geometry / scratch, apply needs in / out too */
B200_API int b200_fg_prep(int bitdepth_max, const B200FgFrame *frame, void *stream);
B200_API int b200_fg_apply(int bitdepth_max, const B200FgFrame *frame, void *stream);

/* Level 1 (host pointers). Grain LUT entries are int8 (8 bpc) / int16 (10, 12 bpc), pitch 82. */
B200_API int b200_fg_generate_grain(void *buf, const void *buf_y, const B200FilmGrainData *data, int uv,
                                    int ss_hor, int ss_ver, int bitdepth_max);   /* uv < 0: luma */
B200_API int b200_fgy_32x32xn(void *dst_row, const void *src_row, ptrdiff_t stride, const B200FilmGrainData *data,
                              size_t pw, const uint8_t *scaling, const void *grain_lut, int bh, int row_num,
                              int bitdepth_max);
B200_API int b200_fguv_32x32xn(void *dst_row, const void *src_row, ptrdiff_t stride, const B200FilmGrainData *data,
                               size_t pw, const uint8_t *scaling, const void *grain_lut, int bh, int row_num,
                               const void *luma_row, ptrdiff_t luma_stride, int uv_pl, int is_id, int ss_hor,
                               int ss_ver, int bitdepth_max);
typedef struct B200FilmGrainDSPContext {
    void *generate_grain_y;
    void *generate_grain_uv[3];
    void *fgy_32x32xn;
    void *fguv_32x32xn[3];
} B200FilmGrainDSPContext;
B200_API void b200_film_grain_dsp_init_8bpc(B200FilmGrainDSPContext *c);
B200_API void b200_film_grain_dsp_init_16bpc(B200FilmGrainDSPContext *c);

/* ==== intra reconstruction of a whole frame ================================================== */
/* One record per TRANSFORM block of an intra-coded block, because dav1d predicts, then adds the residual, at
 * transform-block granularity (dav1d_recon_b_intra, reference src/recon_tmpl.c:1176-1555): each block's edge
 * pixels are the reconstructed pixels of its neighbours. The device prepares the edge arrays itself
 * (dav1d_prepare_intra_edges, reference src/ipred_prepare_tmpl.c:75-204), predicts, adds the inverse transform
 * and publishes the block in a per-4x4 "done" map; a persistent grid takes records in order and each CTA waits
 * for the map cells its edges read. Records must therefore be in a topological order of those dependencies
 * (decode order is one; sorted by wavefront number is the efficient one). */
enum { B200_INTRA_HAVE_LEFT = 1, B200_INTRA_HAVE_TOP = 2, B200_INTRA_TOP_HAS_RIGHT = 4, B200_INTRA_LEFT_HAS_BOTTOM = 8 };
enum { B200_INTRA_MODE_FILTER = 13, B200_INTRA_MODE_CFL = 14,   /* besides enum IntraPredMode DC_PRED(0)..PAETH_PRED(12) */
       /* inter-intra (reference src/recon_tmpl.c:1601-1626, 1737-1777): the block's inter prediction is already in the
        * picture (prediction stage); an II record predicts `angle` (= DC / VERT / HOR / SMOOTH_PRED) over the whole
        * block (`tx` = the block's size) from the reconstructed neighbours and blends it in with the mask at `luma_off`
        * bytes into B200IntraFrame.mask (pitch = block width). It carries no residual: the block's transform blocks
        * follow as RESID records, which add their residual to the pixels in place. cfl_alpha != 0 in the II record says
        * that RESID records follow (the done map then holds 2 = "predicted" until they publish 1 = "final"). */
       B200_INTRA_MODE_II = 15, B200_INTRA_MODE_RESID = 16,
       /* palette (reference src/recon_tmpl.c:1201-1223, 1400-1419; pal_pred_c src/ipred_tmpl.c:717-730): a PAL record covers
        * the whole block (`tx` = the block's size); `luma_off` = byte offset into B200IntraFrame.pal of 8 palette entries
        * (pixels) followed by the w x h index map, two 4-bit indices per byte, low nibble first, pitch w / 2 (dav1d's
        * packed pal_idx). Like II it carries no residual: RESID records follow when cfl_alpha != 0. */
       B200_INTRA_MODE_PAL = 17,
       /* intra block copy (reference src/recon_tmpl.c:1583-1596, src/decode.c:1286-1345): the block is predicted from an
        * already reconstructed area of the SAME picture with dav1d's bilinear put (luma vectors are whole samples, sub-sampled
        * chroma may sit on a half sample). An IBC record covers the whole block (`tx` = its size, blocks wider / taller than
        * 64 come as several records); `luma_off` = source position in this plane, (y << 16) | x, samples; cfl_w_pad /
        * cfl_h_pad = the mx / my phase handed to mc[FILTER_2D_BILINEAR] (0 or 8). Source samples are clamped to the plane
        * area w4 * 4 x h4 * 4 (emu_edge). The record waits until every 4x4 cell it reads is final. Like II it carries no
        * residual: RESID records follow when cfl_alpha != 0. Per-transform-block schedule only (not with B200IntraFrame.sb). */
       B200_INTRA_MODE_IBC = 18 };
typedef struct B200IntraTx {
    uint32_t dst_off;              /* sample offset of the transform block in the picture (plane offset included) */
    uint32_t coef_off;             /* into d_coef, dav1d's transposed layout, min(w,32) x min(h,32) */
    uint32_t luma_off;             /* CFL only: sample offset of the co-located luma block (y_src, :1346) */
    int16_t eob;                   /* < 0: no residual */
    uint16_t x4, y4;               /* position in this plane, 4-sample units (t->bx >> ss_hor, t->by >> ss_ver) */
    uint16_t xend4, yend4;         /* ts->tiling.col_end / row_end (>> ss) : where available edge pixels stop */
    int16_t max_w, max_h;          /* the Z2 limits handed to intra_pred (:1276-1277, :1474-1477) */
    uint16_t angle_flags;          /* sm_flag | sm_uv_flag (512), intra_edge_filter << 10 (:1205, :1233) */
    uint8_t tx, txtp;              /* enum RectTxfmSize, enum TxfmType */
    uint8_t mode;                  /* y_mode / uv_mode as coded, B200_INTRA_MODE_FILTER, B200_INTRA_MODE_CFL */
    int8_t angle;                  /* y_angle / uv_angle (-3..3); filter-intra: the filter index */
    uint8_t plane;
    uint8_t flags;                 /* B200_INTRA_* availability bits (have_left/have_top and enum EdgeFlags) */
    int8_t cfl_alpha;              /* CFL: alpha of this plane (0 = plain DC_PRED, :1446-1451) */
    uint8_t cfl_w_pad, cfl_h_pad;  /* CFL: cfl_ac padding arguments, 4-sample units (:1359-1362) */
    uint8_t pad[3];
} B200IntraTx;
/* Superblock-granular scheduling (optional, 64x64 superblocks): records sorted by superblock, decode order inside;
 * one B200IntraSb per superblock in ticket order, which must be a topological order of the superblock
 * dependencies left / top-left / top / top-right (raster order is one; sorted by sx + 2*sy is the efficient one). */
typedef struct B200IntraSb {
    uint32_t first, count;         /* records [first, first + count) of d_tx */
    uint16_t sx, sy;               /* superblock position */
} B200IntraSb;
typedef struct B200IntraFrame {
    void *pic;                     /* device picture being reconstructed */
    int32_t stride[3];
    int32_t ss_hor, ss_ver;
    int32_t w4[3], h4[3];          /* per plane: frame size in 4-sample units (done-map geometry) */
    void *d_coef;
    int32_t zero_coefs;
    int32_t grid;                  /* CTAs to launch; 0 = default */
    void *scratch;                 /* device, >= b200_intra_scratch_bytes(frame) */
    uint32_t plane_off[3];         /* superblock mode and band-sliced jobs: sample offset of each plane in pic */
    int32_t n_sb, sb_w, sb_h;      /* superblock mode: number of B200IntraSb, superblock grid */
    const B200IntraSb *sb;         /* device; NULL = per-transform-block dataflow */
    const uint8_t *mask;           /* device or NULL: blend masks of B200_INTRA_MODE_II records (per-transform-block mode only) */
    const uint8_t *pal;            /* device or NULL: palettes + index maps of B200_INTRA_MODE_PAL records */
    const uint8_t *done_init;      /* device or NULL; per-transform-block mode only. Frames that mix inter and intra blocks:
                                      an image of the scratch (b200_intra_scratch_bytes: 256 zero bytes, then one byte per
                                      4x4 cell for plane 0, 1, 2, each map padded to a multiple of 256 bytes) in which the
                                      cells NOT covered by an intra record are 1 — their pixels are final before the
                                      kernel starts (the inter stages ran) — and the cells of intra records are 0 */
} B200IntraFrame;
B200_API size_t b200_intra_scratch_bytes(const B200IntraFrame *frame);
B200_API int b200_intra_frame(int bitdepth_max, const B200IntraFrame *frame, const B200IntraTx *d_tx, int n_tx,
                              void *stream);
/* Several independent frames (same bit depth) in one call: up to 24 frames share a launch (one grid row per frame), so
 * the number of frames in flight is not tied to the number of streams / hardware work queues. */
B200_API int b200_intra_frames(int bitdepth_max, const B200IntraFrame *frames, const B200IntraTx *const *d_tx,
                               const int32_t *n_tx, int n_frames, void *stream);

/* ==== compact coefficient upload ============================================================= */
/* Per coded transform block the emitter may ship only coefficients 0 .. eob in scan order (dav1d_scans[tx],
 * reference src/scan.c) instead of the dense block: b200_coef_expand scatters them into the (zeroed) dense buffer
 * the transform kernels read. In a B200FrameJob: d_expand / n_expand / d_ccoef / coef_bytes; b200_frame_run then
 * zeroes d_coef[0 .. coef_bytes) and expands before anything else. */
typedef struct B200CoefBlock {
    uint32_t dense_off;            /* coefficient index of the block in the dense buffer (= its coef_off) */
    uint32_t compact_off;          /* coefficient index of its first value in the compact stream */
    int16_t eob;
    uint8_t tx, pad;
} B200CoefBlock;
B200_API int b200_coef_expand(int bitdepth_max, const B200CoefBlock *d_blocks, int n_blocks, const void *d_compact,
                              void *d_dense, void *stream);

/* ==== whole-frame job: reconstruction + post-filter sweep ================================= */
/* What a dav1d `f->bd_fn` record emitter hands over per frame (SURVEY.md §8b level 2): the block
 * records of pass 2 (prediction blocks, compound / blend / warp records, transform blocks bucketed by
 * transform size with their coefficient stream) and the post-filter parameters, all already in HBM.
 * b200_frame_run enqueues, on `stream`:
 *    prediction (put/prep) -> warp -> compound -> compound stage 2 -> blend -> blend stage 2 -> inverse transforms (one launch per size)
 *    -> deblock (2 sweeps, in place on the reconstructed picture) -> CDEF (out of place) -> loop
 *    restoration (out of place) -> film grain (out of place, into the display copy).
 * Stages whose counts / run_* flags are zero are skipped. Picture chaining is the caller's: typically
 * mc.dst == lf.pic == cdef.src == lr.dbl, cdef.dst == lr.cdef, lr.dst = output. */
typedef struct B200FrameJob {
    int32_t bitdepth_max;
    int32_t zero_coefs;
    B200McFrame mc;
    const B200McBlock *d_pred;   int32_t n_pred;   int32_t pad0;
    const B200WarpBlock *d_warp; int32_t n_warp;   int32_t pad1;
    const B200CompBlock *d_comp; int32_t n_comp;   int32_t pad2;
    const B200CompBlock *d_comp2; int32_t n_comp2; int32_t pad2b;  /* second compound stage: chroma `mask` blocks that
                                                                      consume the mask a luma w_mask of stage 1 produced */
    const B200BlendBlock *d_blend; int32_t n_blend; int32_t pad3;
    const B200ItxBlock *d_itx[B200_N_RECT_TX_SIZES];
    int32_t n_itx[B200_N_RECT_TX_SIZES];
    int32_t pad4;
    void *d_coef;
    int32_t itx_stride[3];       /* picture strides (pixels) for the transform add */
    int32_t run_lf, run_cdef, run_lr;
    B200LfFrame lf;
    B200CdefFrame cdef;
    B200LrFrame lr;
    const B200IntraTx *d_intra;  /* intra transform blocks (run after the inter stages, before the post filters) */
    int32_t n_intra, pad6;
    B200IntraFrame intra;
    const B200McScaledBlock *d_scaled;   /* predictions from scaled references (run with the put / prep stage) */
    int32_t n_scaled, pad7;
    const B200CompFusedBlock *d_cfused;  /* fused compound prediction, stage 1 and stage 2 (stage 2 = blocks that consume */
    const B200CompFusedBlock *d_cfused2; /* a mask emitted by a w_mask block of stage 1) */
    int32_t n_cfused, n_cfused2;
    const B200CoefBlock *d_expand;       /* compact coefficient upload (optional, see b200_coef_expand) */
    int32_t n_expand, pad8;
    const void *d_ccoef;
    uint64_t coef_bytes;
    int32_t run_fg, pad5;        /* film grain on the output copy (fg.in = lr.dst typically); the grain LUT preparation
                                    runs on an internal side stream concurrently with reconstruction */
    B200FgFrame fg;
    const B200BlendBlock *d_blend2;      /* second blend stage, after d_blend: OBMC blends the predictions of the blocks above */
    int32_t n_blend2, pad9;              /* (blend_h, stage 1) and then those of the blocks to the left (blend_v, stage 2) */
    /* super-resolution (reference src/recon_tmpl.c:2053-2086, src/lf_apply_tmpl.c:73-87): after CDEF the frame, coded at a
     * reduced width, is upscaled horizontally; loop restoration (lr.*) then runs on the upscaled pictures. resize[0] upscales the
     * CDEF output (or the deblocked picture when CDEF is off), resize[1] the deblocked picture loop restoration reads its
     * stripe-boundary rows from (n_planes = 0: not needed). */
    int32_t run_resize, pad10;
    B200ResizeFrame resize[2];
} B200FrameJob;
B200_API int b200_frame_run(const B200FrameJob *job, void *stream);
/* n independent jobs of the same bit depth on one stream: reconstruction of every job, then ONE batched intra launch
 * (b200_intra_frames), then every job's post filters. */
B200_API int b200_frame_run_batch(const B200FrameJob *const *jobs, int n_jobs, void *stream);
/* sizeof() of the ABI structs as compiled into the library (binding self-check): 0 McFrame, 1 McBlock, 2 CompBlock,
 * 3 BlendBlock, 4 WarpBlock, 5 ItxBlock, 6 LfFrame, 7 CdefFrame, 8 LrFrame, 9 FrameJob, 10 Av1Filter, 11 Av1Restoration,
 * 12 FgFrame, 13 FilmGrainData, 14 IntraTx, 15 IntraFrame, 16 McScaledBlock, 17 CoefBlock, 18 IntraSb, 19 CompFusedBlock,
 * 20 FrameBand, 21 ResizeFrame */
B200_API int b200_struct_size(int which);

/* ==== band-sliced frame job + cross-GPU reference exchange (SURVEY.md §8e) ===================== */
/* dav1d lets frame n+1 start while frame n is still being decoded: a tile superblock row may run as soon as every
 * reference picture has progressed past the lowest pixel row it reads (check_tile, reference src/thread_task.c:393-436,
 * `lowest_pixel` :415; progress counters src/picture.h:52-63). The device-side counterpart: a frame job is cut into
 * horizontal BANDS (luma rows [y0, y1), multiples of 64 except the bottom of the picture; blocks never straddle a band
 * because bands are superblock aligned). b200_frame_run_band enqueues, for one band,
 *     coefficient expansion / prediction / compound / blends / inverse transforms of the band's records,
 *     deblock of its rows (column edges, then the row edges at y0 .. y1-1),
 *     then the part of CDEF and loop restoration whose inputs that makes final:
 *       CDEF tile rows (32 luma rows) below y1 - 32, loop-restoration tile rows whose stripe ends at or above y1 - 8,
 *     and, for the last band, everything down to the bottom edge + film grain.
 * After band k the restored picture is final down to b200_band_progress(): the rows a dependent frame may predict from.
 * Bands must be run in order, top to bottom, on one stream; the result is bit-identical to b200_frame_run.
 * Intra records (d_intra, per-transform-block schedule) are band-sliced too: band k runs records [intra[0], +intra[1]),
 * a topological order of their dependencies inside the band, after its inter stages. A record may depend on anything in
 * its own band or above, never below: bands fall on superblock rows, and no bottom-left edge or intra-block-copy source
 * reaches below the band's last row (with 128x128 superblocks a band edge inside a superblock can break this; such plans
 * are the caller's to reject). The done map is set up once, by the top band (from intra.done_init, or zeroed). Since the
 * post filters of band k may rewrite its last rows while band k+1 is reconstructed, the reconstruction of band k ends by
 * saving the last row of each plane (luma y1 - 1, chroma (y1 >> ss_ver) - 1; dav1d's f->ipred_edge, reference
 * src/recon_tmpl.c:2111-2135) into edge_bottom, and band k+1's records on its first row read their top edge (top-left,
 * top-right included) from there: its edge_top is band k's edge_bottom. An edge buffer holds the Y, U and V rows back to
 * back, intra.stride[p] samples each; the rows are read at intra.plane_off[p] of intra.pic, which band-sliced jobs with
 * intra records must fill. Both are needed only when the job has intra records: edge_top when y0 > 0 and the band has
 * records, edge_bottom unless the band is the bottom one. Intra block copy reads the picture above directly, which is
 * only valid because such frames run with deblocking, CDEF and loop restoration off. The superblock-granular schedule
 * (intra.sb) runs as a single band only. b200_frame_run_band_phase returns -2, before enqueueing anything, on a band
 * that breaks these rules where it can see it without reading device memory. */
typedef struct B200FrameBand {
    int32_t y0, y1;                 /* luma rows reconstructed by this band */
    int32_t last;                   /* 1: bottom band (y1 = picture height; sweeps run to the bottom edge) */
    int32_t pad;
    /* [first, count) of the job's record arrays that belong to this band */
    int32_t pred[2], warp[2], comp[2], comp2[2], blend[2], blend2[2], scaled[2], cfused[2], cfused2[2], expand[2];
    int32_t itx[B200_N_RECT_TX_SIZES][2];
    int32_t intra[2];               /* [first, count) of d_intra (see below) */
    void *edge_top;                 /* device: the rows above y0 that the band above saved (NULL for the top band) */
    void *edge_bottom;              /* device: where this band saves its last rows (NULL for the bottom band) */
} B200FrameBand;
B200_API int b200_frame_run_band(const B200FrameJob *job, const B200FrameBand *band, void *stream);
/* The two halves of a band for callers that pipeline them on two streams: B200_BAND_RECON = coefficient expansion,
 * prediction, compound, blends, transforms (reads the references, writes the band's rows of the reconstruction);
 * B200_BAND_POST = deblock / CDEF / LR / grain rows (needs RECON of the same band and POST of the previous band). The
 * reconstruction of band k+1 then runs beside the post filters of band k. */
enum { B200_BAND_RECON = 1, B200_BAND_POST = 2 };
B200_API int b200_frame_run_band_phase(const B200FrameJob *job, const B200FrameBand *band, int phases, void *stream);
/* rows of plane `plane` of the restored picture (lr.dst, or cdef.dst / the reconstruction when later stages are off) that
 * are final once the band ending at luma row y1 has run (`last` != 0: the plane height) */
B200_API int b200_band_progress(const B200FrameJob *job, int y1, int last, int plane);

/* Reference pictures cross GPUs as one-sided puts over NVLink peer memory (one process per GPU: the consumer exports
 * its landing buffer with b200_ipc_export, the producer maps it with b200_ipc_open): after a band, the producer copies
 * the rows that became final into each consumer's buffer (b200_copy_async: cudaMemcpyAsync, peer pointers allowed) and
 * then raises that consumer's progress flag (b200_flag_signal, a system-scope store issued behind the copy on the same
 * stream); the consumer's stream waits for the value it needs (b200_flag_wait_geq) before the band that reads those rows.
 * On one GPU the same dependency is a CUDA event (b200_event_*). */
#define B200_IPC_HANDLE_BYTES 64
B200_API int b200_ipc_export(void *dev_ptr, uint8_t handle[B200_IPC_HANDLE_BYTES]);
B200_API void *b200_ipc_open(const uint8_t handle[B200_IPC_HANDLE_BYTES]);
B200_API int b200_ipc_close(void *peer_ptr);
B200_API int b200_copy_async(void *dst, const void *src, size_t bytes, void *stream);
B200_API int b200_flag_signal(uint32_t *flag, uint32_t value, void *stream);           /* flag: device memory, local or peer */
B200_API int b200_flag_wait_geq(const uint32_t *flag, uint32_t value, void *stream);   /* flag: local device memory */
/* One band's whole put in ONE launch: copies up to 3 byte ranges (the rows of the three planes that became final) to up to
 * two destinations each (the landing buffers of the ranks decoding frames n+1 and n+2: peer pointers, stores travel over
 * NVLink) and, when the last CTA has finished, raises those ranks' progress flags behind a system-scope fence. Replaces 6
 * cudaMemcpyAsync + 2 flag kernels per band (~10 us each on the copy engines: the exchange, not the reconstruction, set the
 * pace of a banded frame). `src` and `dst` must have the same alignment modulo 16 bytes. Flag value: add, or
 * ((*base - sub) << shift) + add when base != NULL. `counter`: a zero-initialised device word owned by the caller's stream. */
typedef struct B200PutRange { const void *src; void *dst[2]; uint64_t bytes; } B200PutRange;
typedef struct B200PutFlag { uint32_t *flag; const uint32_t *base; int32_t sub, shift, add, pad; } B200PutFlag;
B200_API int b200_put_rows(const B200PutRange *ranges, int n_ranges, const B200PutFlag *flags, int n_flags,
                           uint32_t *counter, void *stream);
/* The same flag operations with the value taken from device memory when the operation EXECUTES:
 * value = ((*base - sub) << shift) + add. A frame's whole schedule (bands, puts, waits) can then be captured once into a
 * CUDA graph and replayed for every later frame of the set: only the word at `base` (the frame's sequence number) changes. */
B200_API int b200_flag_signal_rel(uint32_t *flag, const uint32_t *base, int32_t sub, int32_t shift, int32_t add, void *stream);
B200_API int b200_flag_wait_geq_rel(const uint32_t *flag, const uint32_t *base, int32_t sub, int32_t shift, int32_t add, void *stream);
/* CUDA graphs for C hosts: everything enqueued on `stream` (and on streams joined to it through events) between begin and
 * end is recorded instead of executed; b200_graph_end returns an executable graph (NULL on failure). */
B200_API int b200_graph_begin(void *stream);
B200_API void *b200_graph_end(void *stream);
B200_API int b200_graph_launch(void *graph_exec, void *stream);
B200_API void b200_graph_destroy(void *graph_exec);
B200_API void *b200_event_create(void);
B200_API void b200_event_destroy(void *event);
B200_API int b200_event_record(void *event, void *stream);
B200_API int b200_stream_wait_event(void *stream, void *event);

/* The same job fed from HOST buffers (the end-to-end path): every (host, dev, bytes) pair of `uploads`
 * is copied host->device first, the job runs, then every pair of `downloads` is copied device->host and
 * the stream is synchronised. Device buffers are the ones the job's pointers refer to. */
typedef struct B200Xfer { void *host; void *dev; uint64_t bytes; } B200Xfer;
B200_API int b200_frame_run_host(const B200FrameJob *job, const B200Xfer *uploads, int n_uploads,
                                 const B200Xfer *downloads, int n_downloads, void *stream);
/* Asynchronous halves of the above, for callers that keep several frames in flight on different streams
 * (the device-side counterpart of dav1d's frame threading, n_fc frame contexts): submit enqueues
 * uploads + job + downloads and returns; wait blocks until everything enqueued on `stream` is done.
 * Host buffers must be page-locked for the copies to overlap other streams' work. */
B200_API int b200_frame_submit_host(const B200FrameJob *job, const B200Xfer *uploads, int n_uploads,
                                    const B200Xfer *downloads, int n_downloads, void *stream);
B200_API int b200_frame_submit_host_batch(const B200FrameJob *const *jobs, int n_jobs, const B200Xfer *uploads,
                                          int n_uploads, const B200Xfer *downloads, int n_downloads, void *stream);
B200_API int b200_frame_wait(void *stream);

#ifdef __cplusplus
}
#endif
#endif /* B200AV1_H */
