/*
 * integration/dav1d/b200_hooks.c — back-end loading and per-frame-context state for the dav1d record emitters.
 * The back end (dav1d_b200/libb200av1.so) is bound at run time through its C ABI (include/b200av1.h); there is no
 * CPU fallback: without a back end every frame fails with an error.
 */
#include <dlfcn.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "b200_hooks.h"

#include "dav1d/dav1d.h"

#define API __attribute__((visibility("default")))

/* The record emitters run in dav1d's pass 2 (frame_thread.pass == 2: the frame's symbols were decoded in pass 1 and its
 * coefficients sit in frame_thread.cf). dav1d only decodes in two passes with more than one frame context (reference
 * src/thread_task.c:741-744, src/decode.c:2801-2896), and the number of frame contexts is min(max_frame_delay, n_threads)
 * or ceil(sqrt(n_threads)) (src/lib.c). A caller that asks for one thread / no frame delay would get the single-pass mode,
 * which the emitters cannot serve (they would have to run the entropy decoder themselves): open with two threads and two
 * frame contexts instead — same pictures, one frame more of output delay. lib.c's own dav1d_open is renamed by the Makefile. */
int b200real_dav1d_open(Dav1dContext **c_out, const Dav1dSettings *s);
int dav1d_default_picture_alloc(Dav1dPicture *p, void *cookie);       /* src/picture.c: what dav1d_default_settings installs */
static int pinned_pic_alloc(Dav1dPicture *p, void *cookie);
static void pinned_pic_release(Dav1dPicture *p, void *cookie);
static int backend_bound_quietly(void);
API int dav1d_open(Dav1dContext **const c_out, const Dav1dSettings *const s)
{
    if (!s) return b200real_dav1d_open(c_out, s);
    Dav1dSettings s2 = *s;
    if (s2.n_threads == 1) s2.n_threads = 2;
    if (s2.max_frame_delay == 1) s2.max_frame_delay = 2;
    /* output pictures in page-locked memory (a Dav1dPicAllocator, reference include/dav1d/picture.h:107-146), unless the caller
     * brought an allocator of its own: the copy of a finished picture into it is then a true asynchronous copy on the frame's
     * stream, and the worker thread that submitted the job is not held up by it (B200HOOK_PINNED_PICS=0 keeps dav1d's pool) */
    const char *const e = getenv("B200HOOK_PINNED_PICS");
    if (s2.allocator.alloc_picture_callback == dav1d_default_picture_alloc && (!e || atoi(e) != 0) && backend_bound_quietly()) {
        s2.allocator.cookie = NULL;
        s2.allocator.alloc_picture_callback = pinned_pic_alloc;
        s2.allocator.release_picture_callback = pinned_pic_release;
    }
    return b200real_dav1d_open(c_out, &s2);
}

static B200Backend g_be;
static int g_be_ok;
static pthread_mutex_t g_lock = PTHREAD_MUTEX_INITIALIZER;
static HookFrame g_frames[64];
static B200HookStats g_stats;
static uint64_t g_clock;            /* LRU stamps of the frame-context and picture tables */

API void b200hook_release(void);

API int b200hook_set_backend(const char *path)
{
    /* build the table locally, publish it with one release store: a thread that sees g_be_ok set sees every pointer.
     * (Rebinding while frames are in flight is not supported: the old table is simply kept.) */
    B200Backend be;
    memset(&be, 0, sizeof(be));
    void *h = dlopen(path, RTLD_NOW | RTLD_LOCAL);
    if (!h) { fprintf(stderr, "b200hook: cannot load back end %s: %s\n", path, dlerror()); return -1; }
    be.handle = h;
#define SYM(field, name) do { *(void **)&be.field = dlsym(h, name); \
        if (!be.field) { fprintf(stderr, "b200hook: back end lacks %s\n", name); dlclose(h); return -1; } } while (0)
    SYM(last_error, "b200_last_error");
    SYM(dev_alloc, "b200_dev_alloc"); SYM(dev_free, "b200_dev_free");
    SYM(host_alloc, "b200_host_alloc"); SYM(host_free, "b200_host_free");
    SYM(stream_create, "b200_stream_create"); SYM(stream_destroy, "b200_stream_destroy");
    SYM(intra_scratch_bytes, "b200_intra_scratch_bytes");
    SYM(frame_run_host, "b200_frame_run_host");
    SYM(frame_submit_host, "b200_frame_submit_host"); SYM(frame_wait, "b200_frame_wait"); SYM(copy_async, "b200_copy_async");
    SYM(event_create, "b200_event_create"); SYM(event_destroy, "b200_event_destroy");
    SYM(event_record, "b200_event_record"); SYM(stream_wait_event, "b200_stream_wait_event");
    SYM(struct_size, "b200_struct_size");
#undef SYM
    /* binding self-check: the structs this file was compiled with are the ones the library was compiled with */
    if (be.struct_size(9) != (int)sizeof(B200FrameJob) || be.struct_size(14) != (int)sizeof(B200IntraTx) ||
        be.struct_size(10) != (int)sizeof(B200Av1Filter) || be.struct_size(11) != (int)sizeof(B200Av1Restoration)) {
        fprintf(stderr, "b200hook: ABI struct size mismatch with %s\n", path);
        dlclose(h);
        return -1;
    }
    /* the frame slots' buffers and streams belong to the back end that allocated them: free them through it first */
    if (__atomic_load_n(&g_be_ok, __ATOMIC_ACQUIRE)) b200hook_release();
    pthread_mutex_lock(&g_lock);
    g_be = be;
    __atomic_store_n(&g_be_ok, 1, __ATOMIC_RELEASE);
    pthread_mutex_unlock(&g_lock);
    return 0;
}

/* Device jobs of different frame contexts normally overlap (one stream each). A back end that is not re-entrant
 * (the host emulator the CPU tests bind) asks for one job at a time. */
static int g_serialize;
static pthread_mutex_t g_job_lock = PTHREAD_MUTEX_INITIALIZER;
API void b200hook_set_serialize(int on) { g_serialize = on; }
void b200hook_job_enter(void) { if (g_serialize) pthread_mutex_lock(&g_job_lock); }
void b200hook_job_leave(void) { if (g_serialize) pthread_mutex_unlock(&g_job_lock); }

static int backend_bound_quietly(void)
{
    if (__atomic_load_n(&g_be_ok, __ATOMIC_ACQUIRE)) return 1;
    const char *env = getenv("B200AV1_LIB");
    return env && b200hook_backend() != NULL;
}

/* ---- page-locked output pictures -------------------------------------------------------------------------------------
 * Same layout as dav1d_default_picture_alloc (reference src/picture.c:46-78: planes back to back in one allocation, 128-sample
 * aligned dimensions, 64 bytes more when a stride would be a multiple of 1024) — pic_geom() of the emitters derives the
 * device picture from the host strides. Buffers come from a pool (cudaHostAlloc costs about a millisecond); released
 * pictures go back to it, b200hook_release() frees the idle ones. */
#define PIN_POOL 1024
static struct { void *ptr; size_t cap; int used; } g_pin_pool[PIN_POOL];
static pthread_mutex_t g_pin_lock = PTHREAD_MUTEX_INITIALIZER;
static int pinned_pic_alloc(Dav1dPicture *const p, void *const cookie)
{
    (void)cookie;
    const B200Backend *const be = b200hook_backend();
    if (!be) return -12;
    const int hbd = p->p.bpc > 8;
    const int aligned_w = (p->p.w + 127) & ~127, aligned_h = (p->p.h + 127) & ~127;
    const int has_chroma = p->p.layout != DAV1D_PIXEL_LAYOUT_I400;
    const int ss_ver = p->p.layout == DAV1D_PIXEL_LAYOUT_I420, ss_hor = p->p.layout != DAV1D_PIXEL_LAYOUT_I444;
    ptrdiff_t y_stride = (ptrdiff_t)aligned_w << hbd;
    ptrdiff_t uv_stride = has_chroma ? y_stride >> ss_hor : 0;
    if (!(y_stride & 1023)) y_stride += DAV1D_PICTURE_ALIGNMENT;
    if (!(uv_stride & 1023) && has_chroma) uv_stride += DAV1D_PICTURE_ALIGNMENT;
    const size_t y_sz = (size_t)y_stride * aligned_h, uv_sz = (size_t)uv_stride * (aligned_h >> ss_ver);
    const size_t need = y_sz + 2 * uv_sz + DAV1D_PICTURE_ALIGNMENT;
    int slot = -1, empty = -1;
    pthread_mutex_lock(&g_pin_lock);
    for (int i = 0; i < PIN_POOL; i++) {
        if (!g_pin_pool[i].ptr) { if (empty < 0) empty = i; continue; }
        if (!g_pin_pool[i].used && g_pin_pool[i].cap >= need && (slot < 0 || g_pin_pool[i].cap < g_pin_pool[slot].cap)) slot = i;
    }
    if (slot < 0 && empty < 0)                      /* pool full of buffers that are too small: drop an idle one */
        for (int i = 0; i < PIN_POOL && empty < 0; i++)
            if (!g_pin_pool[i].used) { be->host_free(g_pin_pool[i].ptr); g_pin_pool[i].ptr = NULL; empty = i; }
    if (slot < 0 && empty >= 0) {
        void *const mem = be->host_alloc(need);
        if (mem) { g_pin_pool[empty].ptr = mem; g_pin_pool[empty].cap = need; slot = empty; }
    }
    if (slot >= 0) g_pin_pool[slot].used = 1;
    pthread_mutex_unlock(&g_pin_lock);
    if (slot < 0) { fprintf(stderr, "b200hook: no page-locked memory for a picture: %s\n", be->last_error()); return -12; }
    uint8_t *const buf = g_pin_pool[slot].ptr;
    p->stride[0] = y_stride; p->stride[1] = uv_stride;
    p->allocator_data = (void *)(intptr_t)(slot + 1);
    p->data[0] = buf;
    p->data[1] = has_chroma ? buf + y_sz : NULL;
    p->data[2] = has_chroma ? buf + y_sz + uv_sz : NULL;
    return 0;
}
void b200hook_refpic_forget(const void *key);
static void pinned_pic_release(Dav1dPicture *const p, void *const cookie)
{
    (void)cookie;
    const int slot = (int)(intptr_t)p->allocator_data - 1;
    if (slot < 0 || slot >= PIN_POOL) return;
    /* dav1d dropped its last reference to the picture: nothing decodes from it or outputs it any more, so its device copy's
     * table entry is free for the next picture (its device buffer is kept for reuse). With dav1d's own allocator there is no
     * such signal and the table falls back to least-recently-used recycling. */
    b200hook_refpic_forget(p->data[0]);
    pthread_mutex_lock(&g_pin_lock);
    g_pin_pool[slot].used = 0;
    pthread_mutex_unlock(&g_pin_lock);
}
static void pinned_pool_trim(void)
{
    pthread_mutex_lock(&g_pin_lock);
    for (int i = 0; i < PIN_POOL; i++)
        if (g_pin_pool[i].ptr && !g_pin_pool[i].used && g_be_ok) { g_be.host_free(g_pin_pool[i].ptr); g_pin_pool[i].ptr = NULL; g_pin_pool[i].cap = 0; }
    pthread_mutex_unlock(&g_pin_lock);
}

const B200Backend *b200hook_backend(void)
{
    if (!__atomic_load_n(&g_be_ok, __ATOMIC_ACQUIRE)) {
        /* lazy binding from the environment, once: concurrent first calls serialise here and the losers find it bound */
        static pthread_mutex_t once = PTHREAD_MUTEX_INITIALIZER;
        pthread_mutex_lock(&once);
        int ok = __atomic_load_n(&g_be_ok, __ATOMIC_ACQUIRE);
        if (!ok) {
            const char *env = getenv("B200AV1_LIB");
            ok = env && !b200hook_set_backend(env);
        }
        pthread_mutex_unlock(&once);
        if (!ok) {
            fprintf(stderr, "b200hook: no back end loaded (b200hook_set_backend / B200AV1_LIB) - frame fails\n");
            return NULL;
        }
    }
    return &g_be;
}

int b200hook_buf_reserve(HookBuf *b, size_t bytes, int need_host, int keep)
{
    const B200Backend *be = b200hook_backend();
    if (!be) return -1;
    if (bytes <= b->cap && b->dev && (!need_host || b->host)) return 0;
    size_t cap = b->cap ? b->cap : 4096;
    while (cap < bytes) cap *= 2;
    void *host = NULL, *dev = be->dev_alloc(cap);
    if (!dev) { fprintf(stderr, "b200hook: %s\n", be->last_error()); return -1; }
    if (need_host) {
        host = be->host_alloc(cap);
        if (!host) { fprintf(stderr, "b200hook: %s\n", be->last_error()); be->dev_free(dev); return -1; }
        if (keep && b->host) memcpy(host, b->host, b->cap);
    }
    if (b->host) be->host_free(b->host);
    if (b->dev) be->dev_free(b->dev);
    b->host = host; b->dev = dev; b->cap = cap;
    return 0;
}

void b200hook_buf_free(HookBuf *b)
{
    if (g_be_ok) { if (b->host) g_be.host_free(b->host); if (b->dev) g_be.dev_free(b->dev); }
    memset(b, 0, sizeof(*b));
}

void *b200hook_append(HookBuf *b, int *n, size_t elem)
{
    if (b200hook_buf_reserve(b, (size_t)(*n + 1) * elem, 1, 1)) return NULL;
    void *const p = (uint8_t *)b->host + (size_t)(*n)++ * elem;
    memset(p, 0, elem);
    return p;
}

int b200hook_tiles_reset(HookFrame *const hf, const int n_tiles)
{
    if (n_tiles > hf->cap_tiles) {
        HookTile *const nt = realloc(hf->tiles, (size_t)n_tiles * sizeof(*nt));
        if (!nt) return -1;
        memset(nt + hf->cap_tiles, 0, (size_t)(n_tiles - hf->cap_tiles) * sizeof(*nt));
        hf->tiles = nt; hf->cap_tiles = n_tiles;
    }
    hf->n_tiles = n_tiles;
    for (int t = 0; t < hf->cap_tiles; t++)
        for (int l = 0; l < B200L_COUNT; l++) hf->tiles[t].l[l].n = 0;
    return 0;
}
void *b200hook_tile_grow(HookList *const L, const size_t elem)
{
    const int cap = L->cap ? 2 * L->cap : 256;
    uint8_t *const d = realloc(L->data, (size_t)cap * elem);
    if (!d) return NULL;
    L->data = d; L->cap = cap;
    return d;
}
int b200hook_tiles_gather(HookFrame *const hf, const int list, HookBuf *const dst, const size_t elem)
{
    size_t total = 0;
    for (int t = 0; t < hf->n_tiles; t++) total += (size_t)hf->tiles[t].l[list].n;
    if (b200hook_buf_reserve(dst, (total ? total : 1) * elem, 1, 0)) return -1;
    uint8_t *o = dst->host;
    for (int t = 0; t < hf->n_tiles; t++) {
        const HookList *const L = &hf->tiles[t].l[list];
        if (L->n) memcpy(o, L->data, (size_t)L->n * elem);
        o += (size_t)L->n * elem;
    }
    return (int)total;
}

static HookRefPic g_refs[64];
static pthread_cond_t g_ref_cond = PTHREAD_COND_INITIALIZER;
HookRefPic *b200hook_refpic(const void *key, size_t bytes, int create)
{
    const B200Backend *be = b200hook_backend();
    HookRefPic *r = NULL;
    if (!be || !key) return NULL;
    pthread_mutex_lock(&g_lock);
    for (int i = 0; i < 64 && !r; i++)
        if (g_refs[i].key == key) r = &g_refs[i];
    if (!r && create) {
        /* a free entry: one whose device buffer is already large enough if there is one (the buffer and event of a forgotten
         * picture stay with its entry) */
        for (int i = 0; i < 64; i++)
            if (!g_refs[i].key && (!r || (r->bytes < bytes && g_refs[i].bytes >= bytes))) r = &g_refs[i];
        if (r) { r->key = key; r->ready = 0; r->submitted = 0; }
        if (!r) {
            /* host pictures of closed decoders never come back: recycle the least recently used entry (the live set —
             * 8 reference slots + frames in flight + pictures waiting for output — is far smaller than the table) */
            for (int i = 0; i < 64; i++)
                if (g_refs[i].ready && (!r || g_refs[i].last_use < r->last_use)) r = &g_refs[i];
            if (!r)                              /* only pictures of abandoned frames (never completed) are left: oldest one */
                for (int i = 0; i < 64; i++)
                    if (!r || g_refs[i].last_use < r->last_use) r = &g_refs[i];
            r->key = key; r->ready = 0; r->submitted = 0;
        }
    }
    if (r && create && !r->event) r->event = be->event_create();      /* NULL = no events: consumers then wait for `ready` on the host */
    if (r) r->last_use = ++g_clock;
    if (r && create && r->bytes < bytes) {
        if (r->dev) be->dev_free(r->dev);
        r->dev = be->dev_alloc(bytes);
        r->bytes = r->dev ? bytes : 0;
        if (!r->dev) { fprintf(stderr, "b200hook: %s\n", be->last_error()); r->key = NULL; r = NULL; }
    }
    pthread_mutex_unlock(&g_lock);
    return r;
}
void b200hook_refpic_forget(const void *const key)
{
    if (!key) return;
    pthread_mutex_lock(&g_lock);
    for (int i = 0; i < 64; i++)
        if (g_refs[i].key == key) { g_refs[i].key = NULL; g_refs[i].ready = 0; g_refs[i].submitted = 0; }
    pthread_mutex_unlock(&g_lock);
}
void b200hook_refpic_set_ready(HookRefPic *r, int ready)
{
    pthread_mutex_lock(&g_lock);
    r->ready = ready;
    if (ready) r->submitted = 1;                /* nobody may wait for ever, whatever happened to the job */
    pthread_cond_broadcast(&g_ref_cond);
    pthread_mutex_unlock(&g_lock);
}
void b200hook_refpic_set_submitted(HookRefPic *r, int submitted)
{
    pthread_mutex_lock(&g_lock);
    r->submitted = submitted;
    pthread_cond_broadcast(&g_ref_cond);
    pthread_mutex_unlock(&g_lock);
}
void b200hook_refpic_wait_submitted(HookRefPic *r)
{
    pthread_mutex_lock(&g_lock);
    while (!r->submitted && !r->ready) pthread_cond_wait(&g_ref_cond, &g_lock);
    pthread_mutex_unlock(&g_lock);
}
int b200hook_async(void)
{
    static int v = -1;
    if (v < 0) { const char *e = getenv("B200HOOK_ASYNC"); v = !e || atoi(e) != 0; }
    return v;
}
void b200hook_refpic_wait(HookRefPic *r)
{
    pthread_mutex_lock(&g_lock);
    while (!r->ready) pthread_cond_wait(&g_ref_cond, &g_lock);
    pthread_mutex_unlock(&g_lock);
}

/* Frame contexts come and go with dav1d_open / dav1d_close (there is no hook for either): a context that is not in the
 * table takes over the least recently used idle slot, together with that slot's buffers. */
/* a thread's cached slot: the slot's `users` count says how many threads may take the lock-free path to it; the count is
 * released when the thread caches another slot or exits (pthread key destructor) */
static pthread_key_t g_tls_key;
static pthread_once_t g_tls_once = PTHREAD_ONCE_INIT;
static unsigned g_epoch;            /* bumped by b200hook_release: references taken before it are void */
static void tls_release(void *p)
{
    HookFrame *const h = p;
    if (!h) return;
    pthread_mutex_lock(&g_lock);
    if (h->users > 0 && h->epoch == g_epoch) h->users--;
    pthread_mutex_unlock(&g_lock);
}
static void tls_init(void) { pthread_key_create(&g_tls_key, tls_release); }

HookFrame *b200hook_frame(const void *key)
{
    /* called by every hook, i.e. once per block: the thread's last answer is still right as long as this thread holds a
     * `users` reference on the slot (a slot somebody caches is never handed to another key), so the table lock is taken
     * once per frame and thread, not per block */
    static __thread const void *tl_key;
    static __thread HookFrame *tl_slot;
    static __thread unsigned tl_epoch;
    if (tl_key == key && tl_slot && tl_epoch == __atomic_load_n(&g_epoch, __ATOMIC_ACQUIRE) &&
        __atomic_load_n(&tl_slot->key, __ATOMIC_ACQUIRE) == key) {
        return tl_slot;       /* no write here (it would be one store per block and thread to a line all tile threads read): a slot
                                 somebody caches (`users`) is never taken over, its LRU stamp is refreshed by the slow path */
    }
    pthread_once(&g_tls_once, tls_init);
    HookFrame *r = NULL, *lru = NULL;
    pthread_mutex_lock(&g_lock);
    if (tl_slot) {
        if (tl_epoch == g_epoch && tl_slot->users > 0) tl_slot->users--;
        tl_slot = NULL; tl_key = NULL; pthread_setspecific(g_tls_key, NULL);
    }
    for (int i = 0; i < 64 && !r; i++)
        if (g_frames[i].key == key) r = &g_frames[i];
    for (int i = 0; i < 64 && !r; i++)
        if (!g_frames[i].key) {
            r = &g_frames[i];
            memset(r, 0, sizeof(*r));
            pthread_mutex_init(&r->lock, NULL);
            r->key = key;
        }
    /* table full: take over the least recently used slot — idle ones first (pass 0), then leftovers of decoders that were
     * closed in the middle of a frame (pass 1: live contexts are looked up all the time, so an old busy-looking slot is dead).
     * A slot whose lock is held (its job or its exit handler is running) is skipped. */
    for (int pass = 0; pass < 2 && !r; pass++) {
        uint64_t floor_use = 0;
        for (int tries = 0; tries < 64 && !r; tries++) {
            for (int i = 0; i < 64; i++) {
                HookFrame *const h = &g_frames[i];
                if (h->pinned || h->users || h->pending || h->last_use <= floor_use) continue;      /* pending: its job still uses the buffers */
                if (!pass && (h->started || h->tile_sbrows_done)) continue;
                if (!lru || h->last_use < lru->last_use) lru = h;
            }
            if (!lru) break;
            if (pthread_mutex_trylock(&lru->lock) == 0) {
                lru->started = 0; lru->tile_sbrows_done = 0; lru->cur_pic = NULL;
                lru->key = key; lru->unsupported = 0; r = lru;
                pthread_mutex_unlock(&lru->lock);
            } else {
                floor_use = lru->last_use; lru = NULL;          /* busy right now: next oldest */
            }
        }
    }
    if (!r) fprintf(stderr, "b200hook: no frame-context slot available\n");
    if (r) { r->last_use = ++g_clock; r->users++; r->epoch = g_epoch; pthread_setspecific(g_tls_key, r); }
    tl_epoch = g_epoch;
    pthread_mutex_unlock(&g_lock);
    tl_key = r ? key : NULL; tl_slot = r;
    return r;
}

/* Wavefront order for the device's dataflow kernel (dav1d_b200/csrc/intra.cu): records arrive in decode order, where a
 * window of consecutive records spans only a couple of superblocks; sorted by dependency depth ("wave": 1 + the
 * deepest record among the cells whose pixels the block's edge array reads, the same cells the kernel polls) a window
 * of consecutive tickets spans a whole anti-diagonal of the frame. Stable counting sort: any order in which every
 * record follows its dependencies is valid for the kernel. Returns the number of waves, < 0 on allocation failure. */
static const uint8_t k_tx_w4[19] = { 1, 2, 4, 8, 16, 1, 2, 2, 4, 4, 8, 8, 16, 1, 4, 2, 8, 4, 16 };
static const uint8_t k_tx_h4[19] = { 1, 2, 4, 8, 16, 2, 1, 4, 2, 8, 4, 16, 8, 4, 1, 8, 2, 16, 4 };
static inline int mini(int a, int b) { return a < b ? a : b; }
int b200hook_wave_sort(const B200IntraTx *in, B200IntraTx *out, int n, const int32_t w4[3], const int32_t h4[3],
                       int ss_hor, int ss_ver, void **scratch, size_t *scratch_cap)
{
    size_t cells = 0, off[3];
    for (int p = 0; p < 3; p++) { off[p] = cells; cells += (size_t)w4[p] * h4[p]; }
    /* the cell map (several MB at 4K) and the wave numbers live in a buffer the frame context keeps: a fresh calloc per
     * frame cost more in page faults than the sort itself */
    const size_t need = (cells + (size_t)n + 1) * sizeof(int32_t);
    if (*scratch_cap < need) {
        free(*scratch);
        *scratch = malloc(need + need / 4);
        *scratch_cap = *scratch ? need + need / 4 : 0;
        if (!*scratch) return -1;
    }
    int32_t *const map = *scratch, *const wave = map + cells;
    memset(map, 0, cells * sizeof(*map));
    int n_waves = 0;
    for (int i = 0; i < n; i++) {
        const B200IntraTx *const r = &in[i];
        const int pl = r->plane, mw = w4[pl], mh = h4[pl];
        int32_t *const m = map + off[pl];
        const int x = r->x4, y = r->y4, tw = k_tx_w4[r->tx], th = k_tx_h4[r->tx], xe = r->xend4, ye = r->yend4;
        const int hl = r->flags & B200_INTRA_HAVE_LEFT, ht = r->flags & B200_INTRA_HAVE_TOP;
        int dep = 0;
        if (r->mode == B200_INTRA_MODE_IBC) {             /* waits for every cell its source rectangle touches */
            const int sx = r->luma_off & 0xffff, sy = r->luma_off >> 16;
            const int x1 = mini((sx + tw * 4 - 1 + (r->cfl_w_pad != 0)) >> 2, mw - 1), y1 = mini((sy + th * 4 - 1 + (r->cfl_h_pad != 0)) >> 2, mh - 1);
            for (int yy = mini(sy >> 2, mh - 1); yy <= y1; yy++)
                for (int xx = mini(sx >> 2, mw - 1); xx <= x1; xx++) { const int v = m[(size_t)yy * mw + xx]; if (v > dep) dep = v; }
        } else if (r->mode == B200_INTRA_MODE_RESID) {    /* waits for the inter-intra record that covers it */
            for (int yy = y; yy < y + th && yy < mh; yy++)
                for (int xx = x; xx < x + tw && xx < mw; xx++) { const int v = m[(size_t)yy * mw + xx]; if (v > dep) dep = v; }
        } else if (hl) {
            int rows = mini(th, ye - y);
            if ((r->flags & B200_INTRA_LEFT_HAS_BOTTOM) && y + th < ye) rows += mini(th, ye - y - th);
            for (int k = 0; k < rows && y + k < mh; k++) { const int v = m[(size_t)(y + k) * mw + x - 1]; if (v > dep) dep = v; }
        }
        if (ht && r->mode != B200_INTRA_MODE_RESID) {
            int cols = mini(tw, xe - x);
            if ((r->flags & B200_INTRA_TOP_HAS_RIGHT) && x + tw < xe) cols += mini(tw, xe - x - tw);
            for (int k = 0; k < cols && x + k < mw; k++) { const int v = m[(size_t)(y - 1) * mw + x + k]; if (v > dep) dep = v; }
        }
        if (hl && ht && r->mode != B200_INTRA_MODE_RESID) { const int v = m[(size_t)(y - 1) * mw + x - 1]; if (v > dep) dep = v; }
        if (r->mode == B200_INTRA_MODE_CFL && r->cfl_alpha) {
            const int lx = x << ss_hor, ly = y << ss_ver;
            const int lw = mini((tw - r->cfl_w_pad) << ss_hor, w4[0] - lx), lh = mini((th - r->cfl_h_pad) << ss_ver, h4[0] - ly);
            for (int yy = 0; yy < lh; yy++)
                for (int xx = 0; xx < lw; xx++) { const int v = map[(size_t)(ly + yy) * w4[0] + lx + xx]; if (v > dep) dep = v; }
        }
        const int wv = dep + 1;
        wave[i] = wv;
        if (wv > n_waves) n_waves = wv;
        for (int yy = y; yy < y + th && yy < mh; yy++)
            for (int xx = x; xx < x + tw && xx < mw; xx++) m[(size_t)yy * mw + xx] = wv;
    }
    int32_t *const start = calloc((size_t)n_waves + 2, sizeof(*start));
    if (!start) return -1;
    for (int i = 0; i < n; i++) start[wave[i] + 1]++;
    for (int k = 1; k <= n_waves + 1; k++) start[k] += start[k - 1];
    for (int i = 0; i < n; i++) out[start[wave[i]]++] = in[i];
    free(start);
    return n_waves;
}

/* dav1d's "this frame is over" (completed, failed or flushed; reference src/decode.c:3242, called from src/thread_task.c and
 * src/lib.c:588, which are compiled with the call renamed to this wrapper). A frame that ends without having been handed to
 * the device leaves half a frame of records in its slot: drop them, and release anybody waiting for its picture. */
#include <time.h>
static double now_ms(void) { struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6; }

/* The frame's job was enqueued when its last tile superblock row had been emitted (run_frame); here — in the frame's exit
 * handler, the last thing dav1d does before the picture may be output or the context reused — the host waits for it.
 * In between, later frames have ordered their jobs behind this one on the device (event) without any host-side wait.
 * Called with h->lock held. */
int b200hook_frame_finish(HookFrame *const h)
{
    if (!h->pending) return 0;
    const B200Backend *const be = b200hook_backend();
    int r = be ? be->frame_wait(h->stream) : -1;
    if (r) fprintf(stderr, "b200hook: device job failed (%d): %s\n", r, be ? be->last_error() : "no back end");
    b200hook_account(h->pend_rec, h->pend_coef, h->pend_h2d, h->pend_d2h, now_ms() - h->t_submit, h->pend_kinds, h->pend_prep_ms);
    if (h->pending_out) b200hook_refpic_set_ready(h->pending_out, 1);
    h->pending = 0; h->pending_out = NULL;
    return r;
}

struct Dav1dFrameContext;
void dav1d_decode_frame_exit(struct Dav1dFrameContext *f, int retval);
void b200hook_decode_frame_exit(struct Dav1dFrameContext *const f, int retval)
{
    HookFrame *h = NULL;
    pthread_mutex_lock(&g_lock);
    for (int i = 0; i < 64 && !h; i++)
        if (g_frames[i].key == (const void *)f) h = &g_frames[i];
    pthread_mutex_unlock(&g_lock);
    if (h) {
        pthread_mutex_lock(&h->lock);
        if (b200hook_frame_finish(h) && !retval) retval = -22;      /* DAV1D_ERR(EINVAL): the frame is reported as a decoding error */
        if (h->started) {
            HookRefPic *const out = h->cur_pic ? b200hook_refpic(h->cur_pic, 0, 0) : NULL;
            if (out) b200hook_refpic_set_ready(out, 1);
            h->started = 0; h->tile_sbrows_done = 0; h->n_tx = 0; h->n_coef = 0; h->unsupported = 0;
            h->n_pred = h->n_comp = h->n_comp2 = h->n_warp = h->n_blend = h->n_blend2 = 0;
            h->n_tmp16 = 0; h->n_pxtmp = 0; h->is_inter = 0; h->n_ii = 0; h->n_ibc = 0; h->n_pal = 0; h->refs_used = 0;
            memset(h->n_itx, 0, sizeof(h->n_itx));
        }
        pthread_mutex_unlock(&h->lock);
    }
    dav1d_decode_frame_exit(f, retval);
}

void b200hook_account(uint64_t records, uint64_t coefs, uint64_t h2d, uint64_t d2h, double ms, const uint64_t kinds[11], double prep_ms)
{
    pthread_mutex_lock(&g_lock);
    g_stats.frames++; g_stats.records += records; g_stats.coefs += coefs;
    g_stats.h2d_bytes += h2d; g_stats.d2h_bytes += d2h; g_stats.device_ms += ms;
    g_stats.intra_tx += kinds[0]; g_stats.pred += kinds[1]; g_stats.comp += kinds[2]; g_stats.warp += kinds[3];
    g_stats.host_prep_ms += prep_ms; g_stats.interintra += kinds[7]; g_stats.palette_bytes += kinds[8]; g_stats.ibc += kinds[9]; g_stats.scaled += kinds[10];
    g_stats.blend += kinds[4]; g_stats.itx += kinds[5]; g_stats.inter_frames += kinds[6];
    pthread_mutex_unlock(&g_lock);
}

API void b200hook_get_stats(B200HookStats *out, int reset)
{
    pthread_mutex_lock(&g_lock);
    *out = g_stats;
    if (reset) memset(&g_stats, 0, sizeof(g_stats));
    pthread_mutex_unlock(&g_lock);
}

/* frees every per-frame-context buffer (call after dav1d_close) */
API void b200hook_release(void)
{
    pthread_mutex_lock(&g_lock);
    __atomic_add_fetch(&g_epoch, 1, __ATOMIC_RELEASE);
    for (int i = 0; i < 64; i++) {
        HookFrame *h = &g_frames[i];
        if (!h->key) continue;
        if (h->pending && h->stream && g_be_ok) g_be.frame_wait(h->stream);       /* nothing may still read the buffers below */
        b200hook_buf_free(&h->tx); b200hook_buf_free(&h->tx_sorted); b200hook_buf_free(&h->coef); b200hook_buf_free(&h->mask);
        b200hook_buf_free(&h->level); b200hook_buf_free(&h->lr_mask); b200hook_buf_free(&h->scratch);
        for (int p = 0; p < 3; p++) b200hook_buf_free(&h->pic[p]);
        b200hook_buf_free(&h->pred); b200hook_buf_free(&h->comp); b200hook_buf_free(&h->comp2);
        for (int t = 0; t < 19; t++) b200hook_buf_free(&h->itx[t]);
        b200hook_buf_free(&h->tmp16); b200hook_buf_free(&h->cmask); b200hook_buf_free(&h->done_init);
        b200hook_buf_free(&h->pal);
        b200hook_buf_free(&h->warp); b200hook_buf_free(&h->blend); b200hook_buf_free(&h->blend2); b200hook_buf_free(&h->pxtmp);
        b200hook_buf_free(&h->scaled); b200hook_buf_free(&h->sr[0]); b200hook_buf_free(&h->sr[1]);
        if (h->stream && g_be_ok) g_be.stream_destroy(h->stream);
        for (int t = 0; t < h->cap_tiles; t++)
            for (int l = 0; l < B200L_COUNT; l++) free(h->tiles[t].l[l].data);
        free(h->tiles);
        free(h->sort_scratch);
        pthread_mutex_destroy(&h->lock);
        memset(h, 0, sizeof(*h));
    }
    for (int i = 0; i < 64; i++) {
        if (g_refs[i].dev && g_be_ok) g_be.dev_free(g_refs[i].dev);
        if (g_refs[i].event && g_be_ok) g_be.event_destroy(g_refs[i].event);
        memset(&g_refs[i], 0, sizeof(g_refs[i]));
    }
    pthread_mutex_unlock(&g_lock);
    pinned_pool_trim();
}
