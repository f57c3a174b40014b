/*
 * integration/dav1d/stream_driver.c — a minimal dav1d client (what tools/dav1d.c does, without the muxers).
 *
 * Decodes an AV1 elementary stream (a list of temporal units) through dav1d's PUBLIC API only
 * (dav1d_open / dav1d_send_data / dav1d_get_picture, reference include/dav1d/dav1d.h, src/lib.c)
 * and packs every output picture tightly into one buffer. It knows nothing about either back end: it is linked
 * into oracle/_ref/libdav1d_b200.so (dav1d's front end with the B200 back end behind f->bd_fn) and — by
 * oracle/Makefile — into oracle/_ref/libdav1d_ref.so (the stock CPU decoder = the checker), so a test can compare
 * the two byte for byte.
 */
#include <errno.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include "dav1d/dav1d.h"

#define API __attribute__((visibility("default")))

/* when each picture of the last refdrv_decode_stream call came out of dav1d_get_picture, nanoseconds since the call began
 * (what tools/dav1d.c's --frametimes is made of, reference tools/dav1d.c:94-116) */
#define MAX_TIMES 4096
static uint64_t g_out_ns[MAX_TIMES];
static int g_n_out;
static uint64_t now_ns(void) { struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return (uint64_t)ts.tv_sec * 1000000000ull + (uint64_t)ts.tv_nsec; }
API int refdrv_output_times_ns(uint64_t *out, int max)
{
    const int n = g_n_out < max ? g_n_out : max;
    for (int i = 0; i < n; i++) out[i] = g_out_ns[i];
    return n;
}

static void nop_free(const uint8_t *d, void *c) { (void)d; (void)c; }

static size_t pack(const Dav1dPicture *p, uint8_t *out, size_t cap, int32_t *info)
{
    const int px = p->p.bpc > 8 ? 2 : 1;
    const int ssh = p->p.layout != DAV1D_PIXEL_LAYOUT_I444 && p->p.layout != DAV1D_PIXEL_LAYOUT_I400;
    const int ssv = p->p.layout == DAV1D_PIXEL_LAYOUT_I420;
    const int npl = p->p.layout == DAV1D_PIXEL_LAYOUT_I400 ? 1 : 3;
    size_t pos = 0;
    for (int pl = 0; pl < npl; pl++) {
        const int w = pl ? (p->p.w + ssh) >> ssh : p->p.w, h = pl ? (p->p.h + ssv) >> ssv : p->p.h;
        const size_t row = (size_t)w * px;
        if (pos + row * h > cap) return 0;
        for (int y = 0; y < h; y++)
            memcpy(out + pos + row * y, (const uint8_t *)p->data[pl] + (ptrdiff_t)y * p->stride[!!pl], row);
        pos += row * h;
    }
    info[0] = p->p.w; info[1] = p->p.h; info[2] = p->p.bpc; info[3] = (int32_t)p->p.layout;
    return pos;
}

/* tus: n_tu temporal units back to back in `data`, sizes in tu_sz. Returns the number of pictures written
 * (info: 4 ints per picture, out: pictures back to back), or a negative dav1d error. */
API int refdrv_decode_stream(const uint8_t *data, const uint64_t *tu_sz, int n_tu, int n_threads, int max_frame_delay,
                             int apply_grain, uint8_t *out, uint64_t out_cap, int32_t *info, int max_pics)
{
    Dav1dSettings s;
    Dav1dContext *c = NULL;
    dav1d_default_settings(&s);
    s.n_threads = n_threads;
    s.max_frame_delay = max_frame_delay;
    s.apply_grain = apply_grain;
    const uint64_t t_begin = now_ns();
    g_n_out = 0;
    int res = dav1d_open(&c, &s);
    if (res < 0) return res;
    int n_pics = 0;
    size_t pos = 0;
    const uint8_t *ptr = data;
    for (int i = 0; i <= n_tu; i++) {
        Dav1dData d;
        memset(&d, 0, sizeof(d));
        if (i < n_tu) {
            res = dav1d_data_wrap(&d, ptr, (size_t)tu_sz[i], nop_free, NULL);
            if (res < 0) goto done;
            ptr += tu_sz[i];
        }
        do {
            if (i < n_tu && d.sz) {
                res = dav1d_send_data(c, &d);
                if (res < 0 && res != DAV1D_ERR(EAGAIN)) { dav1d_data_unref(&d); goto done; }
            }
            for (int again = 0;;) {
                Dav1dPicture p;
                memset(&p, 0, sizeof(p));
                const int r = dav1d_get_picture(c, &p);
                /* draining (no more data): the first EAGAIN only arms dav1d's drain mode (src/lib.c, c->drain) */
                if (r == DAV1D_ERR(EAGAIN)) { if (i < n_tu || ++again >= 2) break; continue; }
                again = 0;
                if (r < 0) { res = r; if (i < n_tu) dav1d_data_unref(&d); goto done; }
                if (g_n_out < MAX_TIMES) g_out_ns[g_n_out++] = now_ns() - t_begin;
                if (n_pics < max_pics) {
                    const size_t n = pack(&p, out + pos, (size_t)out_cap - pos, info + 4 * n_pics);
                    if (!n) { dav1d_picture_unref(&p); res = DAV1D_ERR(ENOMEM); if (i < n_tu) dav1d_data_unref(&d); goto done; }
                    pos += n; n_pics++;
                }
                dav1d_picture_unref(&p);
            }
        } while (i < n_tu && d.sz);
    }
    res = n_pics;
done:
    dav1d_close(&c);
    return res;
}

/* Sends the first n_tu temporal units and closes the decoder at once, without draining: whatever frames are still
 * being decoded are flushed by dav1d_close (reference src/lib.c, dav1d_flush / close_internal). Test hook for the
 * back end's handling of abandoned frames. Returns the number of pictures that happened to come out. */
API int refdrv_decode_and_abandon(const uint8_t *data, const uint64_t *tu_sz, int n_tu, int n_threads, int max_frame_delay)
{
    Dav1dSettings s;
    Dav1dContext *c = NULL;
    dav1d_default_settings(&s);
    s.n_threads = n_threads;
    s.max_frame_delay = max_frame_delay;
    if (dav1d_open(&c, &s) < 0) return -1;
    int n_pics = 0;
    const uint8_t *ptr = data;
    for (int i = 0; i < n_tu; i++) {
        Dav1dData d;
        memset(&d, 0, sizeof(d));
        if (dav1d_data_wrap(&d, ptr, (size_t)tu_sz[i], nop_free, NULL) < 0) break;
        ptr += tu_sz[i];
        while (d.sz) {
            const int r = dav1d_send_data(c, &d);
            if (r < 0 && r != DAV1D_ERR(EAGAIN)) { dav1d_data_unref(&d); break; }
            Dav1dPicture p;
            memset(&p, 0, sizeof(p));
            if (dav1d_get_picture(c, &p) == 0) { n_pics++; dav1d_picture_unref(&p); }
        }
    }
    dav1d_close(&c);
    return n_pics;
}
