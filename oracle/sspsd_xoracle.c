/* sspsd_xoracle.c -- CPU restatement of the cross-spectral density of two streams (TEST INFRASTRUCTURE ONLY).
 *
 * The reference has no CSD.  The restatement is Psd::process (psd.rs:196-269) run over x and y in lockstep with
 * |c|^2 (psd.rs:228-233) replaced by conj(cx) cy for the cross row, chained like PsdCascade::process (psd.rs:456-468)
 * and merged like PsdCascade::psd (psd.rs:479-543).  Built on the public API of sspsd_oracle.c (window, detrend,
 * FFT, half-band decimator) and linked with it into its own shared object (oracle/xbinding.py).  Each channel is
 * transformed on its own with orc_fft_forward -- deliberately not the device's two-for-one split -- and the rows
 * accumulate g s + (xr xr + xi xi), g s + (yr yr + yi yi), g s + (xr yr + xi yi) and g s + (xr yi - xi yr) in f32,
 * unfused (-ffp-contract=off), so the x row is bit-equal to orc_cascade's PSD of x.
 */
#include <assert.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "sspsd_oracle.h"

#define XORC_MAX_STAGES 24

typedef struct {
    float *bx, *by;      /* N-sample segment buffers */
    size_t idx;
    float *sxx, *syy;    /* N/2+1 */
    float *sxy;          /* N/2+1 (re, im) pairs */
    uint32_t count, avg;
    size_t drain;
    orc_hbf8 *hx, *hy;
} xstage;

typedef struct orc_xcascade {
    int n, window, hbf;
    float *win;
    float power, nenbw;
    size_t overlap;
    int detrend;
    uint32_t avg_limit, avg_count;
    xstage *st[XORC_MAX_STAGES];
    size_t ns;
    float *zx, *zy;                  /* 2N floats: interleaved complex FFT input / output */
    float *ax[2], *ay[2];            /* 2N floats: ping-pong outputs of the stages (orc_cascade_new's comment) */
} orc_xcascade;

orc_xcascade *orc_xcascade_new(int n, int window, int hbf_preset);
void orc_xcascade_free(orc_xcascade *c);
void orc_xcascade_set_avg(orc_xcascade *c, uint32_t limit, uint32_t count);
void orc_xcascade_set_detrend(orc_xcascade *c, int detrend);
void orc_xcascade_process(orc_xcascade *c, const float *x, const float *y, size_t n);
size_t orc_xcascade_num_stages(const orc_xcascade *c);
size_t orc_xcascade_csd(const orc_xcascade *c, int keep_overlap, uint32_t min_count, int keep_transition_band,
                        float *pxx, float *pyy, float *pxy, orc_break *b, size_t *nb);

orc_xcascade *orc_xcascade_new(int n, int window, int hbf_preset)
{
    if (n < 16 || (n & (n - 1)) != 0 || (window != ORC_WINDOW_RECT && window != ORC_WINDOW_HANN))
        return NULL;
    orc_hbf8 *probe = orc_hbf8_new(hbf_preset);
    if (!probe)
        return NULL;
    orc_hbf8_free(probe);
    orc_xcascade *c = (orc_xcascade *)calloc(1, sizeof(*c));
    c->n = n;
    c->window = window;
    c->hbf = hbf_preset;
    c->win = (float *)calloc((size_t)n, sizeof(float));
    orc_window(n, window, c->win, &c->power, &c->nenbw, &c->overlap);
    c->detrend = ORC_DETREND_NONE;
    c->avg_limit = UINT32_MAX;
    c->avg_count = UINT32_MAX;
    c->zx = (float *)calloc(2 * (size_t)n, sizeof(float));
    c->zy = (float *)calloc(2 * (size_t)n, sizeof(float));
    for (int i = 0; i < 2; i++) {
        c->ax[i] = (float *)calloc(2 * (size_t)n, sizeof(float));
        c->ay[i] = (float *)calloc(2 * (size_t)n, sizeof(float));
    }
    return c;
}

static void xstage_free(xstage *s)
{
    free(s->bx);
    free(s->by);
    free(s->sxx);
    free(s->syy);
    free(s->sxy);
    orc_hbf8_free(s->hx);
    orc_hbf8_free(s->hy);
    free(s);
}

void orc_xcascade_free(orc_xcascade *c)
{
    if (!c)
        return;
    for (size_t i = 0; i < c->ns; i++)
        xstage_free(c->st[i]);
    free(c->win);
    free(c->zx);
    free(c->zy);
    for (int i = 0; i < 2; i++) {
        free(c->ax[i]);
        free(c->ay[i]);
    }
    free(c);
}

/* (avg.count >> (DEPTH * i)).min(avg.limit), psd.rs:434,449 */
static uint32_t stage_avg(const orc_xcascade *c, size_t i)
{
    unsigned sh = (unsigned)(ORC_DEPTH * i);
    uint32_t v = sh >= 32 ? 0u : (c->avg_count >> sh);
    return v < c->avg_limit ? v : c->avg_limit;
}

void orc_xcascade_set_avg(orc_xcascade *c, uint32_t limit, uint32_t count)
{
    c->avg_limit = limit;
    c->avg_count = count;
    for (size_t i = 0; i < c->ns; i++)
        c->st[i]->avg = stage_avg(c, i);
}

void orc_xcascade_set_detrend(orc_xcascade *c, int d) { c->detrend = d; }

size_t orc_xcascade_num_stages(const orc_xcascade *c) { return c->ns; }

static xstage *get_or_add(orc_xcascade *c, size_t i)
{
    const size_t n = (size_t)c->n;
    while (i >= c->ns) { /* psd.rs:445-453, Psd::new psd.rs:137-152 */
        assert(c->ns < XORC_MAX_STAGES);
        xstage *s = (xstage *)calloc(1, sizeof(*s));
        s->bx = (float *)calloc(n, sizeof(float));
        s->by = (float *)calloc(n, sizeof(float));
        s->sxx = (float *)calloc(n / 2 + 1, sizeof(float));
        s->syy = (float *)calloc(n / 2 + 1, sizeof(float));
        s->sxy = (float *)calloc(n + 2, sizeof(float));
        s->hx = orc_hbf8_new(c->hbf);
        s->hy = orc_hbf8_new(c->hbf);
        s->drain = (size_t)orc_hbf_response_length(c->hbf);
        s->avg = stage_avg(c, c->ns);
        c->st[c->ns++] = s;
    }
    return c->st[i];
}

/* psd.rs:235-266 for one channel after a segment: overlap shift, decimate, drain; returns the new output count */
static size_t segment_tail(const orc_xcascade *c, float *buf, orc_hbf8 *h, size_t drain0, int is_first, float *y,
                           size_t n)
{
    const size_t N = (size_t)c->n;
    size_t start;
    if (is_first) {
        start = 0;
    } else {
        memmove(buf, buf + (N - c->overlap), c->overlap * sizeof(float));
        start = c->overlap;
    }
    assert((N - start) % 8 == 0);
    size_t chunks = (N - start) / 8;
    orc_hbf8_block(h, buf + start, chunks, y + n);
    size_t skip = drain0 < chunks ? drain0 : chunks;
    if (skip > 0)
        memmove(y + n, y + n + skip, (chunks - skip) * sizeof(float));
    n += chunks - skip;
    if (is_first)
        memmove(buf, buf + (N - c->overlap), c->overlap * sizeof(float));
    return n;
}

/* Psd::process over x and y in lockstep (psd.rs:196-269) */
static size_t xstage_process(orc_xcascade *c, xstage *s, const float *x, const float *y, size_t nx, float *ox,
                             float *oy)
{
    const size_t N = (size_t)c->n;
    size_t n = 0;
    while (nx > 0) {
        size_t take = nx < N - s->idx ? nx : N - s->idx;
        memcpy(s->bx + s->idx, x, take * sizeof(float));
        memcpy(s->by + s->idx, y, take * sizeof(float));
        x += take;
        y += take;
        nx -= take;
        s->idx += take;
        if (s->idx < N)
            break;

        if (orc_detrend_apply(c->detrend, s->bx, c->win, c->n, c->zx) != 0 ||
            orc_detrend_apply(c->detrend, s->by, c->win, c->n, c->zy) != 0)
            abort(); /* Detrend::Linear panics in the reference */
        orc_fft_forward(c->zx, c->n);
        orc_fft_forward(c->zy, c->n);

        int is_first = s->count == 0;
        float g;
        if (s->count > s->avg) {
            g = (float)s->avg / (float)s->count;
            s->count = s->avg;
        } else {
            g = 1.0f;
        }
        s->count += 1;

        for (size_t k = 0; k <= N / 2; k++) {
            float xr = c->zx[2 * k], xi = c->zx[2 * k + 1], yr = c->zy[2 * k], yi = c->zy[2 * k + 1];
            s->sxx[k] = g * s->sxx[k] + (xr * xr + xi * xi);
            s->syy[k] = g * s->syy[k] + (yr * yr + yi * yi);
            s->sxy[2 * k] = g * s->sxy[2 * k] + (xr * yr + xi * yi);
            s->sxy[2 * k + 1] = g * s->sxy[2 * k + 1] + (xr * yi - xi * yr);
        }
        const size_t drain0 = s->drain;
        size_t m = segment_tail(c, s->by, s->hy, drain0, is_first, oy, n);
        n = segment_tail(c, s->bx, s->hx, drain0, is_first, ox, n);
        assert(m == n);
        size_t chunks = (N - (is_first ? 0 : c->overlap)) / 8;
        s->drain -= drain0 < chunks ? drain0 : chunks;
        s->idx = c->overlap; /* psd.rs:266 */
    }
    return n;
}

void orc_xcascade_process(orc_xcascade *c, const float *x, const float *y, size_t n)
{
    /* psd.rs:456-468: chunks of 8N through the stage chain */
    const size_t chunk = (size_t)c->n << ORC_DEPTH;
    int cur = 0;
    for (size_t off = 0; off < n; off += chunk) {
        const float *xp = x + off, *yp = y + off;
        size_t len = n - off < chunk ? n - off : chunk;
        size_t i = 0;
        while (len > 0) {
            size_t m = xstage_process(c, get_or_add(c, i), xp, yp, len, c->ax[cur], c->ay[cur]);
            xp = c->ax[cur];
            yp = c->ay[cur];
            cur ^= 1;
            len = m;
            i++;
        }
    }
}

/* PsdCascade::psd (psd.rs:479-543) on the three rows; pxy holds (re, im) pairs */
size_t orc_xcascade_csd(const orc_xcascade *c, int keep_overlap, uint32_t min_count, int keep_transition_band,
                        float *pxx, float *pyy, float *pxy, orc_break *b, size_t *nb)
{
    const size_t N = (size_t)c->n;
    size_t plen = 0, blen = 0;
    uint64_t decimation = (uint64_t)1 << (ORC_DEPTH * c->ns);
    size_t end = 0;
    for (size_t r = c->ns; r-- > 0;) {
        const xstage *st = c->st[r];
        decimation >>= ORC_DEPTH;
        size_t start = !keep_overlap ? (end + (1u << ORC_DEPTH) - 1) >> ORC_DEPTH : 0;
        end = (decimation > 1 && !keep_transition_band) ? 2 * N / 5 : N / 2 + 1;
        int include = st->count >= min_count;
        orc_break *bk = &b[blen++];
        memset(bk, 0, sizeof(*bk));
        bk->start = plen;
        bk->count = st->count;
        bk->include = (uint32_t)include;
        bk->avg = st->avg;
        bk->bins_start = start;
        bk->bins_end = end;
        bk->fft_size = N;
        bk->decimation = decimation;
        uint32_t cm1 = st->count > 0 ? st->count - 1 : 0;
        bk->processed = (uint64_t)N * st->count - (uint64_t)c->overlap * cm1;
        bk->pending = st->idx;
        if (include) {
            /* PsdStage::gain, psd.rs:279-283 (N/2 * count in 64 bits like orc_stage_gain) */
            uint64_t nc = (uint64_t)((uint32_t)c->n / 2) * (uint64_t)st->count;
            float gain = (float)nc * c->nenbw * c->power;
            float g = 1.0f / (gain * (float)decimation);
            for (size_t k = start; k < end; k++) {
                pxx[plen] = st->sxx[k] * g;
                pyy[plen] = st->syy[k] * g;
                pxy[2 * plen] = st->sxy[2 * k] * g;
                pxy[2 * plen + 1] = st->sxy[2 * k + 1] * g;
                plen++;
            }
        } else {
            end = start;
        }
    }
    *nb = blen;
    return plen;
}
