/* sspsd_zoracle.c -- CPU restatement of the two-sided spectrum of z = i + i q (TEST INFRASTRUCTURE ONLY).
 *
 * The reference has no two-sided spectrum.  The restatement is sspsd_xoracle.c's lockstep Psd::process over the two
 * real streams i and q (same segments, window, detrend of each, half-band decimators, EWMA factors), with the
 * per-segment step replaced: i and q are detrended and windowed each with orc_detrend_apply, z = i~ + i q~ goes
 * through ONE N-point complex orc_fft_forward, and the stage accumulates, over all k = 0 .. N/2, in f32, unfused
 * (-ffp-contract=off):
 *   P+[k] = g s + (zr zr + zi zi) of Z[k],   P-[k] = g s + (zr zr + zi zi) of Z[(N - k) mod N].
 * P+ and P- live in the xstage's sxx and syy rows, so orc_xcascade_csd merges them (pxx = P+, pyy = P-, with
 * 1/(gain_i 8^i)); the binding halves both into the two-sided density.  sspsd_xoracle.c is compiled into this
 * object unchanged, so the CSD restatement keeps its outputs bit for bit.
 */
#include "sspsd_xoracle.c"

void orc_zcascade_process(orc_xcascade *c, const float *i, const float *q, size_t n);

/* xstage_process with the two-sided step: sxx <- P+, syy <- P- (sxy unused) */
static size_t zstage_process(orc_xcascade *c, xstage *s, const float *x, const float *y, size_t nx, float *ox,
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
        for (size_t k = 0; k < N; k++)
            c->zx[2 * k + 1] = c->zy[2 * k]; /* z = i~ + i q~ (both real after the detrend and window) */
        orc_fft_forward(c->zx, c->n);

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
            const size_t m = (N - k) % N;
            float pr = c->zx[2 * k], pi = c->zx[2 * k + 1], mr = c->zx[2 * m], mi = c->zx[2 * m + 1];
            s->sxx[k] = g * s->sxx[k] + (pr * pr + pi * pi);
            s->syy[k] = g * s->syy[k] + (mr * mr + mi * mi);
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

/* orc_xcascade_process with zstage_process */
void orc_zcascade_process(orc_xcascade *c, const float *i, const float *q, size_t n)
{
    const size_t chunk = (size_t)c->n << ORC_DEPTH;
    int cur = 0;
    for (size_t off = 0; off < n; off += chunk) {
        const float *xp = i + off, *yp = q + off;
        size_t len = n - off < chunk ? n - off : chunk;
        size_t st = 0;
        while (len > 0) {
            size_t m = zstage_process(c, get_or_add(c, st), xp, yp, len, c->ax[cur], c->ay[cur]);
            xp = c->ax[cur];
            yp = c->ay[cur];
            cur ^= 1;
            len = m;
            st++;
        }
    }
}
