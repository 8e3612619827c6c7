/* sspsd_poracle.c -- CPU restatement of the plants of include/sspsd.h (sspsd_plant_*, DESIGN.md 3d), TEST
 * INFRASTRUCTURE ONLY.  The inputs come from this oracle's own sources: NOISE(e, seed) is orc_source NOISE(e, seed)
 * read sequentially from position 0, and a TONE is a * c(phi_n) with c the mixer's cosine factor restated with f64
 * libm from the same exact integer phase (quadrant from the top two bits, the rest an exact f64 argument, one
 * rounding to f32).  Each output is the f64 sum over m ascending, then t ascending, rounded to f32 once. */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "sspsd_oracle.h"

enum { ORC_PLANT_NOISE = 0, ORC_PLANT_TONE = 1 };

/* cos(2 pi phi / 2^32) as the heterodyne mixer forms it */
float orc_plant_cos(uint32_t phi)
{
    const uint32_t quad = phi >> 30;
    const double a = (double)(phi & 0x3fffffffu) * 0x1p-31 * 3.14159265358979323846;
    const float cf = (float)cos(a), sf = (float)sin(a);
    switch (quad) {
    case 0: return cf;
    case 1: return -sf;
    case 2: return -cf;
    default: return sf;
    }
}

/* positions [pos, pos + n) of all k outputs into out[i * n + j]; inputs are generated from position 0.
 * Returns 0, or -1 for a kind or exponent the plant refuses, -2 when out of memory. */
int orc_plant_generate(uint32_t k, uint32_t m, uint32_t taps_len, const float *taps, const int32_t *kinds,
                       const int64_t *params, const uint64_t *seeds, const float *amps, uint64_t pos, size_t n,
                       float *out)
{
    const size_t len = (size_t)pos + n;
    float *u = malloc(sizeof(float) * (len ? len : 1) * m);
    if (!u)
        return -2;
    for (uint32_t q = 0; q < m; q++) {
        float *uq = u + (size_t)q * len;
        if (kinds[q] == ORC_PLANT_NOISE) {
            if (params[q] < 0 || params[q] > 8) {
                free(u);
                return -1;
            }
            orc_source *s = orc_source_new(ORC_SOURCE_NOISE, params[q], seeds[q]);
            if (!s) {
                free(u);
                return -2;
            }
            orc_source_get(s, uq, len);
            orc_source_free(s);
        } else if (kinds[q] == ORC_PLANT_TONE) {
            const uint32_t ftw = (uint32_t)params[q];
            for (size_t j = 0; j < len; j++)
                uq[j] = amps[q] * orc_plant_cos((uint32_t)((uint64_t)j * ftw));
        } else {
            free(u);
            return -1;
        }
    }
    for (uint32_t i = 0; i < k; i++)
        for (size_t j = 0; j < n; j++) {
            const uint64_t p = pos + j;
            double acc = 0.0;
            for (uint32_t q = 0; q < m; q++)
                for (uint32_t t = 0; t < taps_len && t <= p; t++)
                    acc += (double)taps[((size_t)i * m + q) * taps_len + t] * (double)u[(size_t)q * len + (p - t)];
            out[(size_t)i * n + j] = (float)acc;
        }
    free(u);
    return 0;
}
