/* Reference of the rectification into output axes of any size (cc_rectify_axes_*): warp(img, tform, axs) with
 * axs = axs_min .+ (0:out_sz1-1, 0:out_sz2-1).  TEST INFRASTRUCTURE ONLY, built by tests/rectify_axes_ref.py with
 * the flags of oracle/Makefile and linked against the oracle: the source coordinate of every output index is the
 * oracle's own cco_rectify_coord, the bounds rule and the blend are cco_rectify_f32c1 / cco_rectify_u8c3's,
 * operation for operation.  Only the output geometry differs: output pixel (a+1, b+1) of frame f is at
 * dst + f*out_frame_stride + b*out_pitch + a (u8c3: times 3 bytes); the source frames are sz1 x sz2. */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

#include "camcal_oracle.h"

/* the oracle's bilinear rule: outside [1, n] -> 0; i = floor(x), pulled back by one when x == n */
static int lin_pos(double x, int n, int *i0, double *d)
{
    if (!(x >= 1.0 && x <= (double)n)) return 0;
    double xf = floor(x);
    if (xf > (double)(n - 1)) xf -= 1.0;
    *d = x - xf;
    *i0 = (int)xf - 1;
    return 1;
}

void ref_rectify_f32c1_axes(const cco_chain *ch, double inv_ratio, const long long axs_min[2], const float *src,
                            int sz1, int sz2, size_t pitch, size_t frame_stride, float *dst, int out_sz1,
                            int out_sz2, size_t out_pitch, size_t out_frame_stride, int nframes, float fill)
{
    for (int f = 0; f < nframes; ++f)
        for (int b = 0; b < out_sz2; ++b) {
            const float *s = src + (size_t)f * frame_stride;
            float *o = dst + (size_t)f * out_frame_stride + (size_t)b * out_pitch;
            for (int a = 0; a < out_sz1; ++a) {
                double row, col, d1, d2;
                int i1, i2;
                cco_rectify_coord(ch, inv_ratio, axs_min[0] + a, axs_min[1] + b, &row, &col);
                if (!lin_pos(row, sz1, &i1, &d1) || !lin_pos(col, sz2, &i2, &d2)) {
                    o[a] = fill;
                    continue;
                }
                const float *p = s + (size_t)i2 * pitch + i1;
                double a00 = p[0], a10 = p[1], a01 = p[pitch], a11 = p[pitch + 1];
                double e1 = 1.0 - d1, e2 = 1.0 - d2;
                double lo = fma(d2, a01, e2 * a00);
                double hi = fma(d2, a11, e2 * a10);
                o[a] = (float)fma(d1, hi, e1 * lo);
            }
        }
}

void ref_rectify_u8c3_axes(const cco_chain *ch, double inv_ratio, const long long axs_min[2], const uint8_t *src,
                           int sz1, int sz2, size_t pitch, size_t frame_stride, uint8_t *dst, int out_sz1,
                           int out_sz2, size_t out_pitch, size_t out_frame_stride, int nframes,
                           const uint8_t fill[3])
{
    for (int f = 0; f < nframes; ++f)
        for (int b = 0; b < out_sz2; ++b) {
            const uint8_t *s = src + (size_t)f * frame_stride * 3;
            uint8_t *o = dst + ((size_t)f * out_frame_stride + (size_t)b * out_pitch) * 3;
            for (int a = 0; a < out_sz1; ++a) {
                double row, col, d1, d2;
                int i1, i2;
                cco_rectify_coord(ch, inv_ratio, axs_min[0] + a, axs_min[1] + b, &row, &col);
                if (!lin_pos(row, sz1, &i1, &d1) || !lin_pos(col, sz2, &i2, &d2)) {
                    o[3 * a] = fill[0]; o[3 * a + 1] = fill[1]; o[3 * a + 2] = fill[2];
                    continue;
                }
                const uint8_t *p = s + ((size_t)i2 * pitch + i1) * 3;
                double e1 = 1.0 - d1, e2 = 1.0 - d2;
                for (int c = 0; c < 3; ++c) {
                    double a00 = p[c], a10 = p[3 + c];
                    double a01 = p[3 * pitch + c], a11 = p[3 * pitch + 3 + c];
                    double lo = fma(d2, a01, e2 * a00);
                    double hi = fma(d2, a11, e2 * a10);
                    double val = rint(fma(d1, hi, e1 * lo));
                    if (val < 0.0) val = 0.0;
                    if (val > 255.0) val = 255.0;
                    o[3 * a + c] = (uint8_t)val;
                }
            }
        }
}
