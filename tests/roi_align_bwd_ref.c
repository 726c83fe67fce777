/* Oracle (test-only): ROI Align backward, CPU, the literal transpose of oracle/csrc/roi_align_ref.c.
 *
 * For every grad_out element g[k][c][ph][pw] and every sample of its bin that the forward op reads (same
 * geometry, same float32 sample positions and bilinear weights as the forward oracle and as torchvision's
 * CPU _roi_align_backward), each of the four taps receives the float32 value g * w / count; those values
 * are summed in double, so the result does not depend on summation order.  ROIs whose batch index is
 * outside [0,B) contribute nothing.  When `mag` is given, |g * w / count| is summed into it as well: because
 * every bilinear weight is non-negative that is, per map cell, the sum of the magnitudes of all contributions
 * -- the scale of the rounding error any order of float32 additions can make.
 * Compile with -ffp-contract=off so coordinate arithmetic rounds like the wheel's.
 */
#include <math.h>
#include <stdint.h>

static void tap4_bwd(double *plane, double *mplane, int H, int W, float y, float x, float g, float count)
{
    if (!(y >= -1.0f && y <= (float)H && x >= -1.0f && x <= (float)W)) return;   /* NaN positions too */
    if (y <= 0.0f) y = 0.0f;
    if (x <= 0.0f) x = 0.0f;
    int y0 = (int)y, x0 = (int)x, y1, x1;
    if (y0 >= H - 1) { y0 = y1 = H - 1; y = (float)y0; } else y1 = y0 + 1;
    if (x0 >= W - 1) { x0 = x1 = W - 1; x = (float)x0; } else x1 = x0 + 1;
    float ly = y - (float)y0, lx = x - (float)x0, hy = 1.0f - ly, hx = 1.0f - lx;
    float v[4] = {g * (hy * hx) / count, g * (hy * lx) / count, g * (ly * hx) / count, g * (ly * lx) / count};
    plane[y0 * W + x0] += v[0];
    plane[y0 * W + x1] += v[1];
    plane[y1 * W + x0] += v[2];
    plane[y1 * W + x1] += v[3];
    if (mplane) {
        mplane[y0 * W + x0] += fabsf(v[0]);
        mplane[y0 * W + x1] += fabsf(v[1]);
        mplane[y1 * W + x0] += fabsf(v[2]);
        mplane[y1 * W + x1] += fabsf(v[3]);
    }
}

/* grad_out: [K,C,PH,PW] float32; rois: [K,5] = (batch, x1, y1, x2, y2); grad_in and mag (or NULL): [B,C,H,W]
 * double, added to. */
void oracle_roi_align_bwd_f32(const float *grad_out, int B, int C, int H, int W, const float *rois, int64_t K,
                              int PH, int PW, float scale, int sampling_ratio, int aligned, double *grad_in,
                              double *mag)
{
    const float off = aligned ? 0.5f : 0.0f;
    for (int64_t k = 0; k < K; ++k) {
        const float *r = rois + 5 * k;
        int b = (int)r[0];
        if (!(r[0] == r[0]) || b < 0 || b >= B) continue;
        float sw = r[1] * scale - off, sh = r[2] * scale - off;
        float ew = r[3] * scale - off, eh = r[4] * scale - off;
        float rw = ew - sw, rh = eh - sh;
        if (!aligned) { rw = fmaxf(rw, 1.0f); rh = fmaxf(rh, 1.0f); }
        float bh = rh / (float)PH, bw = rw / (float)PW;
        int gh = sampling_ratio > 0 ? sampling_ratio : (int)ceilf(rh / (float)PH);
        int gw = sampling_ratio > 0 ? sampling_ratio : (int)ceilf(rw / (float)PW);
        float count = (float)(gh * gw > 1 ? gh * gw : 1);
        for (int c = 0; c < C; ++c) {
            double *plane = grad_in + ((int64_t)b * C + c) * H * W;
            double *mplane = mag ? mag + ((int64_t)b * C + c) * H * W : 0;
            const float *g = grad_out + ((k * C + c) * PH) * PW;
            for (int ph = 0; ph < PH; ++ph)
                for (int pw = 0; pw < PW; ++pw)
                    for (int iy = 0; iy < gh; ++iy) {
                        float y = sh + (float)ph * bh + ((float)iy + 0.5f) * bh / (float)gh;
                        for (int ix = 0; ix < gw; ++ix) {
                            float x = sw + (float)pw * bw + ((float)ix + 0.5f) * bw / (float)gw;
                            tap4_bwd(plane, mplane, H, W, y, x, g[ph * PW + pw], count);
                        }
                    }
        }
    }
}
