/* roiaware_oracle.c -- CPU restatement of the roiaware_pool3d ops (TEST INFRASTRUCTURE): points_in_boxes (GPU and CPU
 * forms), the RoIAwarePool3d forward (voxel lists, max / avg pooling), in the order the contract of
 * csrc/roiaware_pool3d.cu states.  Compiled with -ffp-contract=off: the only fused multiply-adds are the explicit fmaf()
 * calls of the GPU form's local coordinates. */
#include <limits.h>
#include <math.h>
#include <string.h>

#define EXPORT __attribute__((visibility("default")))

/* the reference's test; fused = 1: local_x = fmaf(sx, cosa, sy * -sina), local_y = fmaf(sy, cosa, sx * sina) (the
 * contraction nvcc makes of the reference's expressions), 0: every product rounded (the CPU form) */
static int in_box(const float* pt, const float* b, float margin, int fused, float* lx, float* ly) {
    const float x = pt[0], y = pt[1], z = pt[2];
    if (!(fabsf(z - b[2]) <= b[5] / 2.0)) return 0; /* upstream writes `> dz / 2.0`; a NaN fails here on purpose */
    const float cosa = cosf(-b[6]), sina = sinf(-b[6]);
    const float sx = x - b[0], sy = y - b[1];
    if (fused) {
        *lx = fmaf(sx, cosa, sy * -sina);
        *ly = fmaf(sy, cosa, sx * sina);
    } else {
        *lx = sx * cosa + sy * -sina;
        *ly = sx * sina + sy * cosa;
    }
    return fabs(*lx) < b[3] / 2.0 + margin && fabs(*ly) < b[4] / 2.0 + margin;
}

/* cvt.rzi.s32.f32: truncation, NaN -> 0, saturation at the int range */
static int f2i_rz(float v) {
    if (v != v) return 0;
    if (v >= 2147483648.0f) return INT_MAX;
    if (v <= -2147483648.0f) return INT_MIN;
    return (int)v;
}

/* (unsigned) int((l + half) / res), then the unsigned min(max(i, 0), n - 1) */
static unsigned cell(float l, float half, float res, int n) {
    const unsigned i = (unsigned)f2i_rz((l + half) / res);
    return i < (unsigned)(n - 1) ? i : (unsigned)(n - 1);
}

/* out (B, N), pre-filled by the caller: the first box k of the frame holding the point (margin 1e-5, GPU form) */
EXPORT void rao_points_in_boxes(int b, int t, int n, const float* boxes, const float* pts, int* out) {
    float lx, ly;
    for (int f = 0; f < b; ++f)
        for (int k = 0; k < n; ++k)
            for (int j = 0; j < t; ++j)
                if (in_box(pts + ((size_t)f * n + k) * 3, boxes + ((size_t)f * t + j) * 7, 1e-5f, 1, &lx, &ly)) {
                    out[(size_t)f * n + k] = j;
                    break;
                }
}

/* out (M, N): 0 / 1 for every pair (margin 1e-2, every product rounded) */
EXPORT void rao_points_in_boxes_cpu(int m, int n, const float* boxes, const float* pts, int* out) {
    float lx, ly;
    for (int i = 0; i < m; ++i)
        for (int k = 0; k < n; ++k) out[(size_t)i * n + k] = in_box(pts + (size_t)k * 3, boxes + (size_t)i * 7, 1e-2f, 0, &lx, &ly);
}

/* the forward on zeroed outputs: idx (R, X, Y, Z, L), argmax / pooled (R, X, Y, Z, C); method 0 max, 1 avg */
EXPORT void rao_forward(int r, int p, int c, int X, int Y, int Z, int L, const float* rois, const float* pts,
                        const float* feats, int* argmax, int* idx, float* pooled, int method) {
    const size_t V = (size_t)X * Y * Z;
    for (int i = 0; i < r; ++i) {
        const float* b = rois + (size_t)i * 7;
        const float dx = b[3], dy = b[4], dz = b[5];
        const float rx = dx / X, ry = dy / Y, rz = dz / Z;
        int* lists = idx + (size_t)i * V * L;
        for (int k = 0; k < p; ++k) {
            float lx, ly;
            const float* pt = pts + (size_t)k * 3;
            if (!in_box(pt, b, 1e-5f, 1, &lx, &ly)) continue;
            const float lz = pt[2] - b[2];
            const unsigned ix = cell(lx, dx / 2, rx, X), iy = cell(ly, dy / 2, ry, Y), iz = cell(lz, dz / 2, rz, Z);
            int* v = lists + ((size_t)(ix * Y + iy) * Z + iz) * L;
            if (v[0] < L - 1) {
                v[v[0] + 1] = k;
                v[0] += 1;
            }
        }
        for (size_t g = 0; g < V; ++g) {
            const int* v = lists + g * L;
            const size_t o = ((size_t)i * V + g) * c;
            for (int ch = 0; ch < c; ++ch) {
                if (method == 0) {
                    float best = -INFINITY; /* the reference's float max_val = -1e50 */
                    int arg = -1;
                    for (int k = 1; k <= v[0]; ++k)
                        if (feats[(size_t)v[k] * c + ch] > best) {
                            best = feats[(size_t)v[k] * c + ch];
                            arg = v[k];
                        }
                    if (arg != -1) pooled[o + ch] = best;
                    argmax[o + ch] = arg;
                } else {
                    float s = 0.f;
                    for (int k = 1; k <= v[0]; ++k) s += feats[(size_t)v[k] * c + ch];
                    if (v[0] > 0) pooled[o + ch] = s / v[0];
                }
            }
        }
    }
}
