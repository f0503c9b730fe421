/* vector_pool_oracle.c -- CPU restatement of pointnet2_stack's vector-pool functions (TEST INFRASTRUCTURE), one centre
 * after another, in the order the contract of csrc/stack_vector_pool.cu states.  Compiled with -ffp-contract=off: the
 * only fused multiply-adds are the explicit fmaf() calls of the distance. */
#include <math.h>
#include <string.h>

#define VPO_CAP 1000
#define EXPORT __attribute__((visibility("default")))

static int frame_of(int p, int b, const int* mcnt) {
    int acc = 0;
    for (int k = 0; k < b; ++k) {
        acc += mcnt[k];
        if (p < acc) return k;
    }
    return b - 1;
}

static int frame_start(int f, const int* ncnt) {
    int s = 0;
    for (int k = 0; k < f; ++k) s += ncnt[k];
    return s;
}

static int is_hit(float lx, float ly, float lz, float d, int ball) {
    if (ball == 1) {
        const float r2 = d * d;
        return fmaf(lz, lz, fmaf(lx, lx, ly * ly)) <= r2;
    }
    return fabsf(lx) <= d && fabsf(ly) <= d && fabsf(lz) <= d;
}

/* lists (M, 1000): the first min(hits, 1000, nsample if > 0) hits of every centre as global rows; lens (M) */
EXPORT void vpo_local_idxs(int b, int m, const float* xyz, const int* ncnt, const float* new_xyz, const int* mcnt,
                           float d, int nsample, int ball, int* lists, int* lens) {
    const int cap = nsample > 0 && nsample < VPO_CAP ? nsample : VPO_CAP;
    for (int p = 0; p < m; ++p) {
        const int f = frame_of(p, b, mcnt), s = frame_start(f, ncnt);
        int cnt = 0;
        for (int k = 0; k < ncnt[f] && cnt < cap; ++k) {
            const float* q = xyz + 3 * (size_t)(s + k);
            const float lx = q[0] - new_xyz[3 * p], ly = q[1] - new_xyz[3 * p + 1], lz = q[2] - new_xyz[3 * p + 2];
            if (is_hit(lx, ly, lz, d, ball)) lists[(size_t)p * VPO_CAP + cnt++] = s + k;
        }
        lens[p] = cnt;
    }
}

/* idx / dist2 (M, G, 3): strict-< cascade over each centre's list (lists (M, 1000), lens (M)) from every sub-voxel
 * centre (M, G, 3); unfilled slots (+inf, -1) */
EXPORT void vpo_three_nn(int m, int G, const float* xyz, const float* centres, const int* lists, const int* lens, int* idx,
                         float* dist2) {
    for (int p = 0; p < m; ++p)
        for (int g = 0; g < G; ++g) {
            const size_t r = (size_t)p * G + g;
            const float* c = centres + 3 * r;
            float b1 = INFINITY, b2 = INFINITY, b3 = INFINITY;
            int i1 = -1, i2 = -1, i3 = -1;
            for (int j = 0; j < lens[p]; ++j) {
                const int k = lists[(size_t)p * VPO_CAP + j];
                const float* q = xyz + 3 * (size_t)k;
                const float dx = c[0] - q[0], dy = c[1] - q[1], dz = c[2] - q[2];
                const float dd = fmaf(dz, dz, fmaf(dx, dx, dy * dy));
                if (dd < b1) {
                    b3 = b2; i3 = i2; b2 = b1; i2 = i1; b1 = dd; i1 = k;
                } else if (dd < b2) {
                    b3 = b2; i3 = i2; b2 = dd; i2 = k;
                } else if (dd < b3) {
                    b3 = dd; i3 = k;
                }
            }
            dist2[3 * r] = b1; dist2[3 * r + 1] = b2; dist2[3 * r + 2] = b3;
            idx[3 * r] = i1; idx[3 * r + 1] = i2; idx[3 * r + 2] = i3;
        }
}

/* vector_pool_wrapper on zeroed outputs: new_features (M, cout), new_local_xyz (M, 3G), cnt (M, G), triples
 * (max_triples, 3) in centre-then-index order; returns the exact number of triples */
EXPORT long long vpo_pool(int b, int m, const float* xyz, const int* ncnt, const float* feats, int cin, const float* new_xyz,
                          const int* mcnt, int nx, int ny, int nz, int cout, float d, int use_xyz, int nsample, int ball,
                          int pooling, float* new_features, float* new_local_xyz, int* cnt, int* triples,
                          long long max_triples) {
    const int G = nx * ny * nz, cpg = cout / G;
    const float gsx = d * 2 / nx, gsy = d * 2 / ny, gsz = d * 2 / nz;
    long long total = 0;
    for (int p = 0; p < m; ++p) {
        const int f = frame_of(p, b, mcnt), s = frame_start(f, ncnt);
        float* nf = new_features + (size_t)p * cout;
        float* nl = new_local_xyz + (size_t)p * 3 * G;
        int* nc = cnt + (size_t)p * G;
        int taken = 0;
        for (int k = 0; k < ncnt[f]; ++k) {
            const float* q = xyz + 3 * (size_t)(s + k);
            const float l[3] = {q[0] - new_xyz[3 * p], q[1] - new_xyz[3 * p + 1], q[2] - new_xyz[3 * p + 2]};
            if (!is_hit(l[0], l[1], l[2], d, ball)) continue;
            const int ix = (int)floorf((l[0] + d) / gsx), iy = (int)floorf((l[1] + d) / gsy),
                      iz = (int)floorf((l[2] + d) / gsz);
            int g = ix * ny * nz + iy * nz + iz;
            g = g < 0 ? 0 : (g > G - 1 ? G - 1 : g);
            const float* fk = feats + (size_t)(s + k) * cin;
            if (pooling == 0) {
                nc[g] += 1;
                for (int i = 0; i < cin; ++i) nf[g * cpg + i % cpg] += fk[i];
                if (use_xyz)
                    for (int a = 0; a < 3; ++a) nl[3 * g + a] += l[a];
            } else {
                if (nc[g] != 0) continue;
                nc[g] = 1;
                for (int i = 0; i < cin; ++i) nf[g * cpg + i % cpg] = fk[i];
                if (use_xyz)
                    for (int a = 0; a < 3; ++a) nl[3 * g + a] = l[a];
            }
            if (total < max_triples) {
                triples[3 * total] = s + k; triples[3 * total + 1] = p; triples[3 * total + 2] = g;
            }
            ++total;
            ++taken;
            if (nsample > 0 && taken >= nsample) break;
            if (pooling != 0 && taken >= G) break;
        }
    }
    return total;
}
