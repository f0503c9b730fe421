/*
 * tests/stack_bq_oracle.c -- CPU restatement of the reference's stacked ball query (TEST INFRASTRUCTURE ONLY),
 * /root/reference/pcdet/ops/pointnet2/pointnet2_stack/src/ball_query_gpu.cu:15-62 ball_query_kernel_stack.
 * Built by tests/stack_bq_oracle.py with gcc -O2 -ffp-contract=off, so only the explicit fmaf() fuses.
 *
 * new_xyz (M,3), xyz (N,3) stacked, counts (B) -> idx (M,nsample), zeroed by the caller: centre p belongs to the first
 * frame k with p < M0 + ... + Mk (the search stops at B - 1); frame-local indices; the first hit fills every slot
 * before the hits are written in order; a centre without hits gets idx[p,0] = -1 only.  The distance is nvcc 12.9's
 * contraction of (nx-x)*(nx-x) + (ny-y)*(ny-y) + (nz-z)*(nz-z) for sm_100a (PTX of the reference kernel body:
 * "mul dy,dy; fma dx,dx,_; fma dz,dz,_"), compared strictly against the fp32 product radius * radius.
 */
#include <math.h>
#include <stddef.h>

__attribute__((visibility("default"))) void sbq_stack_ball_query(int b, int m, float radius, int nsample,
                                                                 const float *new_xyz, const int *new_xyz_batch_cnt,
                                                                 const float *xyz, const int *xyz_batch_cnt,
                                                                 int *idx_all) {
    const float radius2 = radius * radius;
    for (int pt = 0; pt < m; ++pt) {
        int bs = 0, acc = new_xyz_batch_cnt[0];
        for (int q = 1; q < b; ++q) {
            if (pt < acc) break;
            acc += new_xyz_batch_cnt[q];
            bs = q;
        }
        size_t start = 0;
        for (int k = 0; k < bs; ++k) start += xyz_batch_cnt[k];
        const float *pts = xyz + start * 3;
        int *idx = idx_all + (size_t)pt * nsample;
        const float nx = new_xyz[pt * 3 + 0], ny = new_xyz[pt * 3 + 1], nz = new_xyz[pt * 3 + 2];
        const int n = xyz_batch_cnt[bs];
        int cnt = 0;
        for (int k = 0; k < n; ++k) {
            const float dx = nx - pts[k * 3 + 0], dy = ny - pts[k * 3 + 1], dz = nz - pts[k * 3 + 2];
            const float d2 = fmaf(dz, dz, fmaf(dx, dx, dy * dy));
            if (d2 < radius2) {
                if (cnt == 0)
                    for (int l = 0; l < nsample; ++l) idx[l] = k;
                idx[cnt] = k;
                ++cnt;
                if (cnt >= nsample) break;
            }
        }
        if (cnt == 0) idx[0] = -1;
    }
}
