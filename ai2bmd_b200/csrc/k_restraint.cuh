// Hookean restraints on the whole-protein state: the position restraints of the reference's pre-equilibration and the
// hydrogen-bond springs of its --constraints option (src/AIMD/simulator.py:139-180; ASE 3.22 ase/constraints.py Hookean,
// recalled, restated on the host in ai2bmd_b200/restraints.py `hookean`, which is this file's checker).
//   point (a, p0, k, rt): d = p0 - x_a, r = |d|; r > rt:  F_a += k (r - rt) d/r,               E += k (r - rt)^2 / 2
//   pair  (i, j, k, rt):  d = x_j - x_i, r = |d|; r > rt: F_i += k (r - rt) d/r, F_j -= same,  E += k (r - rt)^2 / 2
// No atomics: the restraints are a CSR over destination atoms (entry = restraint id * 2 + role, role 1 = second atom of a
// pair), one thread gathers all terms of an atom in fp64, and a restraint's energy is counted by the owner of its first
// atom through a fixed-order block reduction -- two calls on the same input are bit-identical.  [lo, hi) are the atoms
// this handle computes, so the slices of a sharded run sum to the whole term under the all-reduce.  One CTA: a few
// hundred to a few thousand atoms, next to single-CTA MD kernels.
#pragma once
#include <cuda_runtime.h>

namespace vb {

constexpr int RS_THREADS = 256;

struct RsParams {
    int n;                        // protein atoms
    int lo, hi;                   // destination atoms this handle computes
    int n_point;                  // ids [0, n_point) are point restraints, [n_point, n_point + n_pair) pair restraints
    const int* row;               // [n+1] CSR over destination atoms
    const int* ent;               // restraint id * 2 + role
    const double* point_anchor;   // [n_point][3] Angstrom
    const double* point_k;        // eV / Angstrom^2
    const double* point_rt;       // Angstrom
    const int* pair_ij;           // [n_pair][2]
    const double* pair_k;
    const double* pair_rt;
};

__global__ void __launch_bounds__(RS_THREADS) restraint_kernel(RsParams p, const double* __restrict__ pos, float* __restrict__ ef) {
    __shared__ double red[RS_THREADS / 32];
    double e = 0.0;
    for (int a = p.lo + threadIdx.x; a < p.hi; a += RS_THREADS) {
        const int r0 = p.row[a], r1 = p.row[a + 1];
        if (r0 == r1) continue;
        const double xa = pos[3 * a], ya = pos[3 * a + 1], za = pos[3 * a + 2];
        double fx = 0.0, fy = 0.0, fz = 0.0;
        for (int m = r0; m < r1; m++) {
            const int id = p.ent[m] >> 1;
            const bool second = p.ent[m] & 1;
            double dx, dy, dz, k, rt;
            if (id < p.n_point) {
                dx = p.point_anchor[3 * id] - xa; dy = p.point_anchor[3 * id + 1] - ya; dz = p.point_anchor[3 * id + 2] - za;
                k = p.point_k[id]; rt = p.point_rt[id];
            } else {
                const int q = id - p.n_point, i = p.pair_ij[2 * q], j = p.pair_ij[2 * q + 1];
                dx = pos[3 * j] - pos[3 * i]; dy = pos[3 * j + 1] - pos[3 * i + 1]; dz = pos[3 * j + 2] - pos[3 * i + 2];
                k = p.pair_k[q]; rt = p.pair_rt[q];
            }
            const double r = sqrt(dx * dx + dy * dy + dz * dz);
            if (!(r > rt)) continue;                       // flat bottom (also r = rt = 0: no force, no 0/0)
            const double s = k * (r - rt), c = (second ? -s : s) / r;
            fx += c * dx; fy += c * dy; fz += c * dz;
            if (!second) e += 0.5 * s * (r - rt);
        }
        ef[3 * a] += (float)fx; ef[3 * a + 1] += (float)fy; ef[3 * a + 2] += (float)fz;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) e += __shfl_xor_sync(0xffffffffu, e, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = e;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < RS_THREADS / 32; w++) t += red[w];
        ef[3 * p.n] += (float)t;
    }
}

}  // namespace vb
