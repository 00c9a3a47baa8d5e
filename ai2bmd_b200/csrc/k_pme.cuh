// PME non-bonded term of the fragment calculator: the reference's `--fragment-longrange-calc pme` choice,
// PMENonBondedCalculator (src/Calculators/pme.py:77-214; checker oracle/pme_ref.py).
//   E = [k (E_rec + E_dir(P, erfc) + E_adj(X, -erf) + slf + neutral - E_dir(X, erfc)) + E_LJ(P) - E_LJ(X)] * kJ/mol
//   F = sum_P (F_LJ + F_C) - sum_X (F_LJ + F_C)  on dst, F_C = k q q vec / d^3 (plain Coulomb; E_rec gives no force)
// P: ordered pairs i != j with d < cutoff (no periodic images, pairs inside a dipeptide included); X: every ordered pair
// inside a dipeptide; every pair sum carries 1/2.  The direct kernel uses the net value of each pair: an excluded pair
// inside the cutoff adds only its erf term (its P and X contributions cancel in exact arithmetic -- the reference's fp32
// subtraction of ~1e6 kJ/mol sums is not reproduced), one beyond the cutoff also subtracts its LJ, Coulomb force and
// erfc term.  Per-pair arithmetic in fp32 in the reference's operation order, per-atom sums in fp64 (warp-ordered).
//
// E_rec is smooth PME (order-4 B-splines, Euler exponential-spline moduli) in fp64 on the orthorhombic K1 x K2 x K3 grid:
//   bin (1 CTA: spline weights, atoms binned by their base plane on axis 1) -> spread (gather per grid point, no atomics)
//   -> dft3 (real -> Hermitian half along axis 3) -> dft2 -> dft1 + energy (per-CTA partial sums)
// The DFTs are direct per-axis sums over host-made fp64 twiddle tables: the grid sizes int(L / 1 A) are arbitrary
// (often prime) and the library links no FFT library.  Every sum runs in a fixed order, so two calls are bit-identical.
// A final single-CTA launch adds the direct sums, E_rec and the constants into ef[3n] in eV.  Only a handle whose slice
// starts at atom 0 computes E_rec and the constants, so the all-reduce of a sharded run counts them once.
#pragma once
#include <cuda_runtime.h>

namespace vb {

constexpr int PME_THREADS = 256;
enum { PME_DIR = 0, PME_ADJ, PME_EX, PME_LJ, PME_LJEX, PME_NATOM };                 // per-atom fp64 components
enum { PT_DIR = 0, PT_ADJ, PT_EX, PT_REC, PT_SLF, PT_NEUTRAL, PT_LJ, PT_LJEX, PT_N };  // vb_debug_read("pme_terms")

struct PmeParams {
    int n;                        // atoms
    int lo, hi;                   // destination atoms of the direct sums
    bool recip;                   // add E_rec + slf + neutral (the handle whose slice starts at atom 0)
    const float* q;               // [n] e
    const float* sigma;           // [n] nm
    const float* eps;             // [n] kJ/mol
    const int* excl_rowptr;       // [n+1]
    const int* excl_col;          // sorted within a row
    float coulomb_k, kj_mol;      // as NbParams
    float beta, rc2;              // fp32 screening parameter (1/A) and cutoff^2 (A^2) of the direct sums
    double beta64, k64, kj64, slf, neutral;
    int K1, K2, K3, H3;           // grid; H3 = K3/2 + 1 (Hermitian half along axis 3)
    double L1, L2, L3;            // cell (A)
    const double* tw;             // [(K1 + K2 + K3) * 2] cos, sin(2 pi j / K) per axis
    const double* bmod;           // [K1 + K2 + K3] |b(m)|^2
    int* base;                    // [n][3] spline base grid index per axis
    double* w;                    // [n][3][4] weight of grid point base - t
    int* bin_ptr;                 // [K1 + 1]
    int* bin_atom;                // [n] atoms by base plane on axis 1, ascending within a plane
    double* Q;                    // [K1][K2][K3]
    double2* A;                   // [K1][K2][H3]
    double2* B;                   // [K1][K2][H3]  (axis 2 transformed)
    double* partial;              // [ceil(K1 K2 H3 / PME_THREADS)]
    double* eatom;                // [n][PME_NATOM]
    double* terms;                // [PT_N]
};

__device__ __forceinline__ double pme_block_sum(double s, double* red) {   // fixed-order sum; valid in thread 0
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    double t = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < PME_THREADS / 32; w++) t += red[w];
    return t;
}

template <typename PosT>
__global__ void __launch_bounds__(PME_THREADS) pme_bin_kernel(PmeParams p, const PosT* __restrict__ pos) {
    const int K[3] = {p.K1, p.K2, p.K3};
    const double L[3] = {p.L1, p.L2, p.L3};
    for (int a = threadIdx.x; a < p.n; a += PME_THREADS) {
        for (int ax = 0; ax < 3; ax++) {
            const double u = (double)pos[3 * a + ax] * K[ax] / L[ax];
            const double fl = floor(u), x = u - fl;
            int b = (int)fmod(fl, (double)K[ax]);
            if (b < 0) b += K[ax];
            p.base[3 * a + ax] = b;
            double* w = p.w + 12 * a + 4 * ax;          // M4(x + t), t = 0..3
            w[0] = x * x * x / 6.0;
            w[1] = (((-3.0 * x + 3.0) * x + 3.0) * x + 1.0) / 6.0;
            w[2] = ((3.0 * x - 6.0) * x * x + 4.0) / 6.0;
            w[3] = (1.0 - x) * (1.0 - x) * (1.0 - x) / 6.0;
        }
    }
    __syncthreads();
    for (int b = threadIdx.x; b < p.K1; b += PME_THREADS) {
        int c = 0;
        for (int a = 0; a < p.n; a++) c += p.base[3 * a] == b;
        p.bin_ptr[b + 1] = c;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        p.bin_ptr[0] = 0;
        for (int b = 0; b < p.K1; b++) p.bin_ptr[b + 1] += p.bin_ptr[b];
    }
    __syncthreads();
    for (int b = threadIdx.x; b < p.K1; b += PME_THREADS) {
        int m = p.bin_ptr[b];
        for (int a = 0; a < p.n; a++)
            if (p.base[3 * a] == b) p.bin_atom[m++] = a;
    }
}

// Q(k1,k2,k3) = sum_a q_a M4(w1 + t1) M4(w2 + t2) M4(w3 + t3), t = (base_a - k) mod K in [0, 4): a gather over the atoms
// of the base planes k1 .. k1+3 (grid dimensions >= 4, so t is unique)
__global__ void __launch_bounds__(PME_THREADS) pme_spread_kernel(PmeParams p) {
    const int g = blockIdx.x * PME_THREADS + threadIdx.x;
    if (g >= p.K1 * p.K2 * p.K3) return;
    const int k3 = g % p.K3, k2 = (g / p.K3) % p.K2, k1 = g / (p.K3 * p.K2);
    double s = 0.0;
    for (int t1 = 0; t1 < 4; t1++) {
        const int b = (k1 + t1) % p.K1;
        for (int m = p.bin_ptr[b]; m < p.bin_ptr[b + 1]; m++) {
            const int a = p.bin_atom[m];
            int t2 = p.base[3 * a + 1] - k2, t3 = p.base[3 * a + 2] - k3;
            if (t2 < 0) t2 += p.K2;
            if (t3 < 0) t3 += p.K3;
            if (t2 < 4 && t3 < 4) s += (double)p.q[a] * p.w[12 * a + t1] * p.w[12 * a + 4 + t2] * p.w[12 * a + 8 + t3];
        }
    }
    p.Q[g] = s;
}

// A(k1,k2,m3) = sum_k3 Q(k1,k2,k3) exp(-2 pi i m3 k3 / K3), m3 < H3
__global__ void __launch_bounds__(PME_THREADS) pme_dft3_kernel(PmeParams p) {
    const int g = blockIdx.x * PME_THREADS + threadIdx.x;
    if (g >= p.K1 * p.K2 * p.H3) return;
    const int m3 = g % p.H3, row = g / p.H3;
    const double* tw = p.tw + 2 * (p.K1 + p.K2);
    const double* q = p.Q + (size_t)row * p.K3;
    double re = 0.0, im = 0.0;
    for (int k = 0, j = 0; k < p.K3; k++, j = (j + m3 >= p.K3) ? j + m3 - p.K3 : j + m3) {
        re += q[k] * tw[2 * j];
        im -= q[k] * tw[2 * j + 1];
    }
    p.A[g] = make_double2(re, im);
}

// B(k1,m2,m3) = sum_k2 A(k1,k2,m3) exp(-2 pi i m2 k2 / K2)
__global__ void __launch_bounds__(PME_THREADS) pme_dft2_kernel(PmeParams p) {
    const int g = blockIdx.x * PME_THREADS + threadIdx.x;
    if (g >= p.K1 * p.K2 * p.H3) return;
    const int m3 = g % p.H3, m2 = (g / p.H3) % p.K2, k1 = g / (p.H3 * p.K2);
    const double* tw = p.tw + 2 * p.K1;
    const double2* a = p.A + (size_t)k1 * p.K2 * p.H3 + m3;
    double re = 0.0, im = 0.0;
    for (int k = 0, j = 0; k < p.K2; k++, j = (j + m2 >= p.K2) ? j + m2 - p.K2 : j + m2) {
        const double2 v = a[(size_t)k * p.H3];
        const double c = tw[2 * j], s = tw[2 * j + 1];
        re += v.x * c + v.y * s;
        im += v.y * c - v.x * s;
    }
    p.B[g] = make_double2(re, im);
}

// F(m) = sum_k1 B(k1,m2,m3) exp(-2 pi i m1 k1 / K1); partial[cta] = sum over the CTA's m of
// wgt exp(-pi^2 |m|^2 / beta^2) / |m|^2 B1 B2 B3 |F(m)|^2 (m = 0 left out; wgt 2 for the m3 whose mirror K3 - m3 is not stored)
__global__ void __launch_bounds__(PME_THREADS) pme_dft1_energy_kernel(PmeParams p) {
    __shared__ double red[PME_THREADS / 32];
    const int g = blockIdx.x * PME_THREADS + threadIdx.x;
    double e = 0.0;
    if (g < p.K1 * p.K2 * p.H3) {
        const int m3 = g % p.H3, m2 = (g / p.H3) % p.K2, m1 = g / (p.H3 * p.K2);
        const double2* b = p.B + (size_t)m2 * p.H3 + m3;
        const size_t stride = (size_t)p.K2 * p.H3;
        double re = 0.0, im = 0.0;
        for (int k = 0, j = 0; k < p.K1; k++, j = (j + m1 >= p.K1) ? j + m1 - p.K1 : j + m1) {
            const double2 v = b[k * stride];
            const double c = p.tw[2 * j], s = p.tw[2 * j + 1];
            re += v.x * c + v.y * s;
            im += v.y * c - v.x * s;
        }
        if (m1 | m2 | m3) {
            const double f1 = (m1 <= p.K1 / 2 ? m1 : m1 - p.K1) / p.L1, f2 = (m2 <= p.K2 / 2 ? m2 : m2 - p.K2) / p.L2;
            const double f3 = m3 / p.L3, msq = f1 * f1 + f2 * f2 + f3 * f3;
            const double wgt = (m3 == 0 || 2 * m3 == p.K3) ? 1.0 : 2.0;
            const double pb = 3.14159265358979323846 / p.beta64;
            e = wgt * exp(-pb * pb * msq) / msq * p.bmod[m1] * p.bmod[p.K1 + m2] * p.bmod[p.K1 + p.K2 + m3] * (re * re + im * im);
        }
    }
    const double t = pme_block_sum(e, red);
    if (threadIdx.x == 0) p.partial[blockIdx.x] = t;
}

template <typename PosT>
__global__ void __launch_bounds__(256) pme_direct_kernel(PmeParams p, const PosT* __restrict__ pos, float* __restrict__ ef) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int i = p.lo + warp;
    if (i >= p.hi) return;
    const float xi = (float)pos[3 * i], yi = (float)pos[3 * i + 1], zi = (float)pos[3 * i + 2];
    const float qi = p.q[i], si = p.sigma[i], ei = p.eps[i];
    const int x0 = p.excl_rowptr[i], x1 = p.excl_rowptr[i + 1];
    float fx = 0.f, fy = 0.f, fz = 0.f;
    double e_dir = 0.0, e_adj = 0.0, e_ex = 0.0, e_lj = 0.0, e_ljex = 0.0;
    for (int j = lane; j < p.n; j += 32) {
        if (j == i) continue;
        int a = x0, b = x1;                       // binary search of j among the excluded partners of i
        while (a < b) {
            const int m = (a + b) >> 1;
            if (p.excl_col[m] < j) a = m + 1; else b = m;
        }
        const bool excluded = a < x1 && p.excl_col[a] == j;
        // vec = pos[dst] - pos[src]   (pme.py:167-169)
        const float vx = xi - (float)pos[3 * j], vy = yi - (float)pos[3 * j + 1], vz = zi - (float)pos[3 * j + 2];
        const float d2 = vx * vx + vy * vy + vz * vz;
        const float d = sqrtf(d2);
        const float qq = p.q[j] * qi;
        if (excluded) e_adj += (double)(qq * erff(p.beta * d) / d);          // electro_adj, pme.py:90-96
        const bool inside = d2 < p.rc2;
        if (excluded == inside) continue;         // excluded inside the cutoff: P and X cancel
        // LJ (pme.py:175-180), plain Coulomb force (:203)
        const float sij = 0.5f * (p.sigma[j] + si) * 10.0f;
        const float eij = sqrtf(p.eps[j] * ei);
        const float t = sij * sij / d2;
        const float c6 = t * t * t, c12 = c6 * c6;
        const float elj = 4.0f * eij * (c12 - c6);
        const float f_lj = 24.0f * eij * (2.0f * c12 - c6) / d2;
        const float f_c = p.coulomb_k * p.q[j] * qi / d / d2;
        const float f = excluded ? -(f_lj + f_c) : f_lj + f_c;
        const double ec = (double)(qq * erfcf(p.beta * d) / d);            // electro_dir, pme.py:77-83
        fx += f * vx; fy += f * vy; fz += f * vz;
        if (excluded) { e_ex += ec; e_ljex += (double)elj; }
        else          { e_dir += ec; e_lj += (double)elj; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        fx += __shfl_xor_sync(0xffffffffu, fx, o); fy += __shfl_xor_sync(0xffffffffu, fy, o);
        fz += __shfl_xor_sync(0xffffffffu, fz, o);
        e_dir += __shfl_xor_sync(0xffffffffu, e_dir, o); e_adj += __shfl_xor_sync(0xffffffffu, e_adj, o);
        e_ex += __shfl_xor_sync(0xffffffffu, e_ex, o); e_lj += __shfl_xor_sync(0xffffffffu, e_lj, o);
        e_ljex += __shfl_xor_sync(0xffffffffu, e_ljex, o);
    }
    if (lane == 0) {
        ef[3 * i] += fx * p.kj_mol; ef[3 * i + 1] += fy * p.kj_mol; ef[3 * i + 2] += fz * p.kj_mol;
        double* ea = p.eatom + PME_NATOM * i;
        ea[PME_DIR] = e_dir; ea[PME_ADJ] = e_adj; ea[PME_EX] = e_ex; ea[PME_LJ] = e_lj; ea[PME_LJEX] = e_ljex;
    }
}

// terms (pair sums halved) and ef[3n] += E in eV, all sums in a fixed order
__global__ void __launch_bounds__(PME_THREADS) pme_energy_kernel(PmeParams p, int n_partial, float* __restrict__ ef) {
    __shared__ double red[PME_THREADS / 32];
    double c[PME_NATOM];
    for (int k = 0; k < PME_NATOM; k++) {
        double s = 0.0;
        for (int i = p.lo + threadIdx.x; i < p.hi; i += PME_THREADS) s += p.eatom[PME_NATOM * i + k];
        c[k] = pme_block_sum(s, red);
    }
    double s = 0.0;
    if (p.recip)
        for (int b = threadIdx.x; b < n_partial; b += PME_THREADS) s += p.partial[b];
    const double rec = pme_block_sum(s, red);
    if (threadIdx.x == 0) {
        double* t = p.terms;
        t[PT_DIR] = 0.5 * c[PME_DIR]; t[PT_ADJ] = -0.5 * c[PME_ADJ]; t[PT_EX] = 0.5 * c[PME_EX];
        t[PT_LJ] = 0.5 * c[PME_LJ]; t[PT_LJEX] = 0.5 * c[PME_LJEX];
        t[PT_REC] = p.recip ? rec / (2.0 * 3.14159265358979323846 * p.L1 * p.L2 * p.L3) : 0.0;
        t[PT_SLF] = p.recip ? p.slf : 0.0;
        t[PT_NEUTRAL] = p.recip ? p.neutral : 0.0;
        const double e_c = t[PT_REC] + t[PT_DIR] + t[PT_ADJ] + t[PT_SLF] + t[PT_NEUTRAL] - t[PT_EX];
        ef[3 * p.n] += (float)((p.k64 * e_c + t[PT_LJ] - t[PT_LJEX]) * p.kj64);
    }
}

inline int pme_partials(const PmeParams& p) { return (p.K1 * p.K2 * p.H3 + PME_THREADS - 1) / PME_THREADS; }

// The whole term on `st`: reciprocal chain (if p.recip, five launches), direct sums over [lo, hi), final energy.
template <typename PosT>
void pme_launch(const PmeParams& p, const PosT* pos, float* ef, cudaStream_t st) {
    if (p.recip) {
        const int ng = (p.K1 * p.K2 * p.K3 + PME_THREADS - 1) / PME_THREADS, nh = pme_partials(p);
        pme_bin_kernel<PosT><<<1, PME_THREADS, 0, st>>>(p, pos);
        pme_spread_kernel<<<ng, PME_THREADS, 0, st>>>(p);
        pme_dft3_kernel<<<nh, PME_THREADS, 0, st>>>(p);
        pme_dft2_kernel<<<nh, PME_THREADS, 0, st>>>(p);
        pme_dft1_energy_kernel<<<nh, PME_THREADS, 0, st>>>(p);
    }
    if (p.hi > p.lo) pme_direct_kernel<PosT><<<(p.hi - p.lo + 7) / 8, 256, 0, st>>>(p, pos, ef);
    pme_energy_kernel<<<1, PME_THREADS, 0, st>>>(p, pme_partials(p), ef);
}

}  // namespace vb
