// kernels.cuh — sm_100a device code for Wafer's imaginary-time FDTD hot path.
//
// Reference semantics (file:line under the Libbum/Wafer tree):
//   sweep         src/grid.rs:567-673   psi' = psi*A + ((B*dt)*S)/den, S = 3/5/7-point Laplacian sum
//   observables   src/grid.rs:303-445
//   norm/GS       src/grid.rs:454-492
//   A,B           src/potential.rs:101-110
//
// Arithmetic contract: every product/sum below uses the round-to-nearest intrinsics (__dmul_rn, __dadd_rn,
// __dsub_rn, __ddiv_rn, __dsqrt_rn), which nvcc never contracts into FMAs, in exactly the reference's
// left-to-right association.  The sweep is therefore BIT-IDENTICAL to the reference's CPU arithmetic.
//
// Device layout of a field ("slab"): planes i in [-gx, L+gx) of (ny + 2e) rows of zp doubles,
//   offset(i,j,k) = ((i+gx)*yp + (j+e))*zp + k,   yp = ny+2e, zp = round_up(nz+2e, 16),
// rows are 128-byte aligned, interior column 0 sits at a row start.  The y ghost rows, the z pad columns
// [nz, zp) and the x ghost planes outside the global lattice hold the Dirichlet zeros of the reference's
// padding ring (config.rs:597-622) and are never written by any kernel, so a z neighbour k-1 at k=0 reads the
// (zero) pad tail of the previous row and no kernel needs boundary predication on loads.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace wafer {

struct Geom {
    int L;            // owned x planes
    int ny, nz;       // work rows / columns
    int e;            // stencil extent 1|2|3
    int gx;           // x ghost depth (>= e)
    int yp, zp;       // rows per plane, row pitch (doubles)
    long long plane;  // yp*zp
    long long gnx, gny, gnz;  // global work sizes (r2 centre, potentials)
    long long x0;     // global work index of owned plane 0
    __host__ __device__ long long off(int i, int j, int k) const {
        return ((long long)(i + gx) * yp + (j + e)) * zp + k;
    }
    __host__ __device__ long long total() const { return (long long)(L + 2 * gx) * plane; }
};

#define D_MUL __dmul_rn
#define D_ADD __dadd_rn
#define D_SUB __dsub_rn
#define D_DIV __ddiv_rn

// ---------------------------------------------------------------------------------------------------------
// Laplacian sum in the reference's association order.  p[m-1]/m_[m-1] hold the +m / -m neighbours per axis.
template <int E>
struct Lap;

template <>
struct Lap<1> {  // grid.rs:582-588 / 326-331
    __device__ __forceinline__ static double sum(const double* xp, const double* xm, const double* yp,
                                                 const double* ym, const double* zp, const double* zm, double w) {
        double s = D_ADD(xp[0], xm[0]);
        s = D_ADD(s, yp[0]);
        s = D_ADD(s, ym[0]);
        s = D_ADD(s, zp[0]);
        s = D_ADD(s, zm[0]);
        return D_SUB(s, D_MUL(6., w));
    }
};

template <>
struct Lap<2> {  // grid.rs:608-620 / 350-362
    __device__ __forceinline__ static double axis(double s, const double* p, const double* m) {
        s = D_SUB(s, p[1]);
        s = D_ADD(s, D_MUL(16., p[0]));
        s = D_ADD(s, D_MUL(16., m[0]));
        return D_SUB(s, m[1]);
    }
    __device__ __forceinline__ static double sum(const double* xp, const double* xm, const double* yp,
                                                 const double* ym, const double* zp, const double* zm, double w) {
        double s = -xp[1];
        s = D_ADD(s, D_MUL(16., xp[0]));
        s = D_ADD(s, D_MUL(16., xm[0]));
        s = D_SUB(s, xm[1]);
        s = axis(s, yp, ym);
        s = axis(s, zp, zm);
        return D_SUB(s, D_MUL(90., w));
    }
};

template <>
struct Lap<3> {  // grid.rs:642-659 / 382-399
    __device__ __forceinline__ static double axis(double s, const double* p, const double* m) {
        s = D_ADD(s, D_MUL(2., p[2]));
        s = D_SUB(s, D_MUL(27., p[1]));
        s = D_ADD(s, D_MUL(270., p[0]));
        s = D_ADD(s, D_MUL(270., m[0]));
        s = D_SUB(s, D_MUL(27., m[1]));
        return D_ADD(s, D_MUL(2., m[2]));
    }
    __device__ __forceinline__ static double sum(const double* xp, const double* xm, const double* yp,
                                                 const double* ym, const double* zp, const double* zm, double w) {
        double s = D_SUB(D_MUL(2., xp[2]), D_MUL(27., xp[1]));
        s = D_ADD(s, D_MUL(270., xp[0]));
        s = D_ADD(s, D_MUL(270., xm[0]));
        s = D_SUB(s, D_MUL(27., xm[1]));
        s = D_ADD(s, D_MUL(2., xm[2]));
        s = axis(s, yp, ym);
        s = axis(s, zp, zm);
        return D_SUB(s, D_MUL(1470., w));
    }
};

// potential.rs:104-110, from V on the fly:  b = 1/(1 + dt*v/2),  a = (1 - dt*v/2)*b
__device__ __forceinline__ void ab_from_v(double v, double dt, double& a, double& b) {
    const double h = D_MUL(D_MUL(dt, v), 0.5);  // (dt*v)/2: halving is exact, identical to the division
    b = D_DIV(1., D_ADD(1., h));
    a = D_MUL(D_SUB(1., h), b);
}

// grid.rs:580-589:  (w*pa) + (((pb*dt)*S)/den)
__device__ __forceinline__ double update(double w, double a, double b, double dt, double s, double den) {
    return D_ADD(D_MUL(w, a), D_DIV(D_MUL(D_MUL(b, dt), s), den));
}

// ---------------------------------------------------------------------------------------------------------
// Deterministic block reduction of NS running sums; thread 0 writes partials[s*nblocks + bid].
template <int NS>
__device__ __forceinline__ void block_reduce_store(double (&v)[NS], double* __restrict__ partials, int nblocks,
                                                   int bid) {
    __shared__ double red[NS][32];
    const int tid = threadIdx.x + blockDim.x * (threadIdx.y + blockDim.y * threadIdx.z);
    const int nthreads = blockDim.x * blockDim.y * blockDim.z;
    const int lane = tid & 31, warp = tid >> 5, nwarps = (nthreads + 31) >> 5;
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        double x = v[s];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x = D_ADD(x, __shfl_down_sync(0xffffffffu, x, o));
        if (lane == 0) red[s][warp] = x;
    }
    __syncthreads();
    if (warp == 0) {
#pragma unroll
        for (int s = 0; s < NS; ++s) {
            double x = lane < nwarps ? red[s][lane] : 0.0;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) x = D_ADD(x, __shfl_down_sync(0xffffffffu, x, o));
            if (lane == 0) partials[(long long)s * nblocks + bid] = x;
        }
    }
}

// One CTA sums partials[s][0..nblocks) in a fixed order -> out[s]: run-to-run deterministic, no f64 atomics.
template <int NS>
__global__ void __launch_bounds__(1024) finalize_kernel(const double* __restrict__ partials, int nblocks,
                                                        double* __restrict__ out) {
    double v[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) {
        double acc = 0.0;
        for (int i = threadIdx.x; i < nblocks; i += blockDim.x) acc = D_ADD(acc, partials[(long long)s * nblocks + i]);
        v[s] = acc;
    }
    __shared__ double fin[NS];
    block_reduce_store<NS>(v, fin, 1, 0);
    __syncthreads();
    if (threadIdx.x < NS) out[threadIdx.x] = fin[threadIdx.x];
}

// ---------------------------------------------------------------------------------------------------------
// Plain register-queue sweep ("simple" variant): CTA = SW_BX x SW_BY threads, each thread owns two adjacent
// z columns of one row and marches along x with a (2E+1)-deep register queue; y/z neighbours come through L1.
// (measured on B200, profiles/: letting ptxas pick the register count — 58..64 — beats forcing 5-6 CTAs/SM for
// the 5/7-point and norm-fused variants; only the plain 3-point variant gains from 40 registers, and that case is
// served by the time-tiled kernel anyway)
constexpr int SW_BX = 32, SW_BY = 8, SW_XCH = 32;

template <int E, bool ONFLY, bool NORM>
__global__ void __launch_bounds__(SW_BX * SW_BY)
    sweep_simple_kernel(const double* __restrict__ cur, double* __restrict__ nxt, const double* __restrict__ fa,
                        const double* __restrict__ fb, Geom g, int xb, int xe, double dt, double den,
                        double* __restrict__ partials) {
    const int k = (blockIdx.x * SW_BX + threadIdx.x) * 2;
    const int j = blockIdx.y * SW_BY + threadIdx.y;
    const int i0 = xb + blockIdx.z * SW_XCH;
    const int i1 = min(i0 + SW_XCH, xe);
    const bool active = (j < g.ny) && (k < g.nz);
    const bool second = (k + 1 < g.nz);
    double acc[1] = {0.0};
    if (active) {
        const long long P = g.plane;
        const int zp_ = g.zp;
        const double* c = cur + g.off(i0, j, k);
        double2 q[2 * E + 1];
#pragma unroll
        for (int m = 0; m < 2 * E; ++m) q[m] = *reinterpret_cast<const double2*>(c + (long long)(m - E) * P);
        for (int i = i0; i < i1; ++i) {
            q[2 * E] = *reinterpret_cast<const double2*>(c + (long long)E * P);
            const double2 w = q[E];
            double xp0[E], xm0[E], xp1[E], xm1[E], yp0[E], ym0[E], yp1[E], ym1[E], zp0[E], zm0[E], zp1[E], zm1[E];
#pragma unroll
            for (int m = 1; m <= E; ++m) {
                xp0[m - 1] = q[E + m].x; xp1[m - 1] = q[E + m].y;
                xm0[m - 1] = q[E - m].x; xm1[m - 1] = q[E - m].y;
                const double2 a = *reinterpret_cast<const double2*>(c + (long long)m * zp_);
                const double2 b = *reinterpret_cast<const double2*>(c - (long long)m * zp_);
                yp0[m - 1] = a.x; yp1[m - 1] = a.y;
                ym0[m - 1] = b.x; ym1[m - 1] = b.y;
            }
            // z neighbours: columns k-E..k-1 and k+2..k+1+E from memory, the pair itself from registers
            double zl[E], zr[E];
#pragma unroll
            for (int m = 0; m < E; ++m) { zl[m] = c[-1 - m]; zr[m] = c[2 + m]; }
            zp0[0] = w.y; zm1[0] = w.x;
#pragma unroll
            for (int m = 1; m <= E; ++m) {
                zm0[m - 1] = zl[m - 1];
                zp1[m - 1] = zr[m - 1];
                if (m >= 2) { zp0[m - 1] = zr[m - 2]; zm1[m - 1] = zl[m - 2]; }
            }
            const double s0 = Lap<E>::sum(xp0, xm0, yp0, ym0, zp0, zm0, w.x);
            const double s1 = Lap<E>::sum(xp1, xm1, yp1, ym1, zp1, zm1, w.y);
            double a0, b0, a1, b1;
            const long long o = c - cur;
            if (ONFLY) {
                const double2 v = *reinterpret_cast<const double2*>(fa + o);
                ab_from_v(v.x, dt, a0, b0);
                ab_from_v(v.y, dt, a1, b1);
            } else {
                const double2 a = *reinterpret_cast<const double2*>(fa + o);
                const double2 b = *reinterpret_cast<const double2*>(fb + o);
                a0 = a.x; a1 = a.y; b0 = b.x; b1 = b.y;
            }
            double2 r;
            r.x = update(w.x, a0, b0, dt, s0, den);
            r.y = second ? update(w.y, a1, b1, dt, s1, den) : 0.0;  // pad column stays 0
            *reinterpret_cast<double2*>(nxt + o) = r;
            if (NORM) acc[0] = D_ADD(acc[0], D_ADD(D_MUL(r.x, r.x), D_MUL(r.y, r.y)));
#pragma unroll
            for (int m = 0; m < 2 * E; ++m) q[m] = q[m + 1];
            c += P;
        }
    }
    if (NORM) {
        const int nb = gridDim.x * gridDim.y * gridDim.z;
        const int bid = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
        block_reduce_store<1>(acc, partials, nb, bid);
    }
}

// ---------------------------------------------------------------------------------------------------------
// compute_observables (grid.rs:303-445): one pass, four sums.  POTSUB: 0 none, 1 scalar, 2 array.
// partial sums: [0] energy integrand ((v*w)*w) - ((w*S)/den), [1] w*w, [2] (w*w)*potsub, [3] (w*w)*r2(work idx)
template <int E, int POTSUB>
__global__ void __launch_bounds__(SW_BX* SW_BY)
    observables_kernel(const double* __restrict__ cur, const double* __restrict__ v, const double* __restrict__ potsub_arr,
                       double potsub, Geom g, double den, double* __restrict__ partials) {
    const int k = blockIdx.x * SW_BX + threadIdx.x;
    const int j = blockIdx.y * SW_BY + threadIdx.y;
    const int i0 = blockIdx.z * SW_XCH;
    const int i1 = min(i0 + SW_XCH, g.L);
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    if (j < g.ny && k < g.nz) {
        const long long P = g.plane;
        const int zp_ = g.zp;
        const double* c = cur + g.off(i0, j, k);
        const double cy = D_SUB((double)j, D_DIV(D_ADD((double)g.gny, 1.), 2.));
        const double cz = D_SUB((double)k, D_DIV(D_ADD((double)g.gnz, 1.), 2.));
        const double yz2 = D_MUL(cy, cy);
        const double zz2 = D_MUL(cz, cz);
        double q[2 * E + 1];
#pragma unroll
        for (int m = 0; m < 2 * E; ++m) q[m] = c[(long long)(m - E) * P];
        for (int i = i0; i < i1; ++i) {
            q[2 * E] = c[(long long)E * P];
            const double w = q[E];
            double xp[E], xm[E], yp[E], ym[E], zp[E], zm[E];
#pragma unroll
            for (int m = 1; m <= E; ++m) {
                xp[m - 1] = q[E + m]; xm[m - 1] = q[E - m];
                yp[m - 1] = c[(long long)m * zp_]; ym[m - 1] = c[-(long long)m * zp_];
                zp[m - 1] = c[m]; zm[m - 1] = c[-m];
            }
            const double s = Lap<E>::sum(xp, xm, yp, ym, zp, zm, w);
            const long long o = c - cur;
            const double en = D_SUB(D_MUL(D_MUL(v[o], w), w), D_DIV(D_MUL(w, s), den));
            const double ww = D_MUL(w, w);
            acc[0] = D_ADD(acc[0], en);
            acc[1] = D_ADD(acc[1], ww);
            if (POTSUB == 1) acc[2] = D_ADD(acc[2], D_MUL(ww, potsub));
            if (POTSUB == 2) acc[2] = D_ADD(acc[2], D_MUL(ww, potsub_arr[o]));
            // potential.rs:366-371 on GLOBAL work indices: (dx*dx + dy*dy) + dz*dz
            const double cx = D_SUB((double)(g.x0 + i), D_DIV(D_ADD((double)g.gnx, 1.), 2.));
            const double r2 = D_ADD(D_ADD(D_MUL(cx, cx), yz2), zz2);
            acc[3] = D_ADD(acc[3], D_MUL(ww, r2));
#pragma unroll
            for (int m = 0; m < 2 * E; ++m) q[m] = q[m + 1];
            c += P;
        }
    }
    const int nb = gridDim.x * gridDim.y * gridDim.z;
    const int bid = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
    block_reduce_store<4>(acc, partials, nb, bid);
}

// ---------------------------------------------------------------------------------------------------------
// Flat element-wise passes over a whole slab buffer (ghost planes included, so neighbouring ranks keep
// bit-identical ghost copies without a halo exchange); reductions count only [own_b, own_e).
// All work on double2 (buffers are 128-byte aligned and a multiple of 16 doubles long).
constexpr int EW_THREADS = 256;

// ---------------------------------------------------------------------------------------------------------
// Gram-Schmidt in two passes instead of 2k (grid.rs:477-492 is k sequential "dot, then axpy" sweeps):
//   pass 1  dots_kernel<K>      raw_i = sum q_i * psi over the owned planes, all K stored states at once (or fused
//                               into the sweep, sweep_tma1.cuh NRED)
//   scalars gs_coeff_kernel     s_0 = d_0,  s_i = d_i - sum_{j<i} G_ij s_j   with d_i = raw_i / sqrt(norm2) and the
//                               Gram matrix G_ij = <q_i, q_j> of the stored states (measured when a state is pushed)
//   pass 2  project_kernel<K>   psi = ((psi / sqrt(norm2)) - q_0 s_0) - q_1 s_1 ...   element-wise in the reference's order
// In exact arithmetic s_i IS the modified-Gram-Schmidt overlap <q_i, psi - sum_{j<i} q_j s_j> of the reference, for
// arbitrary (also non-orthogonal) stored states; in floating point it differs from it like two summation orders do.
constexpr int GS_GROUP = 4;  // stored states handled per pass
struct LowerPtrs {
    const double* q[GS_GROUP];
};

template <int K>
__global__ void __launch_bounds__(EW_THREADS)
    dots_kernel(const double* __restrict__ psi, LowerPtrs lw, long long own_b2, long long own_e2, double* __restrict__ partials) {
    double acc[K];
#pragma unroll
    for (int k = 0; k < K; ++k) acc[k] = 0.0;
    const double2* p2 = reinterpret_cast<const double2*>(psi);
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = own_b2 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < own_e2; i += stride) {
        const double2 w = p2[i];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const double2 q = __ldg(reinterpret_cast<const double2*>(lw.q[k]) + i);
            acc[k] = D_ADD(acc[k], D_ADD(D_MUL(q.x, w.x), D_MUL(q.y, w.y)));
        }
    }
    block_reduce_store<K>(acc, partials, gridDim.x, blockIdx.x);
}

// psi = psi / sqrt(*norm2_ptr) (NORMALISE, grid.rs:465-468: a true division), then psi -= q_k * coef[k] for k = 0..K-1 in
// order (grid.rs:488-490), over the whole slab buffer (ghost planes included: every rank applies the same scalars, so
// neighbouring ranks keep bit-identical ghost copies without a halo exchange)
template <int K, bool NORMALISE>
__global__ void __launch_bounds__(EW_THREADS)
    project_kernel(double* __restrict__ psi, long long n2, const double* __restrict__ norm2_ptr, LowerPtrs lw,
                   const double* __restrict__ coef) {
    double norm = 1.0, s[K > 0 ? K : 1];
    if (NORMALISE) norm = __dsqrt_rn(*norm2_ptr);
#pragma unroll
    for (int k = 0; k < K; ++k) s[k] = coef[k];
    double2* p2 = reinterpret_cast<double2*>(psi);
    const long long stride = (long long)gridDim.x * blockDim.x;
    // U independent 16-byte loads per stream in flight per thread before the first use (a read + write streaming pass
    // with one load per thread in flight reached 58 % of the copy peak, ncu r2n)
    constexpr int U = K >= 3 ? 2 : 4;
    for (long long i0 = (long long)blockIdx.x * blockDim.x + threadIdx.x; i0 < n2; i0 += U * stride) {
        double2 w[U], q[U][K > 0 ? K : 1];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long i = i0 + u * stride;
            if (i < n2) {
                w[u] = p2[i];
#pragma unroll
                for (int k = 0; k < K; ++k) q[u][k] = __ldg(reinterpret_cast<const double2*>(lw.q[k]) + i);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long i = i0 + u * stride;
            if (i < n2) {
                double2 x = w[u];
                if (NORMALISE) { x.x = D_DIV(x.x, norm); x.y = D_DIV(x.y, norm); }
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    x.x = D_SUB(x.x, D_MUL(q[u][k].x, s[k]));
                    x.y = D_SUB(x.y, D_MUL(q[u][k].y, s[k]));
                }
                p2[i] = x;
            }
        }
    }
}

// One CTA: (REDUCE) fixed-order sums of `nrows` rows of per-CTA partials -> raw[0..nrows); (COEF) the Gram-Schmidt
// coefficients from raw.  Split in two launches only when an all-reduce over ranks sits between them.
//   raw layout: raw[dot0 + i] = sum q_i psi for i < k; norm2_ptr (may be raw[0] or the observables' norm2 or NULL)
template <bool REDUCE, bool COEF>
__global__ void __launch_bounds__(1024)
    gs_coeff_kernel(const double* __restrict__ partials, int nblocks, int nrows, double* __restrict__ raw, int k,
                    const double* __restrict__ dots, const double* __restrict__ norm2_ptr, const double* __restrict__ gram,
                    int gram_ld, double* __restrict__ coef) {
    if (REDUCE) {
        __shared__ double fin[1];
        for (int r = 0; r < nrows; ++r) {
            double v[1] = {0.0};
            for (int i = threadIdx.x; i < nblocks; i += blockDim.x) v[0] = D_ADD(v[0], partials[(long long)r * nblocks + i]);
            __syncthreads();  // the reduction scratch of the previous row is free again
            block_reduce_store<1>(v, fin, 1, 0);
            __syncthreads();
            if (threadIdx.x == 0) raw[r] = fin[0];
        }
        __syncthreads();
    }
    if (COEF && threadIdx.x == 0) {
        const double norm = norm2_ptr ? __dsqrt_rn(*norm2_ptr) : 1.0;
        for (int i = 0; i < k; ++i) {
            double s = norm2_ptr ? D_DIV(dots[i], norm) : dots[i];
            for (int j = 0; j < i; ++j) s = D_SUB(s, D_MUL(gram[(long long)i * gram_ld + j], coef[j]));
            coef[i] = s;
        }
    }
}

// sum of psi^2 over the owned planes (pads and ghost rows are zero, so this equals the work-area norm2)
__global__ void __launch_bounds__(EW_THREADS)
    norm2_kernel(const double* __restrict__ psi, long long own_b2, long long own_e2, double* __restrict__ partials) {
    double acc[1] = {0.0};
    const double2* p2 = reinterpret_cast<const double2*>(psi);
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = own_b2 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < own_e2; i += stride) {
        const double2 w = p2[i];
        acc[0] = D_ADD(acc[0], D_ADD(D_MUL(w.x, w.x), D_MUL(w.y, w.y)));
    }
    block_reduce_store<1>(acc, partials, gridDim.x, blockIdx.x);
}

// h = (dt*v)/2 over a whole slab buffer: the first two operations of potential.rs:104-110, taken out of the time-tiled sweep
__global__ void __launch_bounds__(EW_THREADS)
    build_h_kernel(const double* __restrict__ v, double* __restrict__ h, long long n, double dt) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) h[i] = D_MUL(D_MUL(dt, v[i]), 0.5);
}

// A,B arrays from V over a whole slab buffer (potential.rs:104-110)
__global__ void __launch_bounds__(EW_THREADS)
    build_ab_kernel(const double* __restrict__ v, double* __restrict__ a, double* __restrict__ b, long long n, double dt) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        double aa, bb;
        ab_from_v(v[i], dt, aa, bb);
        a[i] = aa;
        b[i] = bb;
    }
}

// ---------------------------------------------------------------------------------------------------------
// Host layout <-> device layout, staged through a small bounce buffer.  `stg` holds padded (or work-sized) host
// planes [sp0, sp1) of the reference array, py x pz doubles each.  Device plane i in [-gx, L+gx) maps to host
// plane gp = x0 + i + hoff (hoff = e for padded arrays, 0 for work-sized ones); planes outside [sp0, sp1) and
// everything outside the lattice are written as zero.  One launch handles device planes [i0, i1).
// WORKSIZED: host array has no ring (nx,ny,nz) — used for the pot_sub array.
// ring_flag is set when a ring entry of the source is non-zero (CHECK).
template <bool CHECK>
__global__ void __launch_bounds__(256)
    unpack_kernel(const double* __restrict__ stg, double* __restrict__ dev, Geom g, int i0, int i1, long long sp0,
                  long long sp1, int worksized, int* __restrict__ ring_flag) {
    const int py = worksized ? g.ny : g.ny + 2 * g.e, pz = worksized ? g.nz : g.nz + 2 * g.e;
    const int hoff = worksized ? 0 : g.e;
    const long long rows = (long long)(i1 - i0) * g.yp;
    for (long long r = blockIdx.x; r < rows; r += gridDim.x) {
        const int i = i0 + (int)(r / g.yp), jr = (int)(r % g.yp);  // jr = j + e
        const long long gp = g.x0 + i + hoff;                      // host plane index
        const bool plane_ok = gp >= sp0 && gp < sp1;
        const bool x_inside = (g.x0 + i) >= 0 && (g.x0 + i) < g.gnx;
        const bool y_inside = jr >= g.e && jr < g.ny + g.e;
        const int hj = jr - g.e + hoff;
        double* drow = dev + ((long long)(i + g.gx) * g.yp + jr) * g.zp;
        const double* hrow = stg + ((gp - sp0) * py + hj) * (long long)pz;
        for (int k = threadIdx.x; k < g.zp; k += blockDim.x) {
            double val = 0.0;
            if (plane_ok && x_inside && y_inside && k < g.nz) val = hrow[k + hoff];
            drow[k] = val;
        }
        if (CHECK && plane_ok && !worksized && hj >= 0 && hj < py) {
            // ring entries of this host row: whole row if x or y is in the ring, else the 2e end columns
            if (!x_inside || !y_inside) {
                for (int k = threadIdx.x; k < pz; k += blockDim.x)
                    if (hrow[k] != 0.0) *ring_flag = 1;
            } else if (threadIdx.x < 2 * g.e) {
                const int k = threadIdx.x < g.e ? threadIdx.x : pz - 2 * g.e + threadIdx.x;
                if (hrow[k] != 0.0) *ring_flag = 1;
            }
        }
    }
}

// device -> host layout for padded planes [sp0, sp1) into the bounce buffer (ring written as zeros)
__global__ void __launch_bounds__(256)
    pack_kernel(const double* __restrict__ dev, double* __restrict__ stg, Geom g, long long sp0, long long sp1,
                int worksized) {
    const int py = worksized ? g.ny : g.ny + 2 * g.e, pz = worksized ? g.nz : g.nz + 2 * g.e;
    const int hoff = worksized ? 0 : g.e;
    const long long rows = (sp1 - sp0) * py;
    for (long long r = blockIdx.x; r < rows; r += gridDim.x) {
        const long long gp = sp0 + r / py;
        const int hj = (int)(r % py);
        const long long gi = gp - hoff;  // global work x
        const int j = hj - hoff;
        const bool inside = gi >= 0 && gi < g.gnx && j >= 0 && j < g.ny;
        const double* drow = inside ? dev + g.off((int)(gi - g.x0), j, 0) : nullptr;
        double* hrow = stg + r * pz;
        for (int k = threadIdx.x; k < pz; k += blockDim.x) {
            const int kk = k - hoff;
            hrow[k] = (inside && kk >= 0 && kk < g.nz) ? drow[kk] : 0.0;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Position-sensitive, order-independent checksum of the work-area sites of local planes [xb, xe): every site
// contributes mix64(bits(psi) + golden * (global linear work index + 1)); the contributions are combined with
// wrapping integer addition (out[0]) and xor (out[1]), both associative and commutative, so the result does not
// depend on how the lattice is cut into slabs, tiles or threads.  Two slab-decomposed ranks and one single-GPU
// context therefore agree on the checksum of the same planes iff the planes hold the same bits at the same sites.
__device__ __forceinline__ unsigned long long mix64(unsigned long long z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__global__ void __launch_bounds__(256)
    checksum_kernel(const double* __restrict__ psi, Geom g, int xb, int xe, unsigned long long* __restrict__ out) {
    unsigned long long s = 0, x = 0;
    const long long rows = (long long)(xe - xb) * g.ny;
    for (long long r = blockIdx.x; r < rows; r += gridDim.x) {
        const int i = xb + (int)(r / g.ny), j = (int)(r % g.ny);
        const double* row = psi + g.off(i, j, 0);
        const unsigned long long base = ((unsigned long long)(g.x0 + i) * (unsigned long long)g.gny + (unsigned long long)j) * (unsigned long long)g.gnz;
        for (int k = threadIdx.x; k < g.nz; k += blockDim.x) {
            const unsigned long long h = mix64((unsigned long long)__double_as_longlong(row[k]) + 0x9E3779B97F4A7C15ull * (base + k + 1));
            s += h;
            x ^= h;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_down_sync(0xffffffffu, s, o);
        x ^= __shfl_down_sync(0xffffffffu, x, o);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(out, s);      // integer atomics: exact and order independent
        atomicXor(out + 1, x);
    }
}

// busy-wait for `ns` nanoseconds (fault injection for the multi-GPU ordering tests: wafer_debug_halo_delay)
__global__ void spin_kernel(unsigned long long ns) {
    unsigned long long t0, t1;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t0));
    do {
        __nanosleep(1000);
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t1));
    } while (t1 - t0 < ns);
}

}  // namespace wafer
