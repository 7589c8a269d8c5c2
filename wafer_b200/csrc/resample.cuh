// resample.cuh — fill_data (input.rs:149-176) / read_csv (input.rs:641-657) on the device: the array of an input file
// (dense C order (sx, sy, sz), z contiguous, as parsed) is resampled onto the work area of a field, bit-identical to the
// host restatement formats.hpp embed_work / trilerp_resize (interpolation, input.rs:667-716):
//   * every axis has a basis of b = n + 2e points (the PADDED size) of which the work area takes the first n;
//   * look = 0. + step * (double)i, step = (double)(s-1) / ((double)b - 1.) (0 when b <= 1), ndarray 0.11's linspace;
//   * bracket (i0, i1 = i0 + 1) around look, weight d = (look - i0) / (i1 - i0), a division by exactly 1.0;
//   * op(c0, c1, d) = c0*(1-d) + c1*d, x first (c00, c01, c10, c11), then y, then z.
// Every operation is a _rn intrinsic: nothing contracts into an FMA whatever the build flags.
#pragma once

#include "kernels.cuh"

namespace wafer {

#ifdef __CUDA_ARCH__
#define RS_MUL __dmul_rn
#define RS_ADD __dadd_rn
#define RS_SUB __dsub_rn
#define RS_DIV __ddiv_rn
#else  // host: one IEEE operation per call, so the host plan and the device agree on every bracket
inline double RS_MUL(double a, double b) { return a * b; }
inline double RS_ADD(double a, double b) { return a + b; }
inline double RS_SUB(double a, double b) { return a - b; }
inline double RS_DIV(double a, double b) { return a / b; }
#endif

// Output index i of a basis of b points over a source axis of s >= 2 points: lower bracket i0 (upper = i0 + 1) and
// weight d.  The reference scans xx = 0 .. s-2 for the first xx > look, else takes (s-2, s-1); for every finite
// look >= 0 that first xx is floor(look) + 1, which gives the closed form below (integer looks and a look rounded just
// above s-1 included).
__host__ __device__ inline void rs_bracket(long long s, long long b, long long i, long long* i0, double* d) {
    const double step = b > 1 ? RS_DIV((double)(s - 1), RS_SUB((double)b, 1.)) : 0.;
    const double look = RS_ADD(0., RS_MUL(step, (double)i));
    long long lo = (long long)floor(look);  // i1 - 1
    if (lo + 1 >= s - 1) lo = s - 2;
    *i0 = lo;
    *d = RS_SUB(look, (double)lo);  // (look - i0) / (i1 - i0): the divisor is exactly 1.0
}

__device__ __forceinline__ double rs_op(double c0, double c1, double d) {
    return RS_ADD(RS_MUL(c0, RS_SUB(1., d)), RS_MUL(c1, d));
}

constexpr int RS_THREADS = 256;
constexpr int RS_ZTILE = 1024;  // z columns per CTA (blockIdx.y): their brackets and weights live in shared memory

// Device planes [i0, i1) of the slab (ghost planes included; the caller passes planes inside the global lattice only),
// work area only: ring, y ghost rows, z pad columns stay as they are (+0).  `src` holds source x-planes [sp0, ...) of
// the (sx, sy, sz) array.  COPY: the source has the work size and is copied straight in (csv, input.rs:641-650).
// Grid: x strides over the rows (plane, y) of the range, y over z tiles of RS_ZTILE columns.  Stores are coalesced
// along z; the 8 source reads of a site come through L1 / L2.
template <bool COPY>
__global__ void __launch_bounds__(RS_THREADS)
    resample_kernel(double* __restrict__ dst, Geom g, const double* __restrict__ src, long long sp0, long long sx,
                    long long sy, long long sz, int i0, int i1) {
    __shared__ int zlo[COPY ? 1 : RS_ZTILE];
    __shared__ double zw[COPY ? 1 : RS_ZTILE];
    const long long bx = g.gnx + 2 * g.e, by = g.gny + 2 * g.e, bz = g.gnz + 2 * g.e;
    const long long rows = (long long)(i1 - i0) * g.ny, ps = sy * sz;
    for (int k0 = blockIdx.y * RS_ZTILE; k0 < g.nz; k0 += gridDim.y * RS_ZTILE) {
        const int k1 = min(g.nz, k0 + RS_ZTILE);
        if (!COPY) {
            __syncthreads();  // the previous tile's table is no longer read
            for (int k = k0 + threadIdx.x; k < k1; k += blockDim.x) {
                long long lo;
                double d;
                rs_bracket(sz, bz, k, &lo, &d);
                zlo[k - k0] = (int)lo;
                zw[k - k0] = d;
            }
            __syncthreads();
        }
        for (long long r = blockIdx.x; r < rows; r += gridDim.x) {
            const int i = i0 + (int)(r / g.ny), j = (int)(r % g.ny);
            const long long gi = g.x0 + i;
            double* row = dst + g.off(i, j, 0);
            if (COPY) {
                const double* s = src + ((gi - sp0) * sy + j) * sz;
                for (int k = k0 + threadIdx.x; k < k1; k += blockDim.x) row[k] = s[k];
                continue;
            }
            long long x0, y0;
            double xd, yd;
            rs_bracket(sx, bx, gi, &x0, &xd);
            rs_bracket(sy, by, j, &y0, &yd);
            const double* r00 = src + ((x0 - sp0) * sy + y0) * sz;  // (x0, y0)
            const double* r10 = r00 + ps;                           // (x1, y0)
            const double* r01 = r00 + sz;                           // (x0, y1)
            const double* r11 = r10 + sz;                           // (x1, y1)
            for (int k = k0 + threadIdx.x; k < k1; k += blockDim.x) {
                const int z0 = zlo[k - k0], z1 = z0 + 1;
                const double zd = zw[k - k0];
                const double c00 = rs_op(r00[z0], r10[z0], xd);
                const double c01 = rs_op(r00[z1], r10[z1], xd);
                const double c10 = rs_op(r01[z0], r11[z0], xd);
                const double c11 = rs_op(r01[z1], r11[z1], xd);
                const double c0 = rs_op(c00, c10, yd), c1 = rs_op(c01, c11, yd);
                row[k] = rs_op(c0, c1, zd);
            }
        }
    }
}

}  // namespace wafer
