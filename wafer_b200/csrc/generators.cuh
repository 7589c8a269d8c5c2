// generators.cuh — device-side potential and initial-condition generators, so that 1024^3..2048^3 runs never
// materialise a host array.  Formulas follow the reference at PADDED indices (file:line under Libbum/Wafer):
//   potential()              src/potential.rs:188-319
//   calculate_r2             src/potential.rs:366-371
//   alphas / mu              src/potential.rs:374-398   (host, constants of FullCornell)
//   Poschl-Teller script     gen_potential.py:45-60      (kind 100; fills the work area, ring 0)
//   initial conditions       src/config.rs:586-595, 650-683
// Built with -fmad=false: +,-,*,/ and sqrt are IEEE round-to-nearest in the reference's association order, so
// every kind that uses only those (NoPotential, Cube, QuadWell, Coulomb, ComplexCoulomb, ElipticalCoulomb,
// SimpleCornell, Harmonic, ComplexHarmonic, Dodecahedron; Constant/Boolean IC) is bit-identical to the
// reference.  Periodic (sin), FullCornell (exp), Poschl-Teller (cosh) and the Coulomb IC (exp) use CUDA's libm,
// which may differ from the host libm by an ulp.
#pragma once
#include <cmath>

#include "kernels.cuh"

namespace wafer {

enum PotKind {
    POT_NONE = 0, POT_CUBE, POT_QUADWELL, POT_PERIODIC, POT_COULOMB, POT_COMPLEXCOULOMB, POT_ELIPTICAL,
    POT_SIMPLECORNELL, POT_FULLCORNELL, POT_HARMONIC, POT_COMPLEXHARMONIC, POT_DODECAHEDRON, POT_FROMFILE,
    POT_FROMSCRIPT, POT_POSCHLTELLER = 100
};

struct GenParams {
    double dn, mass, sig;
    double alphas_2pit;  // alphas(2*pi*t), t = 1
    double mu_t;         // mu(t), t = 1
};

inline bool potential_kind_supported(int kind) {
    return (kind >= POT_NONE && kind <= POT_DODECAHEDRON) || kind == POT_POSCHLTELLER;
}

// potential.rs:374-391
inline double host_alphas(double mu) {
    const double nf = 2.0;
    const double b0 = 11. - 2. * nf / 3.;
    const double b1 = 51. - 19. * nf / 3.;
    const double b2 = 2857. - 5033. * nf / 9. + 325. * nf * nf / 27.;
    const double r = 2.3;
    const double l = 2. * std::log(mu / r);
    const double ll = std::log(l);
    return 4. * M_PI * (1. - 2. * b1 * ll / (b0 * b0 * l) +
                        4. * b1 * b1 * ((ll - 0.5) * (ll - 0.5) + b2 * b0 / (8. * b1 * b1) - 5.0 / 4.0) /
                            (b0 * b0 * b0 * b0 * l * l)) / (b0 * l);
}

// potential.rs:394-398
inline double host_mu(double t) {
    const double nf = 2.0, tc = 0.2;
    return 1.4 * std::sqrt((1. + nf / 6.) * 4. * M_PI * host_alphas(2. * M_PI * t)) * t * tc;
}

inline GenParams make_gen_params(double dn, double mass, double sig) {
    GenParams gp;
    gp.dn = dn; gp.mass = mass; gp.sig = sig;
    gp.alphas_2pit = host_alphas(2. * M_PI * 1.0);
    gp.mu_t = host_mu(1.0);
    return gp;
}

__device__ inline double dev_r2(long long ix, long long iy, long long iz, const Geom& g) {
    const double dx = (double)ix - ((double)g.gnx + 1.) / 2.;
    const double dy = (double)iy - ((double)g.gny + 1.) / 2.;
    const double dz = (double)iz - ((double)g.gnz + 1.) / 2.;
    return dx * dx + dy * dy + dz * dz;
}

__device__ inline double dev_linspace(double dn, long long n, long long i) {
    // numpy.linspace(-extent, extent, n)[i] with extent = (dn*n - dn)/2   (gen_potential.py:47-54)
    const double extent = (dn * (double)n - dn) / 2.;
    if (n == 1) return -extent;
    const double step = (extent - (-extent)) / (double)(n - 1);
    return i == n - 1 ? extent : (double)i * step + (-extent);
}

__device__ inline double dev_potential(int kind, long long ix, long long iy, long long iz, const Geom& g,
                                       const GenParams& gp) {
    const double nx = (double)g.gnx, ny = (double)g.gny, nz = (double)g.gnz, dn = gp.dn, mass = gp.mass;
    const long long ux = g.gnx, uy = g.gny, uz = g.gnz;
    switch (kind) {
        case POT_CUBE:
            return ((ix > ux / 4 && ix <= 3 * ux / 4) && (iy > uy / 4 && iy <= 3 * uy / 4) &&
                    (iz > uz / 4 && iz <= 3 * uz / 4)) ? -10.0 : 0.0;
        case POT_QUADWELL:
            return ((ix > ux / 4 && ix <= 3 * ux / 4) && (iy > uy / 4 && iy <= 3 * uy / 4) &&
                    (iz > 3 * uz / 8 && iz <= 5 * uz / 8)) ? -10.0 : 0.0;
        case POT_PERIODIC: {
            const double sx = sin(2. * M_PI * ((double)ix - 1.) / (nx - 1.));
            const double sy = sin(2. * M_PI * ((double)iy - 1.) / (ny - 1.));
            const double sz = sin(2. * M_PI * ((double)iz - 1.) / (nz - 1.));
            double t = sx * sx;
            t *= sy * sy;
            t *= sz * sz;
            return -t + 1.;
        }
        case POT_COULOMB:
        case POT_COMPLEXCOULOMB: {
            const double r = dn * sqrt(dev_r2(ix, iy, iz, g));
            return r < dn ? -1. / dn : -1. / r;
        }
        case POT_ELIPTICAL: {
            const double dx = (double)ix - (nx + 1.) / 2.;
            const double dy = (double)iy - (ny + 1.) / 2.;
            const double dz = ((double)iz - (nz + 1.) / 2.) * 2.;
            const double r = dn * sqrt(dx * dx + dy * dy + dz * dz);
            return r < dn ? 0.0 : -1. / r + 1. / dn;
        }
        case POT_SIMPLECORNELL: {
            const double r = dn * sqrt(dev_r2(ix, iy, iz, g));
            if (r < dn) return 4. * mass;
            return (-0.5 * (4. / 3.)) / r + gp.sig * r + 4. * mass;
        }
        case POT_FULLCORNELL: {
            const double xi = 0.0;
            const double dz = (double)iz - (nz + 1.) / 2.;
            const double r = dn * sqrt(dev_r2(ix, iy, iz, g));
            const double md = gp.mu_t * (1. + (0.07 * pow(xi, 0.2)) * (1. - dn * dn * dz * dz / (r * r))) * pow(1. + xi, -0.29);
            if (r < dn) return 4. * mass;
            return (-gp.alphas_2pit * (4. / 3.)) * exp(-md * r) / r + gp.sig * (1. - exp(-md * r)) / md -
                   (0.8 * gp.sig) / (4. * mass * mass * r) + 4. * mass;
        }
        case POT_HARMONIC:
        case POT_COMPLEXHARMONIC: {
            const double r = dn * sqrt(dev_r2(ix, iy, iz, g));
            return r * r / 2.;
        }
        case POT_DODECAHEDRON: {
            const double x = ((double)ix - (nx + 1.) / 2.) / ((nx - 1.) / 2.);
            const double y = ((double)iy - (ny + 1.) / 2.) / ((ny - 1.) / 2.);
            const double z = ((double)iz - (nz + 1.) / 2.) / ((nz - 1.) / 2.);
            const double c0 = 12.70820393249937, c1 = 11.210068307552588, c2 = 14.674169922690343;
            const double c3 = 5.605034153776295, c4 = 3.23606797749979, c5 = 1.2360679774997896;
            const double c6 = 4.23606797749979, c7 = 5.23606797749979, c8 = 18.1382715378281;
            const double c9 = 3.464101615137755, c10 = 9.06913576891405, c11 = 15.70820393249937;
            const double c12 = 9.70820393249937, c13 = 5.605034153776294, c14 = 6.47213595499958;
            const double c15 = 25.41640786499874, c16 = 1.7320508075688772, c17 = 8.47213595499958;
            const bool in = c0 + c1 * x >= c2 * z && c1 * x <= c0 + c2 * z &&
                            c3 * (c4 * x - c5 * z) <= 6. * (c6 + c7 * y) && c8 * x + c9 * z <= c0 &&
                            c10 * x + c11 * y <= c0 + c9 * z && c12 * y <= c0 + c13 * x + c2 * z &&
                            c0 + c13 * x + c12 * y + c2 * z >= 0. && c11 * y + c9 * z <= c0 + c10 * x &&
                            c3 * (-c14 * x - c5 * z) <= c15 && c9 * z <= c10 * x + 3. * (c6 + c7 * y) &&
                            c16 * (c4 * x + c17 * z) <= 3. * (c6 + c4 * y) && c13 * x + c12 * y + c2 * z <= c0;
            return in ? -100. : 0.0;
        }
        case POT_POSCHLTELLER: {
            // work index = padded index - e
            const double lam = 6., coeff = -(lam * (lam + 1.)) / 2.;
            const double cx = 1. / cosh(dev_linspace(dn, ux, ix - g.e));
            const double cy = 1. / cosh(dev_linspace(dn, uy, iy - g.e));
            const double cz = 1. / cosh(dev_linspace(dn, uz, iz - g.e));
            return coeff * (cx * cx) + coeff * (cy * cy) + coeff * (cz * cz);
        }
        default: return 0.0;
    }
}

// one CTA per (plane,row); V is written at work sites only (ring rows/pads stay 0 and are never read)
__global__ void __launch_bounds__(128) gen_potential_kernel(double* __restrict__ v, Geom g, int kind, GenParams gp) {
    const long long rows = (long long)(g.L + 2 * g.gx) * g.ny;
    for (long long r = blockIdx.x; r < rows; r += gridDim.x) {
        const int i = (int)(r / g.ny) - g.gx, j = (int)(r % g.ny);
        const long long gi = g.x0 + i;
        if (gi < 0 || gi >= g.gnx) continue;
        double* row = v + g.off(i, j, 0);
        for (int k = threadIdx.x; k < g.nz; k += blockDim.x)
            row[k] = dev_potential(kind, gi + g.e, (long long)j + g.e, (long long)k + g.e, g, gp);
    }
}

// config.rs:586-595 at padded indices; the ring (config.rs:597-622) is simply never written.
__global__ void __launch_bounds__(128) gen_ic_kernel(double* __restrict__ w, Geom g, int kind, GenParams gp) {
    const long long rows = (long long)(g.L + 2 * g.gx) * g.ny;
    const double px = (double)(g.gnx + 2 * g.e), py = (double)(g.gny + 2 * g.e), pz = (double)(g.gnz + 2 * g.e);
    for (long long r = blockIdx.x; r < rows; r += gridDim.x) {
        const int i = (int)(r / g.ny) - g.gx, j = (int)(r % g.ny);
        const long long gi = g.x0 + i;
        double* row = w + g.off(i, j, 0);
        const bool inside = gi >= 0 && gi < g.gnx;
        for (int k = threadIdx.x; k < g.nz; k += blockDim.x) {
            double val = 0.0;
            if (inside) {
                const long long ix = gi + g.e, iy = j + g.e, iz = k + g.e;
                if (kind == 3) {
                    val = 0.1;  // config.rs:593
                } else if (kind == 4) {
                    // config.rs:680: ((((i % 2) * j) % 2) * k) % 2 in f64 == 1 iff i, j, k are all odd
                    val = ((ix & 1) && (iy & 1) && (iz & 1)) ? 1.0 : 0.0;
                } else {
                    // config.rs:650-669
                    const double dx = (double)ix - px / 2., dy = (double)iy - py / 2., dz = (double)iz - pz / 2.;
                    const double rr = gp.dn * sqrt(dx * dx + dy * dy + dz * dz);
                    const double costheta = gp.dn * dz / rr;
                    const double cosphi = gp.dn * dx / rr;
                    const double mr2 = exp(-gp.mass * rr / 2.);
                    val = exp(-gp.mass * rr) + (2. - gp.mass * rr) * mr2 + gp.mass * rr * mr2 * costheta +
                          gp.mass * rr * mr2 * sqrt(1. - costheta * costheta) * cosphi;
                }
            }
            row[k] = val;
        }
    }
}


// Deterministic excited-state start.  The reference starts state n > 0 from a clone of state n-1 (grid.rs:95) and
// relies on the ~1e-16 rounding residue that survives the first normalise + Gram-Schmidt to seed the new state
// (SURVEY F7); when the sums happen to round exactly (they do on this implementation) the residue is exactly zero
// and the next step divides 0 by 0.  seed = q * f(u,v,w) with a fixed polynomial without any symmetry,
// u,v,w in [-1,1] across the lattice; plain IEEE +,-,*,/ in a fixed order, so a host restatement is bit-identical.
__device__ __host__ inline double seed_poly(long long gi, long long gj, long long gk, long long nx, long long ny, long long nz) {
    const double u = (2. * (double)gi - ((double)nx - 1.)) / (double)nx;
    const double v = (2. * (double)gj - ((double)ny - 1.)) / (double)ny;
    const double w = (2. * (double)gk - ((double)nz - 1.)) / (double)nz;
    double f = 1. + u;
    f = f + 0.5 * v;
    f = f + 0.25 * w;
    f = f + 0.7 * (u * v);
    f = f + 0.4 * (v * w);
    f = f + 0.3 * (u * w);
    f = f + 0.2 * (u * u);
    f = f - 0.1 * (v * v);
    return f;
}

__global__ void __launch_bounds__(128) seed_from_state_kernel(double* __restrict__ w, const double* __restrict__ q, Geom g) {
    const long long rows = (long long)(g.L + 2 * g.gx) * g.ny;
    for (long long r = blockIdx.x; r < rows; r += gridDim.x) {
        const int i = (int)(r / g.ny) - g.gx, j = (int)(r % g.ny);
        const long long gi = g.x0 + i;
        const long long o = g.off(i, j, 0);
        const bool inside = gi >= 0 && gi < g.gnx;
        for (int k = threadIdx.x; k < g.nz; k += blockDim.x)
            w[o + k] = inside ? q[o + k] * seed_poly(gi, j, k, g.gnx, g.gny, g.gnz) : 0.0;
    }
}

// ---- init_symmetry (config.rs:186-197 SymmetryConstraint, applied at config.rs:625 and grid.rs:137-139) ----------------
// Mirror of the work area about its centre along y (AboutY / AntisymAboutY) or z (AboutZ / AntisymAboutZ): with n the
// work size of that axis, psi[.., n-1-t] := s * psi[.., t] for t < n/2 (s = +1 / -1); for odd n and s = -1 the middle
// index becomes +0.  A copy and a sign flip, so the result is exact and applying it twice equals applying it once.
// Sources (t < n/2) and destinations (t >= n - n/2) never overlap, so the update in place is race-free.  Runs over every
// plane of the slab inside the global lattice, ghost planes included: a ghost plane gets the bits its owner computes.
enum SymKind { SYM_NONE = 0, SYM_ABOUT_Z, SYM_ANTI_Z, SYM_ABOUT_Y, SYM_ANTI_Y };

// one CTA per row; the reflected pair (t, t+1) -> (n-2-t, n-1-t) is 16-byte aligned for even nz (rows start 128-byte
// aligned), so even rows move as double2 and odd ones element by element
__global__ void __launch_bounds__(128) symmetrise_z_kernel(double* __restrict__ w, Geom g, double s) {
    const long long rows = (long long)(g.L + 2 * g.gx) * g.ny;
    const int n = g.nz, half = n / 2;
    for (long long r = blockIdx.x; r < rows; r += gridDim.x) {
        const int i = (int)(r / g.ny) - g.gx, j = (int)(r % g.ny);
        const long long gi = g.x0 + i;
        if (gi < 0 || gi >= g.gnx) continue;  // outside the lattice: zeros, and nothing maps onto them
        double* row = w + g.off(i, j, 0);
        if ((n & 1) == 0) {
            double2* row2 = reinterpret_cast<double2*>(row);
            const int pairs = half / 2;  // whole pairs below the centre
            for (int p = threadIdx.x; p < pairs; p += blockDim.x) {
                const double2 a = row2[p];
                row2[n / 2 - 1 - p] = make_double2(s * a.y, s * a.x);
            }
            if ((half & 1) && threadIdx.x == 0) row[half] = s * row[half - 1];  // the pair straddling the centre
        } else {
            for (int t = threadIdx.x; t < half; t += blockDim.x) row[n - 1 - t] = s * row[t];
            if (s < 0. && threadIdx.x == 0) row[half] = 0.0;
        }
    }
}

// one CTA per (plane, destination row): whole-row copies, double2 over the 128-byte aligned rows
__global__ void __launch_bounds__(128) symmetrise_y_kernel(double* __restrict__ w, Geom g, double s) {
    const int half = g.ny / 2, nrows = g.ny - half;  // destination rows ny-1-t for t < half, plus the middle one if odd
    const long long rows = (long long)(g.L + 2 * g.gx) * nrows;
    const int nz2 = g.nz / 2;
    for (long long r = blockIdx.x; r < rows; r += gridDim.x) {
        const int i = (int)(r / nrows) - g.gx, t = (int)(r % nrows);
        const long long gi = g.x0 + i;
        if (gi < 0 || gi >= g.gnx) continue;
        double* dst = w + g.off(i, g.ny - 1 - t, 0);
        if (t < half) {
            const double2* src2 = reinterpret_cast<const double2*>(w + g.off(i, t, 0));
            double2* dst2 = reinterpret_cast<double2*>(dst);
            for (int k = threadIdx.x; k < nz2; k += blockDim.x) {
                const double2 a = src2[k];
                dst2[k] = make_double2(s * a.x, s * a.y);
            }
            if ((g.nz & 1) && threadIdx.x == 0) dst[g.nz - 1] = s * w[g.off(i, t, g.nz - 1)];  // never the pad column
        } else if (s < 0.) {  // middle row of an odd ny
            for (int k = threadIdx.x; k < g.nz; k += blockDim.x) dst[k] = 0.0;
        }
    }
}

// ---- Gaussian initial condition (config.rs:636-642) as a counter-based field ------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11; the Random123 constants), key = seed, counter = global work site index
// s = (gi*gny + j)*gnz + k.  Box-Muller on the first two 53-bit uniforms: u1 in (0, 1], u2 in [0, 1);
// value = sig * (sqrt(-2 log u1) * cos(2 pi u2)).  The value of a site depends on (seed, s) only: not on the slab, the
// rank count or the launch shape, so ghost planes agree with their owners by construction.
struct Philox4 { uint32_t v[4]; };

__device__ __host__ inline Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                 uint32_t k1) {
    for (int r = 0; r < 10; ++r) {
        if (r) { k0 += 0x9E3779B9u; k1 += 0xBB67AE85u; }
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        c0 = n0; c1 = (uint32_t)p1; c2 = n2; c3 = (uint32_t)p0;
    }
    return Philox4{{c0, c1, c2, c3}};
}

__device__ inline double gaussian_site(unsigned long long s, unsigned long long seed, double sig) {
    const Philox4 r = philox4x32_10((uint32_t)s, (uint32_t)(s >> 32), 0u, 0u, (uint32_t)seed, (uint32_t)(seed >> 32));
    const double two_m53 = 1.1102230246251565e-16;  // 2^-53
    const double u1 = ((double)(r.v[0] >> 5) * 67108864.0 + (double)(r.v[1] >> 6) + 1.0) * two_m53;
    const double u2 = ((double)(r.v[2] >> 5) * 67108864.0 + (double)(r.v[3] >> 6)) * two_m53;
    return sig * (sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2));
}

// every work site of every slab plane inside the global lattice (ghost planes included), 0 elsewhere, like gen_ic_kernel
__global__ void __launch_bounds__(128) gen_gaussian_kernel(double* __restrict__ w, Geom g, double sig,
                                                           unsigned long long seed) {
    const long long rows = (long long)(g.L + 2 * g.gx) * g.ny;
    for (long long r = blockIdx.x; r < rows; r += gridDim.x) {
        const int i = (int)(r / g.ny) - g.gx, j = (int)(r % g.ny);
        const long long gi = g.x0 + i;
        double* row = w + g.off(i, j, 0);
        const bool inside = gi >= 0 && gi < g.gnx;
        const unsigned long long s0 = ((unsigned long long)gi * g.gny + j) * g.gnz;
        for (int k = threadIdx.x; k < g.nz; k += blockDim.x) row[k] = inside ? gaussian_site(s0 + k, seed, sig) : 0.0;
    }
}

}  // namespace wafer
