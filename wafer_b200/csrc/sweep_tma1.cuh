// sweep_tma1.cuh — TMA-pipelined ONE-step sweep for the 3/5/7-point stencils (sm_100a).
//
// Reference semantics: one iteration of the `evolve` loop body, src/grid.rs:567-673 (any CentralDifference), with
// the optional fused sum of psi'^2 that the excited-state path needs after every step (grid.rs:674-678).  Same
// round-to-nearest intrinsic chain and association order as kernels.cuh, so it is bit-identical to
// sweep_simple_kernel and to the CPU restatement (tests/test_gpu_parity.py::test_tma_one_step_sweep_bitwise).
//
// Why it exists: sweep_simple_kernel issues its loads right before it needs them and is latency bound (64 % of DRAM
// bandwidth, long-scoreboard stalls; profiles/r1_simple_512_sweep_full.txt).  Here one elected thread keeps an
// (E+3)-stage ring of psi planes (2.5-D streaming along x, halo E in y, HE = E rounded up to even in z) and V planes
// in flight through TMA (cp.async.bulk.tensor.3d + mbarrier), zero-filled outside the lattice = the Dirichlet ring.
// The (2E+1)-deep x queue of every site lives in registers and rotates by renaming (the plane loop is unrolled
// 2E+1 times); y/z neighbours come from the shared-memory stage of the centre plane.  CTA = 32 x TZ output sites
// (TZ = 60, 60, 56), 16 warps, every thread owns a 2x2 site micro-tile per plane.  Opt-in for round 1
// (WAFER_FLAG_TMA_ONE_STEP): it was written after the round's GPU budget for tuning had been spent.
#pragma once
#include <utility>

#include "kernels.cuh"
#include "sweep_tb.cuh"

namespace wafer {
namespace t1 {

using tb::DivConst;

template <int E>
struct Cfg {
    static constexpr int N = 2 * E + 1;         // x queue depth
    static constexpr int HE = (E + 1) & ~1;     // z halo columns per side, even so that column pairs stay aligned
    static constexpr int BW = 64;               // box width
    static constexpr int TZ = BW - 2 * HE;      // output columns per tile
    static constexpr int NWARP = 16;
    static constexpr int TY = 2 * NWARP;        // output rows per tile
    static constexpr int R0 = TY + 2 * E;       // psi box rows
    static constexpr int NST = E + 3;           // ring: planes c .. c+E in use, two more in flight
    static constexpr int THREADS = NWARP * 32;
    static constexpr uint32_t STAGE_BYTES = (R0 * BW + TY * BW) * sizeof(double);
};

template <int E>
struct __align__(128) Stage {
    double psi[Cfg<E>::R0 * Cfg<E>::BW];
    double v[Cfg<E>::TY * Cfg<E>::BW];
};
template <int E>
struct Smem {
    Stage<E> st[Cfg<E>::NST];
    unsigned long long full[Cfg<E>::NST];  // TMA landed
    unsigned long long done[4];            // every thread finished iteration t (ring of 4)
};

// queue slot of plane (newest - j) when the newest plane sits in slot PHASE
template <int E>
__host__ __device__ constexpr int qslot(int phase, int j) {
    return (phase - j + 2 * Cfg<E>::N) % Cfg<E>::N;
}

struct Lane1 {
    int cb;            // element offset of the lane's column pair in row 2*warp of a 64-wide region
    bool st0, st1;     // store column 0 / column 1 of the pair (inside the tile's output columns and the lattice)
    double yy2[2], zz2[2];  // (j - cy)^2 of the two rows, (k - cz)^2 of the two columns (potential.rs:366-371), check modes
};
struct Tile1 {
    bool yin[2];       // slot row inside the lattice
    int xa, xz;        // output planes [xa, xz)
};

// MODE of the kernel:
//   0..5         sweep with NRED = MODE running sums: 1 = sum psi'^2 (grid.rs:675-678), 1 + k = additionally the overlaps
//                sum q_i psi' with k <= MAX_FUSED_LOWERS stored states (grid.rs:482-487), read once at the output sites
//   MODE_OBS+p   compute_observables (grid.rs:303-445) of the INPUT field, nothing stored: four sums
//                [0] ((v w) w) - ((w S)/den), [1] w w, [2] (w w) potsub, [3] (w w) r2;  p = 0 none, 1 scalar, 2 array,
//                p = 3: sum [0] only
//   MODE_CHK+p   sweep that also leaves the three point-wise sums of the check that follows it, taken on psi':
//                [0] w w, [1] (w w) potsub, [2] (w w) r2  (north-star: "block reductions fused into the final sweep
//                before each check"; the energy needs neighbours of psi' and stays a pass of its own)
constexpr int MAX_FUSED_LOWERS = 4;
constexpr int MODE_OBS = 8, MODE_CHK = 16;
template <int MODE>
struct Mode {
    static constexpr bool obs = MODE >= MODE_OBS && MODE < MODE_CHK;
    static constexpr bool chk = MODE >= MODE_CHK;
    static constexpr int potsub = obs ? MODE - MODE_OBS : (chk ? MODE - MODE_CHK : 0);
    static constexpr bool eonly = obs && potsub == 3;  // MODE_OBS + 3: the energy sum alone (the rest came from a MODE_CHK sweep)
    static constexpr int nred = eonly ? 1 : (obs ? 4 : (chk ? 3 : MODE));
    static constexpr int nacc = nred > 0 ? nred : 1;
};
struct Extra {
    const double* q[MAX_FUSED_LOWERS];  // stored states for the fused overlaps
    const double* potsub_arr;           // pot_sub array in the slab layout (potential.rs:135-144), or NULL
    double potsub;                      // pot_sub scalar (potential.rs:148-152)
    int nb_total, bid_off;              // partial-sum row length / this launch's first column when several launches share a row
    int hf;                             // sweep modes: the "V" tensor map describes h = (dt*v)/2 (wafer_b200.cu::ensure_hfield)
};

// cold path of the energy integrand: plain IEEE division (grid.rs:325-332)
__device__ __noinline__ double energy_safe(double v, double w, double s, double den) {
    return D_SUB(D_MUL(D_MUL(v, w), w), D_DIV(D_MUL(w, s), den));
}

template <int E, int MODE, int PHASE>
__device__ __forceinline__ void iteration(Smem<E>& sm, double2 (&q)[2][Cfg<E>::N], int t, int T, const Lane1& ln,
                                          const Tile1& tl, int row_pitch, double*& orow, long long plane_elems, double dt,
                                          const DivConst& dc, double (&acc)[Mode<MODE>::nacc], const Extra& ex,
                                          const double* out_base, double xc0) {
    using C = Cfg<E>;
    using M = Mode<MODE>;
    constexpr int BW = C::BW;
    const int s_new = t % C::NST;
    // the stored states at this iteration's output sites: issued before the wait on the TMA stage and the stencil
    // arithmetic, consumed after them (loading them at the point of use left the whole DRAM latency exposed: the k = 1
    // sweep took 1.0 ms against 0.6 ms for the plain one at 512^3, ncu r2n)
    constexpr int NQ = (M::nred > 1 && !M::obs && !M::chk) ? M::nred - 1 : 0;
    // NPRE of the NQ states are fetched early; more than that spills at the 128-register cap (ptxas -v).  With 3 or 4
    // states, one early, measured at 512^3, k = 3 / 4: 65.1 / 58.1 GLUPS, against 64.7 / 57.8 for none and 62.7 / 55.2 for two
    constexpr int NPRE = E != 1 ? 0 : (NQ <= 2 ? NQ : 1);
    double2 ql[2][NQ > 0 ? NQ : 1];
    if (NPRE > 0 && t >= 2 * E) {
#pragma unroll
        for (int s = 0; s < 2; ++s)
            if (tl.yin[s] && ln.st0) {
#pragma unroll
                for (int i = 0; i < NPRE; ++i)
                    ql[s][i] = __ldg(reinterpret_cast<const double2*>(ex.q[i] + ((orow - out_base) + s * row_pitch)));
            }
    }
    tb::mbar_wait(&sm.full[s_new], (t / C::NST) & 1);
    const double* psn = sm.st[s_new].psi + ln.cb;
#pragma unroll
    for (int s = 0; s < 2; ++s) q[s][PHASE] = *reinterpret_cast<const double2*>(psn + (s + E) * BW);
    if (t >= 2 * E) {
        // ---- output plane c = newest - E; its y/z neighbours sit in the stage loaded E iterations ago
        const int s_ctr = (t - E) % C::NST;
        const double* psc = sm.st[s_ctr].psi + ln.cb;
        const double* vs = sm.st[s_new].v + ln.cb;  // V plane c rides with psi plane c+E
        constexpr int IC = qslot<E>(PHASE, E);
        const bool nofast = !dc.fast;
        double xx2 = 0.0;
        if (M::obs || M::chk) {  // (global x of the output plane - centre)^2; the plane is xa - 2E + t
            const double dx = D_ADD(xc0, (double)t);
            xx2 = D_MUL(dx, dx);
        }
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            const double* row = psc + (s + E) * BW;
            const double2 w = q[s][IC];
            double xp0[E], xm0[E], xp1[E], xm1[E], yp0[E], ym0[E], yp1[E], ym1[E], zp0[E], zm0[E], zp1[E], zm1[E];
            double zl[E], zr[E];
#pragma unroll
            for (int m = 1; m <= E; ++m) {
                const double2 a = q[s][qslot<E>(PHASE, E - m)], b = q[s][qslot<E>(PHASE, E + m)];
                xp0[m - 1] = a.x; xp1[m - 1] = a.y;
                xm0[m - 1] = b.x; xm1[m - 1] = b.y;
                // 2x2 micro-tile: the inner y neighbour at distance 1 is the other slot's centre (a register)
                const double2 up = (m == 1 && s == 0) ? q[1][IC] : *reinterpret_cast<const double2*>(row + m * BW);
                const double2 dn = (m == 1 && s == 1) ? q[0][IC] : *reinterpret_cast<const double2*>(row - m * BW);
                yp0[m - 1] = up.x; yp1[m - 1] = up.y;
                ym0[m - 1] = dn.x; ym1[m - 1] = dn.y;
                zl[m - 1] = row[-m];      // column 2l - m
                zr[m - 1] = row[1 + m];   // column 2l + 1 + m
            }
            zp0[0] = w.y; zm1[0] = w.x;
#pragma unroll
            for (int m = 1; m <= E; ++m) {
                zm0[m - 1] = zl[m - 1];
                zp1[m - 1] = zr[m - 1];
                if (m >= 2) { zp0[m - 1] = zr[m - 2]; zm1[m - 1] = zl[m - 2]; }
            }
            const double s0 = Lap<E>::sum(xp0, xm0, yp0, ym0, zp0, zm0, w.x);
            const double s1 = Lap<E>::sum(xp1, xm1, yp1, ym1, zp1, zm1, w.y);
            const double2 vv = *reinterpret_cast<const double2*>(vs + s * BW);
            const bool row_ok = tl.yin[s];
            const bool w0 = row_ok && ln.st0, w1 = row_ok && ln.st1;
            unsigned b0 = 0u, b1 = 0u;
            if (M::obs) {
                // grid.rs:325-332: ((v w) w) - ((w S)/den); the pad column of an odd nz holds psi = 0 and adds exact zeros
                double e0 = D_SUB(D_MUL(D_MUL(vv.x, w.x), w.x), tb::div_fast(D_MUL(w.x, s0), dc, b0));
                double e1 = D_SUB(D_MUL(D_MUL(vv.y, w.y), w.y), tb::div_fast(D_MUL(w.y, s1), dc, b1));
                if (w0) {
                    if (b0 || b1 || nofast) {
                        e0 = energy_safe(vv.x, w.x, s0, dc.den);
                        e1 = energy_safe(vv.y, w.y, s1, dc.den);
                    }
                    acc[0] = D_ADD(acc[0], D_ADD(e0, e1));
                }
                if (w0 && !M::eonly) {
                    const double ww0 = D_MUL(w.x, w.x), ww1 = D_MUL(w.y, w.y);
                    acc[1] = D_ADD(acc[1], D_ADD(ww0, ww1));
                    if (M::potsub == 1) acc[2] = D_ADD(acc[2], D_ADD(D_MUL(ww0, ex.potsub), D_MUL(ww1, ex.potsub)));
                    if (M::potsub == 2) {
                        const double2 ps = __ldg(reinterpret_cast<const double2*>(ex.potsub_arr + ((orow - out_base) + s * row_pitch)));
                        acc[2] = D_ADD(acc[2], D_ADD(D_MUL(ww0, ps.x), D_MUL(ww1, ps.y)));
                    }
                    const double r20 = D_ADD(D_ADD(xx2, ln.yy2[s]), ln.zz2[0]), r21 = D_ADD(D_ADD(xx2, ln.yy2[s]), ln.zz2[1]);
                    acc[3] = D_ADD(acc[3], D_ADD(D_MUL(ww0, r20), D_MUL(ww1, r21)));
                }
            } else {
                double a0, bd0, a1, bd1;
                if (ex.hf) {  // (CTA-uniform) two DMULs less per site
                    tb::ab_fast_h(vv.x, dt, a0, bd0, b0);
                    tb::ab_fast_h(vv.y, dt, a1, bd1, b1);
                } else {
                    tb::ab_fast(vv.x, dt, a0, bd0, b0);
                    tb::ab_fast(vv.y, dt, a1, bd1, b1);
                }
                double2 r;
                r.x = tb::update_fast(w.x, a0, bd0, s0, dc, b0);
                r.y = tb::update_fast(w.y, a1, bd1, s1, dc, b1);
                if ((w0 && (b0 || nofast)) || (w1 && (b1 || nofast))) {  // cold: an operand left the fast-division window
                    r.x = ex.hf ? tb::site_safe_h(w.x, vv.x, s0, dt, dc.den).u : tb::site_safe(w.x, vv.x, s0, dt, dc.den).u;
                    r.y = ex.hf ? tb::site_safe_h(w.y, vv.y, s1, dt, dc.den).u : tb::site_safe(w.y, vv.y, s1, dt, dc.den).u;
                }
                if (w0) {
                    if (!w1) r.y = 0.0;  // odd nz: the pad column keeps its zero
                    *reinterpret_cast<double2*>(orow + s * row_pitch) = r;
                    if (M::chk) {
                        const double ww0 = D_MUL(r.x, r.x), ww1 = D_MUL(r.y, r.y);
                        acc[0] = D_ADD(acc[0], D_ADD(ww0, ww1));
                        if (M::potsub == 1) acc[1] = D_ADD(acc[1], D_ADD(D_MUL(ww0, ex.potsub), D_MUL(ww1, ex.potsub)));
                        if (M::potsub == 2) {
                            const double2 ps = __ldg(reinterpret_cast<const double2*>(ex.potsub_arr + ((orow - out_base) + s * row_pitch)));
                            acc[1] = D_ADD(acc[1], D_ADD(D_MUL(ww0, ps.x), D_MUL(ww1, ps.y)));
                        }
                        const double r20 = D_ADD(D_ADD(xx2, ln.yy2[s]), ln.zz2[0]), r21 = D_ADD(D_ADD(xx2, ln.yy2[s]), ln.zz2[1]);
                        acc[2] = D_ADD(acc[2], D_ADD(D_MUL(ww0, r20), D_MUL(ww1, r21)));
                    } else {
                        if (M::nred >= 1) acc[0] = D_ADD(acc[0], D_ADD(D_MUL(r.x, r.x), D_MUL(r.y, r.y)));
#pragma unroll
                        for (int i = 1; i < M::nred; ++i) {  // the stored states share psi's layout: same element offset
                            if (i - 1 >= NPRE) ql[s][i - 1] = __ldg(reinterpret_cast<const double2*>(ex.q[i - 1] + ((orow - out_base) + s * row_pitch)));
                            acc[i] = D_ADD(acc[i], D_ADD(D_MUL(ql[s][i - 1].x, r.x), D_MUL(ql[s][i - 1].y, r.y)));
                        }
                    }
                }
            }
        }
    }
    tb::mbar_arrive(&sm.done[t & 3]);
    orow += plane_elems;
    (void)T;
}

template <int E, int MODE, int... PH>
__device__ __forceinline__ void run_phases(std::integer_sequence<int, PH...>, Smem<E>& sm, double2 (&q)[2][Cfg<E>::N], int t0,
                                           int T, const Lane1& ln, const Tile1& tl, int row_pitch, double*& orow,
                                           long long plane_elems, double dt, const DivConst& dc,
                                           double (&acc)[Mode<MODE>::nacc], const Extra& ex, const double* out_base, double xc0,
                                           const CUtensorMap* tm_psi, const CUtensorMap* tm_v, int z0, int y0, int gx) {
    using C = Cfg<E>;
    // after iteration t-1 has been finished by every thread, the stage of its centre plane is free: refill it
    auto refill = [&](int t) {
        if (threadIdx.x == 0 && t >= 1) {
            tb::mbar_wait(&sm.done[(t - 1) & 3], ((t - 1) >> 2) & 1);
            const int j = t - 1 - E;  // plane-iteration whose stage is free now
            if (j >= 0 && j + C::NST < T) {
                const int tn = j + C::NST, sn = tn % C::NST, p = tl.xa - E + tn;
                tb::mbar_expect_tx(&sm.full[sn], C::STAGE_BYTES);
                tb::tma_load_3d(sm.st[sn].psi, tm_psi, z0 - C::HE, y0 - E, p + gx, &sm.full[sn]);
                tb::tma_load_3d(sm.st[sn].v, tm_v, z0 - C::HE, y0, p - E + gx, &sm.full[sn]);
            }
        }
    };
    ((t0 + PH < T ? (iteration<E, MODE, PH>(sm, q, t0 + PH, T, ln, tl, row_pitch, orow, plane_elems, dt, dc, acc, ex, out_base, xc0), refill(t0 + PH))
                  : void()),
     ...);
}

// `out`: the output field; in the observables modes the INPUT field itself (only its address arithmetic is used)
template <int E, int MODE>
__global__ void __launch_bounds__(Cfg<E>::THREADS, 1)
    sweep_tma1_kernel(const __grid_constant__ CUtensorMap tm_psi, const __grid_constant__ CUtensorMap tm_v,
                      double* __restrict__ out, Geom g, int xb, int xe, int xchunk, double dt, double den, int den_ok,
                      double* __restrict__ partials, Extra ex) {
    using M = Mode<MODE>;
    using C = Cfg<E>;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    Smem<E>& sm = *reinterpret_cast<Smem<E>*>(smem_raw);
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
    const int lane = threadIdx.x & 31;
    const int z0 = blockIdx.x * C::TZ, y0 = blockIdx.y * C::TY;
    Tile1 tl;
    tl.xa = xb + blockIdx.z * xchunk;
    tl.xz = min(tl.xa + xchunk, xe);
    const int T = (tl.xz - tl.xa) + 2 * E;  // psi planes xa-E .. xz-1+E

    if (threadIdx.x == 0) {
        for (int s = 0; s < C::NST; ++s) tb::mbar_init(&sm.full[s], 1);
        for (int s = 0; s < 4; ++s) tb::mbar_init(&sm.done[s], C::THREADS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        for (int t = 0; t < C::NST && t < T; ++t) {
            const int p = tl.xa - E + t;
            tb::mbar_expect_tx(&sm.full[t], C::STAGE_BYTES);
            tb::tma_load_3d(sm.st[t].psi, &tm_psi, z0 - C::HE, y0 - E, p + g.gx, &sm.full[t]);
            tb::tma_load_3d(sm.st[t].v, &tm_v, z0 - C::HE, y0, p - E + g.gx, &sm.full[t]);
        }
    }
    __syncthreads();

    DivConst dc;
    dc.den = den;
    dc.r = tb::refined_reciprocal(den);
    dc.fast = den_ok;

    Lane1 ln;
    const int gz = z0 - C::HE + 2 * lane;
    ln.cb = 2 * warp * C::BW + 2 * lane;
    const bool col = lane >= C::HE / 2 && lane < 32 - C::HE / 2;
    ln.st0 = col && gz < g.nz;
    ln.st1 = col && (gz + 1) < g.nz;
#pragma unroll
    for (int s = 0; s < 2; ++s) tl.yin[s] = (y0 + 2 * warp + s) < g.ny;
    // potential.rs:366-371 on global WORK indices: d = idx - (N + 1)/2 per axis
#pragma unroll
    for (int s = 0; s < 2; ++s) {
        const double dy = D_SUB((double)(y0 + 2 * warp + s), D_DIV(D_ADD((double)g.gny, 1.), 2.));
        const double dz = D_SUB((double)(gz + s), D_DIV(D_ADD((double)g.gnz, 1.), 2.));
        ln.yy2[s] = D_MUL(dy, dy);
        ln.zz2[s] = D_MUL(dz, dz);
    }
    // x offset of the output plane of iteration t from the centre: (x0 + xa - 2E + t) - (gnx + 1)/2 = xc0 + t, exact in
    // f64 (integers and half-integers far below 2^52)
    const double xc0 = D_SUB((double)(g.x0 + tl.xa - 2 * E), D_DIV(D_ADD((double)g.gnx, 1.), 2.));
    // running store pointer: the lane's pair in slot 0's row of the output plane of iteration t (= xa - 2E + t)
    double* orow = out + g.off(tl.xa - 2 * E, y0 + 2 * warp, 0) + gz;

    double2 q[2][C::N];
#pragma unroll
    for (int s = 0; s < 2; ++s)
#pragma unroll
        for (int j = 0; j < C::N; ++j) q[s][j] = make_double2(0., 0.);
    double acc[M::nacc];
#pragma unroll
    for (int i = 0; i < M::nacc; ++i) acc[i] = 0.0;

#pragma unroll 1
    for (int t0 = 0; t0 < T; t0 += C::N)
        run_phases<E, MODE>(std::make_integer_sequence<int, C::N>{}, sm, q, t0, T, ln, tl, g.zp, orow, g.plane, dt, dc, acc,
                            ex, out, xc0, &tm_psi, &tm_v, z0, y0, g.gx);

    if (M::nred > 0) {
        const int nb = gridDim.x * gridDim.y * gridDim.z;
        const int bid = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
        block_reduce_store<M::nacc>(acc, partials, ex.nb_total ? ex.nb_total : nb, ex.bid_off + bid);
    }
}

}  // namespace t1
}  // namespace wafer
