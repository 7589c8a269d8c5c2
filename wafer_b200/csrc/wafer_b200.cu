// wafer_b200.cu — context, stream orchestration and the C ABI of include/wafer_b200.h.
//
// One wafer_ctx = one GPU = one x-slab of the lattice.  The reference functions each entry point replaces are
// cited in the header; the driver loop `wafer_solve` restates src/grid.rs:50-246 on top of them.
#include "../../include/wafer_b200.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <new>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include <errno.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include "decode.cuh"
#include "encode.cuh"
#include "generators.cuh"
#include "kernels.cuh"
#include "nccl_dyn.h"
#include "resample.cuh"
#include "sweep_tb.cuh"
#include "sweep_tma1.cuh"

using namespace wafer;

namespace {
std::string g_create_error;

// scalar slots in ctx->scal (device doubles)
// SL_RAW: [0] = sum psi^2 of the last excited-state sweep, [1 + i] = raw overlap sum q_i psi; SL_COEF: Gram-Schmidt s_i
// SL_CHK: [sum psi^2, sum psi^2 potsub, sum psi^2 r2] left by the last sweep of a ground-state evolve (MODE_CHK)
enum { SL_OBS = 0, SL_TMP = 5, SL_CHK = 8, SL_RAW = 16, SL_COEF = 16 + 256, SL_COUNT = 16 + 512 };
constexpr int GRAM_LD = 256;  // at most 255 stored states (wavenum is a u8)

// ---- array files (wafer_write_array): encode kernels over the work sites of this rank's slab -------------------
// Sites are numbered in file order (x slowest, z fastest) from the slab's first work site; block b of the encoder
// owns sites [b ENC_BS, (b + 1) ENC_BS).  encode_len_kernel leaves the bytes of each block's certified sites in
// btot[b] and appends the sites fmt_g17 refuses to a list; the host formats those with snprintf, adds their lengths
// and scans the block totals into byte offsets; encode_emit_kernel writes every site's bytes at its offset, taking a
// refused site's text from the sorted table of host-formatted numbers.
constexpr int ENC_THREADS = 256, ENC_BS = ENC_THREADS * 16;
constexpr unsigned ENC_FLAG_CAP = 16u * ENC_BS;  // refused sites one launch collects; 16 blocks can never overflow it
struct EncFlagIn { double v; unsigned long long site; };
struct EncFlagStr { unsigned long long site; unsigned int len; char s[28]; };
// The power table lives in a device buffer uploaded once (EncTable layout), not in a __device__ array: a module-scope
// array would take a slot in front of the math library's tables and change the code of the kernels that read those.
struct EncTable {
    uint64_t hilo[2 * enc::NPOW];
    int16_t shift[enc::NPOW];
};

// the power table in shared memory: lanes of a warp index different entries
__device__ __forceinline__ enc::Pow10 enc_load_table(EncTable& s, const EncTable* __restrict__ g) {
    for (int i = threadIdx.x; i < 2 * enc::NPOW; i += blockDim.x) s.hilo[i] = g->hilo[i];
    for (int i = threadIdx.x; i < enc::NPOW; i += blockDim.x) s.shift[i] = g->shift[i];
    __syncthreads();
    return enc::Pow10{s.hilo, s.shift};
}

// slab site -> the value and its global (i, j, k)
__device__ __forceinline__ double enc_site(const double* __restrict__ f, const Geom& g, unsigned long long s,
                                           unsigned long long* gi, unsigned long long* j, unsigned long long* k) {
    const unsigned long long plane = (unsigned long long)g.ny * (unsigned long long)g.nz;
    const unsigned long long li = s / plane, r = s - li * plane;
    *j = r / (unsigned long long)g.nz;
    *k = r - *j * (unsigned long long)g.nz;
    *gi = (unsigned long long)g.x0 + li;
    return f[g.off((int)li, (int)*j, (int)*k)];
}

template <int FMT>
__global__ void __launch_bounds__(ENC_THREADS)
    encode_len_kernel(const double* __restrict__ f, Geom g, long long b0, unsigned long long nsites, const EncTable* pow10,
                      unsigned int* __restrict__ btot, EncFlagIn* __restrict__ list, unsigned long long* __restrict__ count) {
    __shared__ EncTable tab;
    __shared__ unsigned int warp_sum[ENC_THREADS / 32];
    const enc::Pow10 t = enc_load_table(tab, pow10);
    const long long b = b0 + blockIdx.x;
    const unsigned long long sb = (unsigned long long)b * ENC_BS, se = min(sb + ENC_BS, nsites);
    unsigned int tot = 0;
    for (unsigned long long s = sb + threadIdx.x; s < se; s += ENC_THREADS) {
        unsigned long long gi, j, k;
        const double v = enc_site(f, g, s, &gi, &j, &k);
        char buf[enc::SITE_MAX];
        const int n = enc::encode_site(FMT, v, gi, j, k, g.x0 == 0 && s == 0, nullptr, 0, buf, t);
        if (n < 0) {
            const unsigned long long at = atomicAdd(count, 1ull);
            if (at < ENC_FLAG_CAP) list[at] = EncFlagIn{v, s};
        } else {
            tot += (unsigned int)n;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tot += __shfl_down_sync(0xffffffffu, tot, o);
    if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = tot;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int s = 0;
        for (int w = 0; w < ENC_THREADS / 32; ++w) s += warp_sum[w];
        btot[b] = s;
    }
}

template <int FMT>
__global__ void __launch_bounds__(ENC_THREADS)
    encode_emit_kernel(const double* __restrict__ f, Geom g, long long b0, unsigned long long nsites, const EncTable* pow10,
                       const unsigned long long* __restrict__ boff, unsigned long long base,
                       const EncFlagStr* __restrict__ host_txt, int n_host, unsigned char* __restrict__ out,
                       unsigned long long* __restrict__ missing) {
    __shared__ EncTable tab;
    __shared__ unsigned char stage[ENC_THREADS * enc::SITE_MAX];
    __shared__ unsigned int warp_sum[ENC_THREADS / 32];
    const enc::Pow10 t = enc_load_table(tab, pow10);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long b = b0 + blockIdx.x;
    const unsigned long long sb = (unsigned long long)b * ENC_BS, se = min(sb + ENC_BS, nsites);
    unsigned long long o = boff[b] - base;
    for (unsigned long long s0 = sb; s0 < se; s0 += ENC_THREADS) {
        const unsigned long long s = s0 + threadIdx.x;
        char buf[enc::SITE_MAX];
        int n = 0;
        if (s < se) {
            unsigned long long gi, j, k;
            const double v = enc_site(f, g, s, &gi, &j, &k);
            const bool first = g.x0 == 0 && s == 0;
            n = enc::encode_site(FMT, v, gi, j, k, first, nullptr, 0, buf, t);
            if (n < 0) {  // refused by fmt_g17: the host's text, found by binary search in the sorted table
                int lo = 0, hi = n_host;
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (host_txt[mid].site < s) lo = mid + 1;
                    else hi = mid;
                }
                if (lo < n_host && host_txt[lo].site == s) {
                    n = enc::encode_site(FMT, v, gi, j, k, first, host_txt[lo].s, (int)host_txt[lo].len, buf, t);
                } else {
                    n = 0;
                    atomicAdd(missing, 1ull);
                }
            }
        }
        // exclusive block scan of the lengths
        unsigned int incl = (unsigned int)n;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const unsigned int y = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += y;
        }
        if (lane == 31) warp_sum[warp] = incl;
        __syncthreads();
        unsigned int before = 0, total = 0;
        for (int w = 0; w < ENC_THREADS / 32; ++w) {
            if (w < warp) before += warp_sum[w];
            total += warp_sum[w];
        }
        const unsigned int at = before + incl - (unsigned int)n;
        for (int c = 0; c < n; ++c) stage[at + c] = (unsigned char)buf[c];
        __syncthreads();
        for (unsigned int c = threadIdx.x; c < total; c += ENC_THREADS) out[o + c] = stage[c];
        o += total;
        __syncthreads();
    }
}

// ---- array files read (wafer_load_array): decode kernels over one chunk of a file's records ---------------------
// A Csv / Json chunk holds whole records (the host carries a split one into the next chunk); a record starts at byte
// 0 and after every separator.  Block b owns the records that start in bytes [b DEC_SEG, (b + 1) DEC_SEG):
// dec_count_kernel counts them, dec_offsets_kernel scans the counts into global record indices, dec_text_kernel lists
// the block's record starts through a block scan, checks each record's grammar (and a Csv record's indices) and
// converts the numbers of the source planes [p0, p1) into dst.  Numbers parse_f64 cannot certify are listed (record,
// offset, length) for strtod on the host.  A Messagepack chunk holds whole 9-byte elements: dec_mpk_kernel.
constexpr int DEC_THREADS = 256, DEC_BYTES = 32, DEC_SEG = DEC_THREADS * DEC_BYTES;
constexpr unsigned DEC_FLAG_CAP = 16u * DEC_SEG;  // numbers one launch lists; 16 blocks can never overflow it
struct DecFlag { unsigned long long rec; unsigned int at, len; double v; };
struct DecDst {  // the converted source planes [p0, p1) of an array of n sites, `plane` = sy sz sites per x-plane
    double* dst;
    unsigned long long n, plane, sz, p0, p1;
};
enum { DEC_ERR = 0, DEC_NFLAG = 1, DEC_WORDS = 2 };  // state words of one chunk

__device__ __forceinline__ bool dec_is_start(const unsigned char* __restrict__ c, unsigned long long p, unsigned char sep) {
    return p == 0 || c[p - 1] == sep;
}

// record starts in this thread's DEC_BYTES bytes of block b's segment, as a bit mask
__device__ __forceinline__ unsigned int dec_starts(const unsigned char* __restrict__ c, unsigned long long len, long long b,
                                                   unsigned char sep, unsigned long long* at) {
    *at = (unsigned long long)b * DEC_SEG + (unsigned long long)threadIdx.x * DEC_BYTES;
    unsigned int m = 0;
    for (int i = 0; i < DEC_BYTES; ++i) {
        const unsigned long long p = *at + i;
        if (p < len && dec_is_start(c, p, sep)) m |= 1u << i;
    }
    return m;
}

__global__ void __launch_bounds__(DEC_THREADS)
    dec_count_kernel(const unsigned char* __restrict__ c, unsigned long long len, unsigned char sep,
                     unsigned int* __restrict__ bcount) {
    __shared__ unsigned int warp_sum[DEC_THREADS / 32];
    unsigned long long at;
    unsigned int n = __popc(dec_starts(c, len, blockIdx.x, sep, &at));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) n += __shfl_down_sync(0xffffffffu, n, o);
    if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = n;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int s = 0;
        for (int w = 0; w < DEC_THREADS / 32; ++w) s += warp_sum[w];
        bcount[blockIdx.x] = s;
    }
}

// one block: boff[b] = records before block b of this chunk, counting from *base; *base += the chunk's records
__global__ void __launch_bounds__(1024)
    dec_offsets_kernel(const unsigned int* __restrict__ bcount, int nb, unsigned long long* __restrict__ boff,
                       unsigned long long* __restrict__ base) {
    __shared__ unsigned long long part[1024];
    const int per = (nb + 1023) / 1024, b0 = threadIdx.x * per, b1 = min(nb, b0 + per);
    unsigned long long s = 0;
    for (int b = b0; b < b1; ++b) s += bcount[b];
    part[threadIdx.x] = s;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {  // inclusive scan of the thread sums
        const unsigned long long y = threadIdx.x >= d ? part[threadIdx.x - d] : 0;
        __syncthreads();
        part[threadIdx.x] += y;
        __syncthreads();
    }
    const unsigned long long first = *base;
    unsigned long long o = first + part[threadIdx.x] - s;
    for (int b = b0; b < b1; ++b) {
        boff[b] = o;
        o += bcount[b];
    }
    __syncthreads();
    if (threadIdx.x == 0) *base = first + part[1023];
}

template <int FMT>
__global__ void __launch_bounds__(DEC_THREADS)
    dec_text_kernel(const unsigned char* __restrict__ c, unsigned long long len, long long b0,
                    const unsigned long long* __restrict__ boff, const EncTable* pow10, DecDst d,
                    DecFlag* __restrict__ list, unsigned long long* __restrict__ st) {
    __shared__ EncTable tab;
    __shared__ unsigned short starts[DEC_SEG];
    __shared__ unsigned int warp_sum[DEC_THREADS / 32];
    const enc::Pow10 t = enc_load_table(tab, pow10);
    const unsigned char sep = FMT == enc::FMT_CSV ? '\n' : ',';
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long b = b0 + blockIdx.x;
    unsigned long long at;
    unsigned int m = dec_starts(c, len, b, sep, &at);
    // exclusive block scan of the start counts: this thread's starts go to starts[before ..]
    const unsigned int n = __popc(m);
    unsigned int incl = n;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned int y = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += y;
    }
    if (lane == 31) warp_sum[warp] = incl;
    __syncthreads();
    unsigned int before = incl - n, total = 0;
    for (int w = 0; w < DEC_THREADS / 32; ++w) {
        if (w < warp) before += warp_sum[w];
        total += warp_sum[w];
    }
    const unsigned long long seg = (unsigned long long)b * DEC_SEG;
    for (; m; m &= m - 1) starts[before++] = (unsigned short)(at - seg + __ffs(m) - 1);
    __syncthreads();
    bool bad = false;
    for (unsigned int r = threadIdx.x; r < total; r += DEC_THREADS) {
        const unsigned long long p = seg + starts[r], rec = boff[b] + r;
        unsigned long long e = p;
        while (e < len && c[e] != sep) ++e;
        if (rec >= d.n) {
            bad = true;
            continue;
        }
        const unsigned char* num = c + p;
        if (FMT == enc::FMT_CSV) {  // record rec carries the indices of site rec
            const unsigned long long i = rec / d.plane, jk = rec - i * d.plane, j = jk / d.sz;
            if (dec::csv_record(c + p, c + e, i, j, jk - j * d.sz, &num) != dec::TOK_OK) {
                bad = true;
                continue;
            }
        }
        double v;
        const int rc = dec::parse_f64(num, c + e, t, &v);
        if (rc == dec::TOK_BAD) {
            bad = true;
            continue;
        }
        const unsigned long long plane = rec / d.plane;
        if (plane < d.p0 || plane >= d.p1) continue;
        if (rc == dec::TOK_OK) {
            d.dst[rec - d.p0 * d.plane] = v;
        } else {
            const unsigned long long k = atomicAdd(st + DEC_NFLAG, 1ull);
            if (k < DEC_FLAG_CAP) list[k] = DecFlag{rec, (unsigned int)(num - c), (unsigned int)(c + e - num), 0.0};
        }
    }
    if (bad) atomicOr(st + DEC_ERR, 1ull);
}

// elements [e0, e0 + nel) of a Messagepack array: 0xcb and the big-endian bits, 9 bytes each
__global__ void __launch_bounds__(DEC_THREADS)
    dec_mpk_kernel(const unsigned char* __restrict__ c, unsigned long long nel, unsigned long long e0, DecDst d,
                   unsigned long long* __restrict__ st) {
    bool bad = false;
    for (unsigned long long i = (unsigned long long)blockIdx.x * DEC_THREADS + threadIdx.x; i < nel;
         i += (unsigned long long)gridDim.x * DEC_THREADS) {
        const unsigned char* q = c + 9 * i;
        if (q[0] != 0xcb) {
            bad = true;
            continue;
        }
        const unsigned long long rec = e0 + i, plane = rec / d.plane;
        if (plane < d.p0 || plane >= d.p1) continue;
        unsigned long long u = 0;
        for (int k = 1; k < 9; ++k) u = (u << 8) | q[k];
        d.dst[rec - d.p0 * d.plane] = __longlong_as_double((long long)u);
    }
    if (bad) atomicOr(st + DEC_ERR, 1ull);
}

// the numbers converted on the host
__global__ void dec_scatter_kernel(DecDst d, const DecFlag* __restrict__ list, int n) {
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x)
        d.dst[list[k].rec - d.p0 * d.plane] = list[k].v;
}
}  // namespace

struct Tb2Sched {  // work lists of the persistent time-tiled sweep for one plane range (device arrays, sweep_tb.cuh Sched)
    tb::Segment *bulk = nullptr, *segs = nullptr;
    int *first = nullptr, *counters = nullptr;
    int ncta = 0, nbulk = 0;
};

// The one path between host memory and the device: two device slots, the copy of one on `copy` overlapping the
// kernels of the other on s_main.  free[b] is recorded when the last user of slot b is done (the kernels that read it,
// or the copy that drained it), full[b] when its contents are ready for the other side.  The array files also get
// pinned host halves of the slot size.  Everything is allocated on first use (ring_reserve).
struct StagingRing {
    cudaStream_t copy = nullptr;
    cudaEvent_t free[2] = {nullptr, nullptr}, full[2] = {nullptr, nullptr};
    void* slot[2] = {nullptr, nullptr};
    unsigned char* host[2] = {nullptr, nullptr};
    size_t bytes = 0;  // of one slot (and of one pinned half)
};

struct wafer_ctx {
    wafer_params p{};
    Geom g{};
    int dev = 0, sm_count = 0;
    int rank = 0, world = 1;
    bool onfly = true;
    bool use_tb = false;            // time-tiled TMA sweep available (ThreePoint, V on the fly)
    CUtensorMap tm_psi[2], tm_v;    // TMA descriptors of the interior of psi[0], psi[1], v
    double* hfield = nullptr;       // h = (dt*v)/2 for the time-tiled sweep, rebuilt when V changes
    CUtensorMap tm_h;
    bool h_valid = false;
    int den_ok = 0;                 // den_in_fast_window(denominator): the sweeps' fast division is exact
    std::map<std::pair<int, int>, Tb2Sched> tb2_sched;  // keyed by the plane range [xb, xe)
    bool use_t1 = false;            // TMA-pipelined one-step sweep (WAFER_FLAG_TMA_ONE_STEP)
    CUtensorMap t1_psi[2], t1_v, t1_h;
    cudaStream_t s_main = nullptr, s_halo = nullptr;
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr, ev_main = nullptr, ev_halo = nullptr;
    double* psi[2] = {nullptr, nullptr};
    int cur = 0;
    double *v = nullptr, *a = nullptr, *b = nullptr, *potsub_arr = nullptr;
    int potsub_mode = 0;
    double potsub_scalar = 0.0;
    std::vector<double*> lowers;
    // CUDA graph of TWO excited-state steps (sweep + coefficients + projection, twice: the ping-pong parity returns), per
    // (wnum, cur): small lattices are launch bound there (three dependent launches of a few microseconds per step)
    std::map<std::pair<int, int>, std::pair<cudaGraphExec_t, int>> step_graphs;  // exec, kernel launches per replay
    bool chk_valid = false;    // scal[SL_CHK..] holds the point-wise check sums of the CURRENT psi (this rank's share)
    double* gram = nullptr;    // G[i][j] = <q_i, q_j>, j < i, of the stored states (device, GRAM_LD x GRAM_LD)
    StagingRing ring;
    EncTable* pow10 = nullptr;      // the 128-bit power table of the encoder and the decoder (allocated on first use)
    // wafer_write_array: the encoder's block totals / offsets, the refused sites of one launch and the host text of
    // those, the all-reduce vector (all allocated on first use)
    unsigned int* wr_btot = nullptr;
    unsigned long long* wr_boff = nullptr;
    long long wr_blocks = 0;        // blocks wr_btot / wr_boff hold
    EncFlagIn* wr_flags = nullptr;
    EncFlagStr* wr_txt = nullptr;
    unsigned long long* wr_count = nullptr;  // [0] refused sites collected, [1] refused sites the emit pass did not find
    unsigned long long* wr_red = nullptr;
    // wafer_load_array, per slot of the ring: the decoder's block counts and record offsets, the uncertified numbers, the
    // chunk's state words (DEC_ERR, DEC_NFLAG) and their pinned mirror; the running record count
    unsigned int* rd_bcount[2] = {nullptr, nullptr};
    unsigned long long* rd_boff[2] = {nullptr, nullptr};
    DecFlag* rd_flags[2] = {nullptr, nullptr};
    unsigned long long* rd_st = nullptr;    // 2 x DEC_WORDS, then the running record count
    unsigned long long* rd_hst = nullptr;   // pinned, 2 x DEC_WORDS
    long long rd_blocks = 0;                // blocks rd_bcount / rd_boff hold
    double* partials = nullptr;
    long long partials_cap = 0;
    double* scal = nullptr;
    double* h_scal = nullptr;  // pinned mirror for D2H of scalars
    int* ring_flag = nullptr;
    bool have_v = false, have_phi = false;
    uint64_t launches = 0;
    NcclComm comm = nullptr;
    // fused halo over peer memory (CUDA IPC): neighbour 0 = rank-1 (lower x), 1 = rank+1
    bool p2p = false;
    double* peer_psi[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};  // [neighbour][buffer index]
    unsigned long long* flags = nullptr;                  // [0] written by rank-1, [1] by rank+1: passes completed
    unsigned long long* peer_flags[2] = {nullptr, nullptr};
    int* p2p_timeout = nullptr;                           // device flag: a wait gave up (peer died)
    unsigned long long pass = 0;                          // boundary passes completed (same on every rank)
    int peer_L[2] = {0, 0};
    int min_L = 0;                                        // smallest slab over all ranks: uniform overlap decision
    unsigned long long dbg_halo_delay_ns = 0;             // fault injection: stall this rank's halo stream every pass
    unsigned long long* d_cksum = nullptr;
    mutable std::string err;
    size_t bytes() const { return (size_t)g.total() * sizeof(double); }
};

static void drop_step_graphs(wafer_ctx* ctx) {
    for (auto& kv : ctx->step_graphs) cudaGraphExecDestroy(kv.second.first);
    ctx->step_graphs.clear();
}

#define CK(call)                                                                                        \
    do {                                                                                                \
        cudaError_t e_ = (call);                                                                        \
        if (e_ != cudaSuccess) {                                                                        \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                             \
            return WAFER_ERR_CUDA;                                                                      \
        }                                                                                               \
    } while (0)

#define NK(call)                                                                                        \
    do {                                                                                                \
        int r_ = (call);                                                                                \
        if (r_ != kNcclSuccess) {                                                                       \
            ctx->err = std::string(#call) + ": " + nccl_api().GetErrorString(r_);                      \
            return WAFER_ERR_NCCL;                                                                      \
        }                                                                                               \
    } while (0)

#define REQUIRE(cond, msg)                                                                              \
    do {                                                                                                \
        if (!(cond)) {                                                                                  \
            ctx->err = msg;                                                                             \
            return WAFER_ERR_INVALID;                                                                   \
        }                                                                                               \
    } while (0)

#define TRY(expr)                                                                                       \
    do {                                                                                                \
        int t_ = (expr);                                                                                \
        if (t_ != WAFER_OK) return t_;                                                                  \
    } while (0)

namespace {

inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

double denominator(const wafer_ctx* c) {
    // grid.rs:569/594/626: r64(k)*dn*dn*mass, left to right
    const double k = c->p.ext == 1 ? 2. : (c->p.ext == 2 ? 24. : 360.);
    return k * c->p.dn * c->p.dn * c->p.mass;
}

// the exponent window of den in which tb::div_fast is exact (sweep_tb.cuh DivConst): 2^-100 < den < 2^100
int den_in_fast_window(double den) { return den > 0x1p-100 && den < 0x1p100 ? 1 : 0; }

int post_launch(wafer_ctx* ctx, int n = 1) {
    ctx->launches += n;
    CK(cudaGetLastError());
    return WAFER_OK;
}

int ew_grid(const wafer_ctx* ctx, long long n2) {
    return (int)std::min<long long>(ceil_div(n2, EW_THREADS), (long long)ctx->sm_count * 8);
}

// reduce `ns` rows of `nblocks` partials into scal[slot..slot+ns) and all-reduce across ranks
int finalize(wafer_ctx* ctx, int ns, int nblocks, int slot, cudaStream_t st) {
    if (ns == 1) finalize_kernel<1><<<1, 1024, 0, st>>>(ctx->partials, nblocks, ctx->scal + slot);
    else finalize_kernel<4><<<1, 1024, 0, st>>>(ctx->partials, nblocks, ctx->scal + slot);
    TRY(post_launch(ctx));
    if (ctx->world > 1)
        NK(nccl_api().AllReduce(ctx->scal + slot, ctx->scal + slot, ns, kNcclFloat64, kNcclSum, ctx->comm, st));
    return WAFER_OK;
}

__global__ void set_scalar_kernel(double* p, double v) { *p = v; }

// ---- sweep dispatch ------------------------------------------------------------------------------------
template <int E>
int launch_sweep_simple(wafer_ctx* ctx, const double* cur, double* nxt, int xb, int xe, bool norm, long long part_off,
                        cudaStream_t st) {
    const Geom& g = ctx->g;
    if (xe <= xb) return WAFER_OK;
    dim3 grid(ceil_div(g.nz, 2 * SW_BX), ceil_div(g.ny, SW_BY), ceil_div(xe - xb, SW_XCH)), block(SW_BX, SW_BY);
    const double den = denominator(ctx), dt = ctx->p.dt;
    double* part = ctx->partials + part_off;
    const double* fa = ctx->onfly ? ctx->v : ctx->a;
    const double* fb = ctx->b;
    if (ctx->onfly) {
        if (norm) sweep_simple_kernel<E, true, true><<<grid, block, 0, st>>>(cur, nxt, fa, fb, g, xb, xe, dt, den, part);
        else sweep_simple_kernel<E, true, false><<<grid, block, 0, st>>>(cur, nxt, fa, fb, g, xb, xe, dt, den, part);
    } else {
        if (norm) sweep_simple_kernel<E, false, true><<<grid, block, 0, st>>>(cur, nxt, fa, fb, g, xb, xe, dt, den, part);
        else sweep_simple_kernel<E, false, false><<<grid, block, 0, st>>>(cur, nxt, fa, fb, g, xb, xe, dt, den, part);
    }
    return post_launch(ctx);
}

int simple_blocks(const wafer_ctx* ctx, int xb, int xe) {
    const Geom& g = ctx->g;
    return ceil_div(g.nz, 2 * SW_BX) * ceil_div(g.ny, SW_BY) * ceil_div(xe - xb, SW_XCH);
}

// forward declarations of the TMA one-step path (defined below, next to the tensor-map helpers)
template <int E> int launch_sweep_t1(wafer_ctx* ctx, int src, int xb, int xe, int mode, cudaStream_t st, int nb_total, int bid_off);
template <int E> int t1_blocks(const wafer_ctx* ctx, int xb, int xe);

// number of per-CTA partial sums the fused-norm sweep over [xb, xe) leaves in ctx->partials
int sweep_blocks(const wafer_ctx* ctx, int xb, int xe);

int launch_sweep(wafer_ctx* ctx, const double* cur, double* nxt, int xb, int xe, int nred, long long part_off,
                 cudaStream_t st, int nb_total = 0, int bid_off = 0);

int launch_sweep_plain(wafer_ctx* ctx, const double* cur, double* nxt, int xb, int xe, bool norm, long long part_off,
                       cudaStream_t st) {
    switch (ctx->p.ext) {
        case 1: return launch_sweep_simple<1>(ctx, cur, nxt, xb, xe, norm, part_off, st);
        case 2: return launch_sweep_simple<2>(ctx, cur, nxt, xb, xe, norm, part_off, st);
        default: return launch_sweep_simple<3>(ctx, cur, nxt, xb, xe, norm, part_off, st);
    }
}

// ---- time-tiled TMA sweep (sweep_tb.cuh): two steps per launch ----------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int make_tensor_map(wafer_ctx* ctx, CUtensorMap* tm, double* field, int box_rows) {  // 64-column boxes
    static EncodeTiledFn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        CK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (!fn || qres != cudaDriverEntryPointSuccess) { ctx->err = "cuTensorMapEncodeTiled not available"; return WAFER_ERR_CUDA; }
        encode = (EncodeTiledFn)fn;
    }
    const Geom& g = ctx->g;
    // the tensor is the lattice interior only: (nz, ny, L+2gx) with the device pitches; everything outside it
    // (y ghost rows, z pads, planes beyond the ghosts) is produced by the TMA zero fill
    cuuint64_t dims[3] = {(cuuint64_t)g.nz, (cuuint64_t)g.ny, (cuuint64_t)(g.L + 2 * g.gx)};
    cuuint64_t strides[2] = {(cuuint64_t)g.zp * sizeof(double), (cuuint64_t)g.plane * sizeof(double)};
    cuuint32_t box[3] = {(cuuint32_t)tb::BW, (cuuint32_t)box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = encode(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, field + (long long)g.e * g.zp, dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { ctx->err = "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")"; return WAFER_ERR_CUDA; }
    return WAFER_OK;
}

int init_tb(wafer_ctx* ctx) {
    ctx->use_tb = false;
    if (ctx->p.ext != 1 || !ctx->onfly || (ctx->p.flags & WAFER_FLAG_SIMPLE_SWEEP)) return WAFER_OK;
    TRY(make_tensor_map(ctx, &ctx->tm_psi[0], ctx->psi[0], tb::R0));
    TRY(make_tensor_map(ctx, &ctx->tm_psi[1], ctx->psi[1], tb::R0));
    TRY(make_tensor_map(ctx, &ctx->tm_v, ctx->v, tb::R1));
    CK(cudaFuncSetAttribute(tb::sweep_tb2_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tb::SMEM_BYTES));
    CK(cudaFuncSetAttribute(tb::sweep_tb2_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tb::SMEM_BYTES));
    CK(cudaFuncSetAttribute(tb::sweep_tb2_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tb::SMEM_BYTES));
    CK(cudaFuncSetAttribute(tb::sweep_tb2_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tb::SMEM_BYTES));
    ctx->use_tb = true;
    return WAFER_OK;
}

// ---- work distribution of the time-tiled sweep (persistent grid; see sweep_tb.cuh Sched) ---------------------------
// Every segment pays 4 plane-iterations of pipeline fill; CTAs that share a tile edge re-read each other's halo cells,
// from L2 only if they pass the same planes at about the same time; and the SMs should finish together.
//   * x is cut into chunks of at most 512 planes; per chunk, whole tile columns in tile order form the BULK list that the
//     CTAs drain through an atomic counter (in-order dispatch keeps neighbouring tiles close in time);
//   * of the last chunk, the ntiles % G columns that would leave most SMs idle in a last partial wave are cut along x
//     into at most G equal shares (even lengths, no stubs shorter than 6 planes): the static TAIL of each CTA.
//   * few tile columns on many CTAs (fewer than 3/4 of a column per CTA: small planes, whose halos live in L2 anyway):
//     no bulk, one contiguous static run of the columns x planes per CTA.
// 512^3 on 148 SMs: one round of 148 columns + 14 columns cut 148 ways = 516 + ~53 plane-iterations per SM, against
// 10 waves x 60 for round 1's uniform grid of 162 tiles x 9 chunks.  The policies measured against this one (round 1's
// grid, statically assigned rounds, one contiguous split everywhere) are in profiles/r2_tb2_variants.md.
// pure host arithmetic (also behind wafer_tb2_plan for the CPU tests): bulk = in-order list, per[k] = static tail of CTA k
struct Tb2Plan {
    std::vector<tb::Segment> bulk;
    std::vector<std::vector<tb::Segment>> per;
};
constexpr int TB2_MAXSEG = 512;  // planes per x chunk of the bulk, at most
Tb2Plan tb2_plan(int ny, int nz, int xb, int xe, int slots) {
    Tb2Plan pl;
    std::vector<tb::Segment>& bulk = pl.bulk;
    std::vector<std::vector<tb::Segment>>& per = pl.per;
    const int ntz = ceil_div(nz, tb::TZ), nty = ceil_div(ny, tb::TY), ntiles = ntz * nty, P = xe - xb;
    auto seg = [&](int tile, int a, int b) { return tb::Segment{(tile / ntz) * tb::TY, (tile % ntz) * tb::TZ, a, b}; };
    const int MINSEG = 6;
    int G = (int)std::max<long long>(1, std::min<long long>(slots, ((long long)ntiles * P + 7) / 8));
    // shares of `cols` tile columns starting at tile `t0`, planes [ca, cz), cut into equal runs -> per[k].  At most
    // Ur / MINSEG shares: a thin slab of a wide plane leaves less than MINSEG planes per CTA, and cutting it G ways would
    // give stubs of 2-4 planes that are mostly pipeline fill; the CTAs past the last share get no tail.
    auto cut_static = [&](int t0, int cols, int ca, int cz) {
        const int Pc = cz - ca;
        const long long Ur = (long long)cols * Pc;
        const int S = (int)std::max<long long>(1, std::min<long long>(G, Ur / MINSEG));
        auto snap = [&](long long u) {
            const long long p = u % Pc;
            if (p == 0) return u;
            if (p < MINSEG) return u - p;
            if (Pc - p < MINSEG) return u + (Pc - p);
            return u - (p & 1);
        };
        for (int k = 0; k < S && Ur > 0; ++k) {
            long long u = snap(k * Ur / S);
            const long long ue = k + 1 == S ? Ur : snap((k + 1) * Ur / S);
            while (u < ue) {
                const int p0 = (int)(u % Pc), len = (int)std::min<long long>(Pc - p0, ue - u);
                per[k].push_back(seg(t0 + (int)(u / Pc), ca + p0, ca + p0 + len));
                u += len;
            }
        }
    };
    if (ntiles * 4 < G * 3) {
        // few tile columns on many CTAs (small planes: every halo lives in L2 anyway): one contiguous static run each
        per.resize(G);
        cut_static(0, ntiles, xb, xe);
        return pl;
    }
    if (ntiles < G) G = ntiles;  // nearly one column per CTA: leave the few spare SMs idle, keep lock step
    per.resize(G);
    // number of x chunks: at least P / TB2_MAXSEG; a few more if that leaves a smaller statically cut tail.  The tail runs
    // out of lock step (its halo re-reads miss L2), which the estimate charges with an empirical factor of 1.6.
    int nchunk = ceil_div(P, TB2_MAXSEG);
    double best = 1e300;
    for (int nc = ceil_div(P, TB2_MAXSEG); nc <= ceil_div(P, TB2_MAXSEG) + 6 && nc * 32 <= P; ++nc) {
        const int ch = (ceil_div(P, nc) + 1) & ~1;
        const long long items = (long long)nc * ntiles, rest = items % G;
        const double cost = (double)(items / G) * (ch + 4) + (rest ? ((double)rest * ch / G + 4) * 1.6 : 0.0);
        if (cost < best * 0.999) { best = cost; nchunk = nc; }
    }
    // in-order dispatch of whole columns, chunk after chunk
    const int chunk = (ceil_div(P, nchunk) + 1) & ~1;
    for (int c = 0; c * chunk < P; ++c) {
        const int ca = xb + c * chunk, cz = std::min(xe, ca + chunk);
        for (int t = 0; t < ntiles; ++t) bulk.push_back(seg(t, ca, cz));
    }
    // the bulk must come out even — a multiple of G columns — or the CTAs that drew one column more finish a whole
    // column late: the last bulk.size() % G columns (all in the last chunk) are cut into G equal static shares
    const int rest = std::min((int)(bulk.size() % G), ntiles);  // (never reaches back into an earlier chunk)
    if (rest > 0) {
        const tb::Segment f = bulk[bulk.size() - rest];
        const int t0 = (f.y0 / tb::TY) * ntz + f.z0 / tb::TZ;
        bulk.resize(bulk.size() - rest);
        cut_static(t0, rest, f.xa, f.xz);
    }
    return pl;
}

int tb2_schedule(wafer_ctx* ctx, int xb, int xe, const Tb2Sched** out) {
    auto it = ctx->tb2_sched.find({xb, xe});
    if (it != ctx->tb2_sched.end()) { *out = &it->second; return WAFER_OK; }
    const Tb2Plan pl = tb2_plan(ctx->g.ny, ctx->g.nz, xb, xe, ctx->sm_count * tb::CTAS_PER_SM);
    const std::vector<tb::Segment>& bulk = pl.bulk;
    std::vector<tb::Segment> flat;
    std::vector<int> first{0};
    for (const auto& v : pl.per) {
        flat.insert(flat.end(), v.begin(), v.end());
        first.push_back((int)flat.size());
    }
    Tb2Sched sc;
    sc.ncta = (int)pl.per.size();
    sc.nbulk = (int)bulk.size();
    CK(cudaMalloc(&sc.bulk, std::max<size_t>(bulk.size(), 1) * sizeof(tb::Segment)));
    CK(cudaMalloc(&sc.segs, std::max<size_t>(flat.size(), 1) * sizeof(tb::Segment)));
    CK(cudaMalloc(&sc.first, first.size() * sizeof(int)));
    CK(cudaMalloc(&sc.counters, 2 * sizeof(int)));
    CK(cudaMemsetAsync(sc.counters, 0, 2 * sizeof(int), ctx->s_main));
    if (!bulk.empty()) CK(cudaMemcpyAsync(sc.bulk, bulk.data(), bulk.size() * sizeof(tb::Segment), cudaMemcpyHostToDevice, ctx->s_main));
    if (!flat.empty()) CK(cudaMemcpyAsync(sc.segs, flat.data(), flat.size() * sizeof(tb::Segment), cudaMemcpyHostToDevice, ctx->s_main));
    CK(cudaMemcpyAsync(sc.first, first.data(), first.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->s_main));
    CK(cudaStreamSynchronize(ctx->s_main));  // the host vectors die here; any stream may launch with the schedule afterwards
    *out = &(ctx->tb2_sched[{xb, xe}] = sc);
    return WAFER_OK;
}

// The time-tiled sweep reads h = (dt*v)/2 instead of V: same bytes, two DMULs less per site and sweep pair, at the price
// of one more field in HBM.  Built lazily on the main stream; every launch of the sweep is ordered after it there.  Until
// h exists (evolves of fewer than 4 steps) or when there is no room for it, the sweep reads V.
// The one-step TMA sweeps can read h too (WAFER_T1_HFIELD=1); measured: no difference for them (5/7-point, excited
// steps within 0.5 %, gpurun_out/r2z) — they are not limited by those two multiplications — so it is off by default.
bool t1_reads_h() {
    static const bool on = getenv("WAFER_T1_HFIELD") && atoi(getenv("WAFER_T1_HFIELD")) == 1;
    return on;
}

int ensure_hfield(wafer_ctx* ctx) {
    if (ctx->h_valid) return WAFER_OK;
    if (!ctx->hfield) {
        if (cudaMalloc(&ctx->hfield, ctx->bytes()) != cudaSuccess) { cudaGetLastError(); ctx->hfield = nullptr; return WAFER_OK; }  // no room: keep V
        TRY(make_tensor_map(ctx, &ctx->tm_h, ctx->hfield, tb::R1));
        if (ctx->use_t1) {
            const int rows = ctx->p.ext == 1 ? t1::Cfg<1>::TY : (ctx->p.ext == 2 ? t1::Cfg<2>::TY : t1::Cfg<3>::TY);
            TRY(make_tensor_map(ctx, &ctx->t1_h, ctx->hfield, rows));
        }
    }
    const long long n = ctx->g.total();
    build_h_kernel<<<ew_grid(ctx, n), EW_THREADS, 0, ctx->s_main>>>(ctx->v, ctx->hfield, n, ctx->p.dt);
    TRY(post_launch(ctx));
    ctx->h_valid = true;
    return WAFER_OK;
}

// two lattice steps: psi[src] -> psi[src^1] for planes [xb, xe); pr != nullptr: also store the boundary planes it names
// into the neighbours' ghost planes (fused halo)
int launch_sweep_tb2(wafer_ctx* ctx, int src, int xb, int xe, cudaStream_t st, const tb::PeerStores* pr = nullptr) {
    if (xe <= xb) return WAFER_OK;
    const Geom& g = ctx->g;
    const bool hf = ctx->h_valid;
    const Tb2Sched* sc = nullptr;
    TRY(tb2_schedule(ctx, xb, xe, &sc));
    double* out = ctx->psi[src ^ 1];
    const tb::Sched ks{sc->bulk, sc->nbulk, sc->segs, sc->first, sc->counters};
    if (pr) {
        if (hf) tb::sweep_tb2_kernel<true, true><<<sc->ncta, tb::THREADS, tb::SMEM_BYTES, st>>>(ctx->tm_psi[src], ctx->tm_h, out, *pr, g, ks, ctx->p.dt, denominator(ctx), ctx->den_ok);
        else tb::sweep_tb2_kernel<true, false><<<sc->ncta, tb::THREADS, tb::SMEM_BYTES, st>>>(ctx->tm_psi[src], ctx->tm_v, out, *pr, g, ks, ctx->p.dt, denominator(ctx), ctx->den_ok);
    } else {
        const tb::PeerStores none{};
        if (hf) tb::sweep_tb2_kernel<false, true><<<sc->ncta, tb::THREADS, tb::SMEM_BYTES, st>>>(ctx->tm_psi[src], ctx->tm_h, out, none, g, ks, ctx->p.dt, denominator(ctx), ctx->den_ok);
        else tb::sweep_tb2_kernel<false, false><<<sc->ncta, tb::THREADS, tb::SMEM_BYTES, st>>>(ctx->tm_psi[src], ctx->tm_v, out, none, g, ks, ctx->p.dt, denominator(ctx), ctx->den_ok);
    }
    return post_launch(ctx);
}

// ---- TMA-pipelined one-step sweep (sweep_tma1.cuh), opt-in ---------------------------------------------------
template <int E>
int t1_tiles(const Geom& g) { return ceil_div(g.nz, t1::Cfg<E>::TZ) * ceil_div(g.ny, t1::Cfg<E>::TY); }

template <int E>
int t1_chunks(const wafer_ctx* ctx, int planes) {
    const long long tiles = t1_tiles<E>(ctx->g);
    int best_nc = 1;
    double best_cost = 1e300;
    for (int nc = 1; nc <= std::min(planes, 64); ++nc) {
        const double cost = (double)ceil_div(tiles * nc, ctx->sm_count) * ((double)ceil_div(planes, nc) + 2.0 * E);
        if (cost < best_cost * 0.999) { best_cost = cost; best_nc = nc; }
    }
    return best_nc;
}

// every instantiated mode of the TMA one-step kernel (sweep_tma1.cuh): sweeps with 0..5 running sums, observables with
// pot_sub none / scalar / array / energy only, sweeps that also leave the check's point-wise sums
#define T1_MODES(X) X(0) X(1) X(2) X(3) X(4) X(5) X(8) X(9) X(10) X(11) X(16) X(17) X(18)

template <int E>
int init_t1_e(wafer_ctx* ctx) {
    TRY(make_tensor_map(ctx, &ctx->t1_psi[0], ctx->psi[0], t1::Cfg<E>::R0));
    TRY(make_tensor_map(ctx, &ctx->t1_psi[1], ctx->psi[1], t1::Cfg<E>::R0));
    TRY(make_tensor_map(ctx, &ctx->t1_v, ctx->v, t1::Cfg<E>::TY));
    const int smem = (int)sizeof(t1::Smem<E>);
#define T1_ATTR(M) CK(cudaFuncSetAttribute(t1::sweep_tma1_kernel<E, M>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    T1_MODES(T1_ATTR)
#undef T1_ATTR
    return WAFER_OK;
}

int init_t1(wafer_ctx* ctx) {
    ctx->use_t1 = false;
    // the default one-step kernel whenever V is kept on the fly (13-24 % faster than the register-queue kernel for
    // 5/7-point, profiles/r1_tma1_one_step.md); boundary / interior sub-range launches of slab runs use it too
    const bool asked = (ctx->p.flags & WAFER_FLAG_TMA_ONE_STEP) != 0;
    const bool by_default = !(ctx->p.flags & WAFER_FLAG_SIMPLE_SWEEP);
    if (!ctx->onfly || !(asked || by_default)) return WAFER_OK;
    if (ctx->p.ext == 1) TRY(init_t1_e<1>(ctx));
    else if (ctx->p.ext == 2) TRY(init_t1_e<2>(ctx));
    else TRY(init_t1_e<3>(ctx));
    ctx->use_t1 = true;
    return WAFER_OK;
}

// mode (sweep_tma1.cuh): 0 plain sweep; 1 fused sum psi'^2; 1 + k: additionally the overlaps with stored states
// 0..k-1 (k <= 4); MODE_OBS + p: observables of psi[src], nothing stored; MODE_CHK + p: sweep + the check's point-wise sums.
// nb_total / bid_off: several launches (boundary + interior planes) share one row of per-CTA partial sums.
template <int E>
int launch_sweep_t1(wafer_ctx* ctx, int src, int xb, int xe, int mode, cudaStream_t st, int nb_total, int bid_off) {
    if (xe <= xb) return WAFER_OK;
    const Geom& g = ctx->g;
    const int planes = xe - xb, chunk = ceil_div(planes, t1_chunks<E>(ctx, planes));
    dim3 grid(ceil_div(g.nz, t1::Cfg<E>::TZ), ceil_div(g.ny, t1::Cfg<E>::TY), ceil_div(planes, chunk));
    const size_t smem = sizeof(t1::Smem<E>);
    t1::Extra ex{};
    if (mode < t1::MODE_OBS)
        for (int i = 0; i + 1 < mode; ++i) ex.q[i] = ctx->lowers[i];
    ex.potsub_arr = ctx->potsub_arr;
    ex.potsub = ctx->potsub_scalar;
    ex.nb_total = nb_total;
    ex.bid_off = bid_off;
    const bool sweep_mode = mode < t1::MODE_OBS || mode >= t1::MODE_CHK;
    ex.hf = t1_reads_h() && sweep_mode && ctx->h_valid ? 1 : 0;
    const CUtensorMap& tmv = ex.hf ? ctx->t1_h : ctx->t1_v;
    // the observables modes read psi[src] and store nothing: `out` only anchors the element offsets
    double* out = (mode >= t1::MODE_OBS && mode < t1::MODE_CHK) ? ctx->psi[src] : ctx->psi[src ^ 1];
#define T1_CASE(M)                                                                                                              \
    case M:                                                                                                                     \
        t1::sweep_tma1_kernel<E, M><<<grid, t1::Cfg<E>::THREADS, smem, st>>>(ctx->t1_psi[src], tmv, out, g, xb, xe, chunk,           \
                                                                             ctx->p.dt, denominator(ctx), ctx->den_ok, ctx->partials, ex); \
        break;
    switch (mode) {
        T1_MODES(T1_CASE)
        default: ctx->err = "internal: unknown mode of the TMA one-step kernel"; return WAFER_ERR_INVALID;
    }
#undef T1_CASE
    return post_launch(ctx);
}

template <int E>
int t1_blocks(const wafer_ctx* ctx, int xb, int xe) {
    const int planes = xe - xb, chunk = ceil_div(planes, t1_chunks<E>(ctx, planes));
    return t1_tiles<E>(ctx->g) * ceil_div(planes, chunk);
}

int sweep_blocks(const wafer_ctx* ctx, int xb, int xe) {
    if (!ctx->use_t1) return simple_blocks(ctx, xb, xe);
    return ctx->p.ext == 1 ? t1_blocks<1>(ctx, xb, xe) : (ctx->p.ext == 2 ? t1_blocks<2>(ctx, xb, xe) : t1_blocks<3>(ctx, xb, xe));
}

// one lattice step cur -> nxt for planes [xb, xe): TMA-pipelined kernel when enabled, register-queue kernel otherwise.
// nred > 1 (fused overlaps) is only available in the TMA kernel: callers ask fused_lowers() first.
int launch_sweep(wafer_ctx* ctx, const double* cur, double* nxt, int xb, int xe, int nred, long long part_off,
                 cudaStream_t st, int nb_total, int bid_off) {
    if (!ctx->use_t1) return launch_sweep_plain(ctx, cur, nxt, xb, xe, nred > 0, part_off, st);
    const int src = cur == ctx->psi[0] ? 0 : 1;
    if (nxt != ctx->psi[src ^ 1]) { ctx->err = "internal: sweep buffers are not the ping-pong pair"; return WAFER_ERR_INVALID; }
    switch (ctx->p.ext) {
        case 1: return launch_sweep_t1<1>(ctx, src, xb, xe, nred, st, nb_total, bid_off);
        case 2: return launch_sweep_t1<2>(ctx, src, xb, xe, nred, st, nb_total, bid_off);
        default: return launch_sweep_t1<3>(ctx, src, xb, xe, nred, st, nb_total, bid_off);
    }
}

// ---- inter-GPU ordering for the fused halo: monotone pass counters in peer-visible memory ------------------
// flags[0] is written by rank-1, flags[1] by rank+1 ("my boundary planes of pass n are in your ghost planes and I
// no longer read the ghost planes you are about to overwrite").  Spins are bounded (~30 s) so a dead peer cannot
// hang the GPU.
__global__ void p2p_wait_kernel(const volatile unsigned long long* flags, unsigned long long need, int has_lo, int has_hi,
                                int* timeout_flag) {
    unsigned long long t0, t1;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t0));
    for (int n = 0; n < 2; ++n) {
        if (!(n == 0 ? has_lo : has_hi)) continue;
        while (flags[n] < need) {
            asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t1));
            if (t1 - t0 > 30000000000ull) { *timeout_flag = 1; return; }
            __nanosleep(200);
        }
    }
    __threadfence_system();  // acquire: the neighbour's ghost-plane stores precede its flag store
}
__global__ void p2p_signal_kernel(volatile unsigned long long* peer_lo, volatile unsigned long long* peer_hi,
                                  unsigned long long value) {
    __threadfence_system();  // release: every store of the preceding kernels in this stream (incl. peer stores)
    if (peer_lo) peer_lo[1] = value;  // I am rank-1's upper neighbour
    if (peer_hi) peer_hi[0] = value;  // I am rank+1's lower neighbour
    __threadfence_system();
}

// ghost-plane halo exchange of `buf` with the x neighbours (NCCL send/recv over NVLink)
int exchange(wafer_ctx* ctx, double* buf, cudaStream_t st) {
    if (ctx->world <= 1) return WAFER_OK;
    const Geom& g = ctx->g;
    // gx planes each way (gx = 2 for the time-tiled ThreePoint sweep, else ext): whole planes are contiguous
    const size_t cnt = (size_t)g.gx * g.plane;
    NcclApi& n = nccl_api();
    NK(n.GroupStart());
    if (ctx->rank > 0) {
        NK(n.Send(buf + g.off(0, -g.e, 0), cnt, kNcclFloat64, ctx->rank - 1, ctx->comm, st));
        NK(n.Recv(buf + g.off(-g.gx, -g.e, 0), cnt, kNcclFloat64, ctx->rank - 1, ctx->comm, st));
    }
    if (ctx->rank < ctx->world - 1) {
        NK(n.Send(buf + g.off(g.L - g.gx, -g.e, 0), cnt, kNcclFloat64, ctx->rank + 1, ctx->comm, st));
        NK(n.Recv(buf + g.off(g.L, -g.e, 0), cnt, kNcclFloat64, ctx->rank + 1, ctx->comm, st));
    }
    NK(n.GroupEnd());
    return WAFER_OK;
}

// ---- normalise + Gram-Schmidt (grid.rs:465-492) in two passes: see kernels.cuh (dots / coefficients / projection) ----
LowerPtrs lower_group(const wafer_ctx* ctx, int first, int count) {
    LowerPtrs lw{};
    for (int i = 0; i < count; ++i) lw.q[i] = ctx->lowers[first + i];
    return lw;
}

// raw overlaps of `psi` with stored states [first, first+count), count <= GS_GROUP -> scal[SL_RAW + 1 + first ...]
int dots_group(wafer_ctx* ctx, const double* psi, int first, int count) {
    const Geom& g = ctx->g;
    const long long ob = (long long)g.gx * g.plane / 2, oe = (long long)(g.gx + g.L) * g.plane / 2;
    const int grid = ew_grid(ctx, oe - ob);
    const LowerPtrs lw = lower_group(ctx, first, count);
    switch (count) {
        case 1: dots_kernel<1><<<grid, EW_THREADS, 0, ctx->s_main>>>(psi, lw, ob, oe, ctx->partials); break;
        case 2: dots_kernel<2><<<grid, EW_THREADS, 0, ctx->s_main>>>(psi, lw, ob, oe, ctx->partials); break;
        case 3: dots_kernel<3><<<grid, EW_THREADS, 0, ctx->s_main>>>(psi, lw, ob, oe, ctx->partials); break;
        default: dots_kernel<4><<<grid, EW_THREADS, 0, ctx->s_main>>>(psi, lw, ob, oe, ctx->partials); break;
    }
    TRY(post_launch(ctx));
    gs_coeff_kernel<true, false><<<1, 1024, 0, ctx->s_main>>>(ctx->partials, grid, count, ctx->scal + SL_RAW + 1 + first, 0, nullptr,
                                                                nullptr, nullptr, 0, nullptr);
    return post_launch(ctx);
}

int project(wafer_ctx* ctx, double* psi, const double* norm2_ptr, int wnum) {
    const long long n2 = ctx->g.total() / 2;
    const int grid = ew_grid(ctx, n2);
    if (wnum == 0) {
        if (norm2_ptr) {
            project_kernel<0, true><<<grid, EW_THREADS, 0, ctx->s_main>>>(psi, n2, norm2_ptr, LowerPtrs{}, nullptr);
            TRY(post_launch(ctx));
        }
        return WAFER_OK;
    }
    for (int first = 0; first < wnum; first += GS_GROUP) {
        const int count = std::min(GS_GROUP, wnum - first);
        const LowerPtrs lw = lower_group(ctx, first, count);
        const double* coef = ctx->scal + SL_COEF + first;
        const bool nrm = first == 0 && norm2_ptr;
#define PROJ(K)                                                                                                  \
    if (nrm) project_kernel<K, true><<<grid, EW_THREADS, 0, ctx->s_main>>>(psi, n2, norm2_ptr, lw, coef);        \
    else project_kernel<K, false><<<grid, EW_THREADS, 0, ctx->s_main>>>(psi, n2, nullptr, lw, coef)
        switch (count) {
            case 1: PROJ(1); break;
            case 2: PROJ(2); break;
            case 3: PROJ(3); break;
            default: PROJ(4); break;
        }
#undef PROJ
        TRY(post_launch(ctx));
    }
    return WAFER_OK;
}

// psi <- normalise(psi, *norm2_ptr) (norm2_ptr == nullptr: skip) then orthogonalise against stored states [0, wnum).
// have: the raw overlaps with the first `have` states (and, in raw[0], sum psi^2) already sit in ctx->partials as
// rows 0..have of `sweep_nb` per-CTA partial sums, left there by the fused sweep.
int gs_apply(wafer_ctx* ctx, double* psi, const double* norm2_ptr, int wnum, int have_rows = 0, int sweep_nb = 0) {
    double* raw = ctx->scal + SL_RAW;
    const bool one_launch = ctx->world == 1 && have_rows == wnum + 1;  // everything came out of the sweep: reduce + solve at once
    if (one_launch) {
        gs_coeff_kernel<true, true><<<1, 1024, 0, ctx->s_main>>>(ctx->partials, sweep_nb, have_rows, raw, wnum, raw + 1, norm2_ptr,
                                                                   ctx->gram, GRAM_LD, ctx->scal + SL_COEF);
        TRY(post_launch(ctx));
        return project(ctx, psi, norm2_ptr, wnum);
    }
    if (have_rows > 0) {
        gs_coeff_kernel<true, false><<<1, 1024, 0, ctx->s_main>>>(ctx->partials, sweep_nb, have_rows, raw, 0, nullptr, nullptr, nullptr,
                                                                    0, nullptr);
        TRY(post_launch(ctx));
    }
    for (int first = std::max(have_rows - 1, 0); first < wnum; first += GS_GROUP)
        TRY(dots_group(ctx, psi, first, std::min(GS_GROUP, wnum - first)));
    if (ctx->world > 1) {
        // one all-reduce per step: [sum psi^2 (when the sweep produced it), overlaps 0..wnum)
        const int off = have_rows > 0 ? 0 : 1, cnt = wnum + 1 - off;
        if (cnt > 0) NK(nccl_api().AllReduce(raw + off, raw + off, cnt, kNcclFloat64, kNcclSum, ctx->comm, ctx->s_main));
    }
    if (wnum > 0) {
        gs_coeff_kernel<false, true><<<1, 32, 0, ctx->s_main>>>(nullptr, 0, 0, raw, wnum, raw + 1, norm2_ptr, ctx->gram, GRAM_LD,
                                                                  ctx->scal + SL_COEF);
        TRY(post_launch(ctx));
    }
    return project(ctx, psi, norm2_ptr, wnum);
}

// a state joins the store: measure its overlaps with the states already there (row of the Gram matrix)
int register_lower(wafer_ctx* ctx, double* q) {
    if (!ctx->gram) CK(cudaMalloc(&ctx->gram, (size_t)GRAM_LD * GRAM_LD * sizeof(double)));
    const int m = (int)ctx->lowers.size();
    for (int first = 0; first < m; first += GS_GROUP) TRY(dots_group(ctx, q, first, std::min(GS_GROUP, m - first)));
    if (m > 0) {
        double* raw = ctx->scal + SL_RAW + 1;
        if (ctx->world > 1) NK(nccl_api().AllReduce(raw, raw, m, kNcclFloat64, kNcclSum, ctx->comm, ctx->s_main));
        CK(cudaMemcpyAsync(ctx->gram + (size_t)m * GRAM_LD, raw, m * sizeof(double), cudaMemcpyDeviceToDevice, ctx->s_main));
    }
    ctx->lowers.push_back(q);
    return WAFER_OK;
}

int observables_device(wafer_ctx* ctx) {
    const Geom& g = ctx->g;
    if (ctx->use_t1) {
        // TMA-pipelined pass (sweep_tma1.cuh MODE_OBS): psi and V stream through the same shared-memory ring as the sweep
        const int nb = sweep_blocks(ctx, 0, g.L);
        if (ctx->chk_valid) {
            // norm2, <pot_sub> and <r2> rode on the last sweep of evolve (grid.rs:405-437 are point-wise in psi): only the
            // energy, which needs the neighbours of the final psi, is left
            TRY(launch_sweep(ctx, ctx->psi[ctx->cur], ctx->psi[ctx->cur ^ 1], 0, g.L, t1::MODE_OBS + 3, 0, ctx->s_main));
            gs_coeff_kernel<true, false><<<1, 1024, 0, ctx->s_main>>>(ctx->partials, nb, 1, ctx->scal + SL_OBS, 0, nullptr, nullptr,
                                                                        nullptr, 0, nullptr);
            TRY(post_launch(ctx));
            CK(cudaMemcpyAsync(ctx->scal + SL_OBS + 1, ctx->scal + SL_CHK, 3 * sizeof(double), cudaMemcpyDeviceToDevice, ctx->s_main));
            if (ctx->world > 1)
                NK(nccl_api().AllReduce(ctx->scal + SL_OBS, ctx->scal + SL_OBS, 4, kNcclFloat64, kNcclSum, ctx->comm, ctx->s_main));
            return WAFER_OK;
        }
        TRY(launch_sweep(ctx, ctx->psi[ctx->cur], ctx->psi[ctx->cur ^ 1], 0, g.L, t1::MODE_OBS + ctx->potsub_mode, 0, ctx->s_main));
        return finalize(ctx, 4, nb, SL_OBS, ctx->s_main);
    }
    dim3 grid(ceil_div(g.nz, SW_BX), ceil_div(g.ny, SW_BY), ceil_div(g.L, SW_XCH)), block(SW_BX, SW_BY);
    const int nb = grid.x * grid.y * grid.z;
    const double den = denominator(ctx);
    const double* cur = ctx->psi[ctx->cur];
#define OBS(E, M) observables_kernel<E, M><<<grid, block, 0, ctx->s_main>>>(cur, ctx->v, ctx->potsub_arr, ctx->potsub_scalar, g, den, ctx->partials)
#define OBS_E(E)                                   \
    if (ctx->potsub_mode == 0) OBS(E, 0);          \
    else if (ctx->potsub_mode == 1) OBS(E, 1);     \
    else OBS(E, 2);
    if (ctx->p.ext == 1) { OBS_E(1) } else if (ctx->p.ext == 2) { OBS_E(2) } else { OBS_E(3) }
#undef OBS_E
#undef OBS
    TRY(post_launch(ctx));
    return finalize(ctx, 4, nb, SL_OBS, ctx->s_main);
}

// a fused-halo wait that gave up (dead or desynchronised neighbour) must not go unnoticed: every call that hands
// numbers back to the host checks the device-side timeout flag after its synchronisation
int check_p2p_timeout(wafer_ctx* ctx) {
    if (!ctx->p2p_timeout) return WAFER_OK;
    int t = 0;
    CK(cudaMemcpyAsync(&t, ctx->p2p_timeout, sizeof(int), cudaMemcpyDeviceToHost, ctx->s_main));
    CK(cudaStreamSynchronize(ctx->s_main));
    if (t) { ctx->err = "fused halo: timed out waiting for a neighbour GPU's pass flag"; return WAFER_ERR_NCCL; }
    return WAFER_OK;
}

int read_scalars(wafer_ctx* ctx, int slot, int n, double* out) {
    CK(cudaMemcpyAsync(ctx->h_scal + slot, ctx->scal + slot, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->s_main));
    CK(cudaStreamSynchronize(ctx->s_main));
    for (int i = 0; i < n; ++i) out[i] = ctx->h_scal[slot + i];
    return check_p2p_timeout(ctx);
}

// ---- host <-> device layout ------------------------------------------------------------------------------
// planes of the reference's padded array held by this rank (owned + ghosts), clipped to the array
void chunk_range(const wafer_ctx* ctx, bool worksized, long long* hp0, long long* hp1) {
    const Geom& g = ctx->g;
    const long long off = worksized ? 0 : g.e, top = worksized ? g.gnx : g.gnx + 2 * g.e;
    *hp0 = std::max<long long>(0, g.x0 + off - g.gx);
    *hp1 = std::min<long long>(top, g.x0 + g.L + off + g.gx);
}

void owned_range(const wafer_ctx* ctx, long long* hp0, long long* hp1) {
    // planes this rank is responsible for in the caller's global array: owned, plus the outer ring at the ends
    const Geom& g = ctx->g;
    *hp0 = g.x0 + g.e;
    *hp1 = g.x0 + g.L + g.e;
    if (ctx->rank == 0) *hp0 = 0;
    if (ctx->rank == ctx->world - 1) *hp1 = g.gnx + 2 * g.e;
}

// ---- the staging ring --------------------------------------------------------------------------------------------
constexpr long long RING_MAX = 128ll << 20;  // no slot grows past it (a field-sized one was 8.8 GB at 1024^3)

long long host_plane(const Geom& g) { return (long long)(g.ny + 2 * g.e) * (g.nz + 2 * g.e); }  // doubles

// Padded planes per chunk of upload / download, and the slots' first size: the smallest of what fits a slot (once there
// are slots), what fits 128 MB (at least one) and the slab.  So growing the slots changes no chunk here.
long long ring_planes(const wafer_ctx* ctx) {
    const Geom& g = ctx->g;
    const long long plane = host_plane(g) * (long long)sizeof(double);
    const long long fit = ctx->ring.bytes ? (long long)ctx->ring.bytes / plane : LLONG_MAX;
    return std::min({fit, std::max(1ll, RING_MAX / plane), (long long)g.L + 2 * g.gx + 2 * g.e});
}

// the slots and pinned halves; with `all` (wafer_destroy) the events and the copy stream too
void ring_free(StagingRing& r, bool all) {
    for (int b = 0; b < 2; ++b) {
        cudaFree(r.slot[b]);
        if (r.host[b]) cudaFreeHost(r.host[b]);
        r.slot[b] = nullptr;
        r.host[b] = nullptr;
        if (all && r.free[b]) cudaEventDestroy(r.free[b]);
        if (all && r.full[b]) cudaEventDestroy(r.full[b]);
    }
    if (all && r.copy) cudaStreamDestroy(r.copy);
    r.bytes = 0;
}

// Slots of at least min_bytes and of ring_planes, with pinned halves of the slot size when `pinned` asks for them or
// they exist.  Every user of the ring synchronises before it returns, so no queued work
// still uses slots that grow here; the old ones are freed before the new ones are allocated.
int ring_reserve(wafer_ctx* ctx, size_t min_bytes, bool pinned) {
    StagingRing& r = ctx->ring;
    for (cudaEvent_t* e : {&r.free[0], &r.free[1], &r.full[0], &r.full[1]})
        if (!*e) CK(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    if (!r.copy) CK(cudaStreamCreateWithFlags(&r.copy, cudaStreamNonBlocking));
    const size_t want = std::max(min_bytes, (size_t)(ring_planes(ctx) * host_plane(ctx->g)) * sizeof(double));
    if (want > r.bytes) {
        pinned = pinned || r.host[0];
        ring_free(r, false);
        for (int b = 0; b < 2; ++b) CK(cudaMalloc(&r.slot[b], want));
        r.bytes = want;
    }
    for (int b = 0; b < 2; ++b)
        if (pinned && !r.host[b]) CK(cudaMallocHost((void**)&r.host[b], r.bytes));
    return WAFER_OK;
}

// Once before a loop of ring_in / ring_out: everything queued on s_main so far precedes the first refill of a slot.
int ring_start(wafer_ctx* ctx) {
    for (int b = 0; b < 2; ++b) CK(cudaEventRecord(ctx->ring.free[b], ctx->s_main));
    return WAFER_OK;
}

// host -> slot b -> s_main: n bytes of `src` are copied on the copy stream once the slot's last users are done with it
// (nothing when n is 0), then use(slot) queues the kernels that read it; the slot is free again after them.
template <class Use>
int ring_in(wafer_ctx* ctx, int b, const void* src, size_t n, Use use) {
    StagingRing& r = ctx->ring;
    if (n) {
        CK(cudaStreamWaitEvent(r.copy, r.free[b], 0));
        CK(cudaMemcpyAsync(r.slot[b], src, n, cudaMemcpyHostToDevice, r.copy));
        CK(cudaEventRecord(r.full[b], r.copy));
        CK(cudaStreamWaitEvent(ctx->s_main, r.full[b], 0));
    }
    TRY(use(r.slot[b]));
    CK(cudaEventRecord(r.free[b], ctx->s_main));
    return WAFER_OK;
}

// s_main -> slot b -> host: make(slot) queues the kernels that fill the slot once its last copy has left it, then
// n bytes of it go to `dst` on the copy stream; the slot is free again (and `dst` written) after that copy.
template <class Make>
int ring_out(wafer_ctx* ctx, int b, void* dst, size_t n, Make make) {
    StagingRing& r = ctx->ring;
    CK(cudaStreamWaitEvent(ctx->s_main, r.free[b], 0));
    TRY(make(r.slot[b]));
    CK(cudaEventRecord(r.full[b], ctx->s_main));
    CK(cudaStreamWaitEvent(r.copy, r.full[b], 0));
    CK(cudaMemcpyAsync(dst, r.slot[b], n, cudaMemcpyDeviceToHost, r.copy));
    CK(cudaEventRecord(r.free[b], r.copy));
    return WAFER_OK;
}

// the host waits until slot b is free: its ring_out copy has landed, or the kernels of its ring_in are done
int ring_wait(wafer_ctx* ctx, int b) {
    CK(cudaEventSynchronize(ctx->ring.free[b]));
    return WAFER_OK;
}

// the host waits for the copy stream and s_main; sets no ctx->err, as DevBuf drains on the way out of failed calls
cudaError_t ring_drain(wafer_ctx* ctx) {
    const cudaError_t e = cudaStreamSynchronize(ctx->ring.copy), m = cudaStreamSynchronize(ctx->s_main);
    return e != cudaSuccess ? e : m;
}

// host -> device.  `host` points at plane `host_p0` of the reference array; planes [hp0, hp1) of it are read.
// Device planes whose host plane lies outside [hp0, hp1) are zeroed (ghost planes a later halo exchange fills).
int upload(wafer_ctx* ctx, const double* host, long long host_p0, long long hp0, long long hp1, double* dst, bool worksized,
           bool check_ring) {
    const Geom& g = ctx->g;
    const long long py = worksized ? g.ny : g.ny + 2 * g.e, pz = worksized ? g.nz : g.nz + 2 * g.e;
    const int hoff = worksized ? 0 : g.e;
    TRY(ring_reserve(ctx, 0, false));
    const long long planes = ring_planes(ctx);
    if (check_ring) CK(cudaMemsetAsync(ctx->ring_flag, 0, sizeof(int), ctx->s_main));
    TRY(ring_start(ctx));
    int k = 0;
    for (int i0 = -g.gx; i0 < g.L + g.gx; i0 += (int)planes, ++k) {
        const int i1 = (int)std::min<long long>(i0 + planes, g.L + g.gx);
        // host planes behind device planes [i0, i1), clipped to what the caller handed over
        const long long sp0 = std::max<long long>(hp0, g.x0 + i0 + hoff), sp1 = std::min<long long>(hp1, g.x0 + i1 + hoff);
        const size_t n = sp1 > sp0 ? (size_t)((sp1 - sp0) * py * pz) * sizeof(double) : 0;
        TRY(ring_in(ctx, k & 1, host + (sp0 - host_p0) * py * pz, n, [&](void* slot) -> int {
            const int grid = (int)std::min<long long>((long long)(i1 - i0) * g.yp, (long long)ctx->sm_count * 16);
            if (check_ring) unpack_kernel<true><<<grid, 256, 0, ctx->s_main>>>((const double*)slot, dst, g, i0, i1, sp0, std::max(sp0, sp1), worksized ? 1 : 0, ctx->ring_flag);
            else unpack_kernel<false><<<grid, 256, 0, ctx->s_main>>>((const double*)slot, dst, g, i0, i1, sp0, std::max(sp0, sp1), worksized ? 1 : 0, ctx->ring_flag);
            return post_launch(ctx);
        }));
    }
    if (check_ring) {
        int flag = 0;
        CK(cudaMemcpyAsync(&flag, ctx->ring_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->s_main));
        CK(cudaStreamSynchronize(ctx->s_main));
        if (flag) {
            ctx->err = "padding ring of the wavefunction is not zero (config.rs:597-622 guarantees it)";
            return WAFER_ERR_RING_NONZERO;
        }
    } else {
        CK(cudaStreamSynchronize(ctx->s_main));  // the caller may free its buffer on return
    }
    return WAFER_OK;
}

// device -> host: padded planes [hp0, hp1) of the global array into `host`, which points at plane host_p0
int download(wafer_ctx* ctx, const double* src, double* host, long long host_p0, long long hp0, long long hp1) {
    const Geom& g = ctx->g;
    const long long py = g.ny + 2 * g.e, pz = g.nz + 2 * g.e;
    TRY(ring_reserve(ctx, 0, false));
    const long long planes = ring_planes(ctx);
    TRY(ring_start(ctx));
    int k = 0;
    for (long long sp0 = hp0; sp0 < hp1; sp0 += planes, ++k) {
        const long long sp1 = std::min(hp1, sp0 + planes);
        TRY(ring_out(ctx, k & 1, host + (sp0 - host_p0) * py * pz, (size_t)((sp1 - sp0) * py * pz) * sizeof(double), [&](void* slot) -> int {
            const int grid = (int)std::min<long long>((sp1 - sp0) * py, (long long)ctx->sm_count * 16);
            pack_kernel<<<grid, 256, 0, ctx->s_main>>>(src, (double*)slot, g, sp0, sp1, 0);
            return post_launch(ctx);
        }));
    }
    CK(ring_drain(ctx));
    return WAFER_OK;
}

// global-array entry points: this rank's chunk (owned + ghost planes) in, its owned planes out
int upload_global(wafer_ctx* ctx, const double* host, double* dst, bool worksized, bool check_ring) {
    long long hp0, hp1;
    chunk_range(ctx, worksized, &hp0, &hp1);
    return upload(ctx, host, 0, hp0, hp1, dst, worksized, check_ring);
}
int download_global(wafer_ctx* ctx, const double* src, double* host) {
    long long hp0, hp1;
    owned_range(ctx, &hp0, &hp1);
    return download(ctx, src, host, 0, hp0, hp1);
}

int alloc_field(wafer_ctx* ctx, double** p) {
    CK(cudaMalloc(p, ctx->bytes()));
    CK(cudaMemsetAsync(*p, 0, ctx->bytes(), ctx->s_main));
    return WAFER_OK;
}

int ensure_ab(wafer_ctx* ctx) {
    if (ctx->onfly) return WAFER_OK;
    if (!ctx->a) TRY(alloc_field(ctx, &ctx->a));
    if (!ctx->b) TRY(alloc_field(ctx, &ctx->b));
    const long long n = ctx->g.total();
    build_ab_kernel<<<ew_grid(ctx, n), EW_THREADS, 0, ctx->s_main>>>(ctx->v, ctx->a, ctx->b, n, ctx->p.dt);
    return post_launch(ctx);
}

// fill_data / read_csv on the device (resample.cuh) into the work area of `dst`: only the source x-planes this rank's
// planes need are copied, run by run, through the staging ring (grown, to at most 128 MB a slot, when two source planes
// do not fit the padded planes a slot carries); the copy of one run overlaps the kernel of the other.  Synchronises.
constexpr long long RS_MAX_STG = RING_MAX / (long long)sizeof(double);  // doubles in one 128 MB slot

bool resample_copies(const wafer_ctx* ctx, uint64_t sx, uint64_t sy, uint64_t sz, uint32_t from_csv) {
    return from_csv && sx == (uint64_t)ctx->g.gnx && sy == (uint64_t)ctx->g.gny && sz == (uint64_t)ctx->g.gnz;
}

// What this rank's planes read of an (sx, sy, sz) source: the global work planes [ga, gb) of the slab inside the
// lattice (ghosts included) and the source x-planes [sp0, sp1) they need.
struct RsPlan {
    bool copy;  // a work-sized Csv source, copied straight in
    long long ga, gb, sp0, sp1;
};

// lowest source plane behind global work plane gi (the planes [lo, lo + 1 + !copy) are read)
long long rs_lo(const wafer_ctx* ctx, const RsPlan& pl, uint64_t sx, long long gi) {
    if (pl.copy) return gi;
    long long i0;
    double d;
    rs_bracket((long long)sx, ctx->g.gnx + 2 * ctx->g.e, gi, &i0, &d);
    return i0;
}

// The shape rules of fill_data / read_csv for both the host-staged entries and wafer_load_array
int resample_shape(wafer_ctx* ctx, uint64_t sx, uint64_t sy, uint64_t sz, uint32_t from_csv, RsPlan* pl) {
    const Geom& g = ctx->g;
    const uint64_t e2 = 2 * (uint64_t)g.e;
    REQUIRE(sx > 0 && sy > 0 && sz > 0, "ArrayShape: the input array has a zero dimension");
    REQUIRE(from_csv || !(sx == g.gnx + e2 && sy == g.gny + e2 && sz == g.gnz + e2),
            "input array already has the padded size: the reference's fill_data cannot load it (input.rs:167-169)");
    pl->copy = resample_copies(ctx, sx, sy, sz, from_csv);
    REQUIRE(pl->copy || (sx >= 2 && sy >= 2 && sz >= 2), "ArrayShape: the input array cannot be resized (needs >= 2 points per axis)");
    pl->ga = std::max<long long>(0, g.x0 - g.gx);
    pl->gb = std::min<long long>(g.gnx, g.x0 + g.L + g.gx);
    pl->sp0 = rs_lo(ctx, *pl, sx, pl->ga);
    pl->sp1 = rs_lo(ctx, *pl, sx, pl->gb - 1) + (pl->copy ? 1 : 2);
    return WAFER_OK;
}

int resample_args(wafer_ctx* ctx, const double* src, uint64_t sx, uint64_t sy, uint64_t sz, uint32_t from_csv, RsPlan* pl) {
    REQUIRE(src, "src is NULL");
    REQUIRE(from_csv <= 1, "from_csv must be 0 (Messagepack / Json) or 1 (Csv)");
    TRY(resample_shape(ctx, sx, sy, sz, from_csv, pl));
    REQUIRE(sy <= (uint64_t)RS_MAX_STG / 2 && sz <= (uint64_t)RS_MAX_STG / 2 / sy,
            "input array: two of its x-planes (2*sy*sz*8 bytes) exceed the 128 MB staging buffer");
    return WAFER_OK;
}

void rs_launch(wafer_ctx* ctx, const RsPlan& pl, double* dst, const double* src, long long s0, uint64_t sx, uint64_t sy,
               uint64_t sz, long long a, long long b) {
    const Geom& g = ctx->g;
    const int ztiles = std::min(ceil_div(g.nz, RS_ZTILE), 65535);
    const int i0 = (int)(a - g.x0), i1 = (int)(b - g.x0);
    const dim3 grid((unsigned)std::min<long long>((long long)(i1 - i0) * g.ny, std::max(1, ctx->sm_count * 8 / ztiles)),
                    (unsigned)ztiles);
    if (pl.copy) resample_kernel<true><<<grid, RS_THREADS, 0, ctx->s_main>>>(dst, g, src, s0, (long long)sx, (long long)sy, (long long)sz, i0, i1);
    else resample_kernel<false><<<grid, RS_THREADS, 0, ctx->s_main>>>(dst, g, src, s0, (long long)sx, (long long)sy, (long long)sz, i0, i1);
}

// the arguments passed resample_args
int resample_into(wafer_ctx* ctx, const RsPlan& pl, const double* src, uint64_t sx, uint64_t sy, uint64_t sz, double* dst) {
    const long long splane = (long long)(sy * sz), need = pl.copy ? 1 : 2;
    auto lo = [&](long long gi) { return rs_lo(ctx, pl, sx, gi); };
    const long long ga = pl.ga, gb = pl.gb;
    long long cap = ring_planes(ctx) * host_plane(ctx->g) / splane;  // source planes per run
    if (cap < need) cap = std::min<long long>(RS_MAX_STG / splane, pl.sp1 - pl.sp0);
    TRY(ring_reserve(ctx, (size_t)(cap * splane) * sizeof(double), false));
    TRY(ring_start(ctx));
    int k = 0;
    for (long long a = ga; a < gb; ++k) {
        const long long s0 = lo(a);
        long long b = a + 1;
        while (b < gb && lo(b) + need - s0 <= cap) ++b;  // lo() is non-decreasing: the run's planes are [s0, lo(b-1)+need)
        const long long s1 = lo(b - 1) + need;
        TRY(ring_in(ctx, k & 1, src + s0 * splane, (size_t)((s1 - s0) * splane) * sizeof(double), [&](void* slot) -> int {
            rs_launch(ctx, pl, dst, (const double*)slot, s0, sx, sy, sz, a, b);
            return post_launch(ctx);
        }));
        a = b;
    }
    CK(cudaStreamSynchronize(ctx->s_main));  // the caller may free `src` on return
    return WAFER_OK;
}

enum { RS_PHI = 0, RS_POTENTIAL, RS_LOWER };

// what setting psi (which = RS_PHI), V (RS_POTENTIAL) or a new lower state (RS_LOWER) changes, for every entry that
// sets one; fill(dst) writes the work area of the field (an upload, a generator, a resample)
template <class Fill>
int set_input(wafer_ctx* ctx, int which, Fill fill) {
    if (which == RS_PHI) {  // the ring is +0 by construction
        ctx->chk_valid = false;  // psi (or what the check sums depend on) changes
        const int rc = fill(ctx->psi[ctx->cur]);
        ctx->have_phi = rc == WAFER_OK;
        return rc;
    }
    if (which == RS_POTENTIAL) {
        ctx->chk_valid = false;
        ctx->h_valid = false;
        TRY(fill(ctx->v));
        TRY(ensure_ab(ctx));
        ctx->have_v = true;
        return WAFER_OK;
    }
    REQUIRE(ctx->lowers.size() < 255, "at most 255 lower states (wavenum is a u8, config.rs:308)");
    double* q = nullptr;
    TRY(alloc_field(ctx, &q));
    int rc = fill(q);
    if (rc == WAFER_OK) rc = register_lower(ctx, q);
    if (rc != WAFER_OK) cudaFree(q);
    return rc;
}

int create_impl(const wafer_params* params, wafer_ctx* ctx) {
    const wafer_params& p = *params;
    REQUIRE(p.nx > 0 && p.ny > 0 && p.nz > 0, "grid.size must be positive");
    REQUIRE(p.ext >= 1 && p.ext <= 3, "ext must be 1 (ThreePoint), 2 (FivePoint) or 3 (SevenPoint)");
    REQUIRE(p.nx < (1u << 30) && p.ny < (1u << 30) && p.nz < (1u << 30), "grid.size too large");
    REQUIRE(std::isfinite(p.dn) && std::isfinite(p.dt) && std::isfinite(p.mass) && p.dn > 0 && p.mass != 0,
            "dn, dt, mass must be finite (dn > 0, mass != 0)");
    ctx->p = p;
    ctx->p.nccl_id = nullptr;
    ctx->world = p.world == 0 ? 1 : (int)p.world;
    ctx->rank = (int)p.rank;
    REQUIRE(ctx->rank < ctx->world, "rank must be < world");
    ctx->onfly = !(p.flags & WAFER_FLAG_AB_ARRAYS);

    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        ctx->err = "no CUDA device visible: this library has no CPU fallback";
        return WAFER_ERR_NO_DEVICE;
    }
    int dev = p.device;
    if (dev < 0) {
        const char* lr = getenv("LOCAL_RANK");
        dev = lr ? atoi(lr) % ndev : 0;
    }
    if (dev >= ndev) { ctx->err = "device ordinal out of range"; return WAFER_ERR_NO_DEVICE; }
    ctx->dev = dev;
    CK(cudaSetDevice(dev));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, dev));
    if (prop.major != 10) {
        ctx->err = std::string("device '") + prop.name + "' is not sm_100 (Blackwell B200); this build targets sm_100a only";
        return WAFER_ERR_NO_DEVICE;
    }
    ctx->sm_count = prop.multiProcessorCount;

    // slab decomposition along x
    Geom& g = ctx->g;
    uint64_t sx0, sx1;
    wafer_slab_partition(p.nx, (uint32_t)ctx->world, (uint32_t)ctx->rank, &sx0, &sx1);
    g.L = (int)(sx1 - sx0);
    g.x0 = (long long)sx0;
    g.ny = (int)p.ny; g.nz = (int)p.nz; g.e = (int)p.ext;
    g.gx = g.e == 1 ? 2 : g.e;  // the time-tiled ThreePoint sweep advances two steps per halo exchange
    g.yp = g.ny + 2 * g.e;
    g.zp = (int)(((long long)g.nz + 2 * g.e + 15) / 16 * 16);
    g.plane = (long long)g.yp * g.zp;
    g.gnx = p.nx; g.gny = p.ny; g.gnz = p.nz;
    ctx->min_L = (int)(p.nx / (uint64_t)ctx->world);  // wafer_slab_partition: the last ranks own floor(nx/world) planes
    REQUIRE(ctx->world == 1 || ctx->min_L >= g.gx, "every rank needs at least as many planes as the ghost depth (2 for ThreePoint, else ext)");

    int lo, hi;
    CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    CK(cudaStreamCreateWithPriority(&ctx->s_main, cudaStreamNonBlocking, lo));
    CK(cudaStreamCreateWithPriority(&ctx->s_halo, cudaStreamNonBlocking, hi));
    CK(cudaEventCreate(&ctx->ev_t0));
    CK(cudaEventCreate(&ctx->ev_t1));
    CK(cudaEventCreateWithFlags(&ctx->ev_main, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ctx->ev_halo, cudaEventDisableTiming));

    TRY(alloc_field(ctx, &ctx->psi[0]));
    TRY(alloc_field(ctx, &ctx->psi[1]));
    TRY(alloc_field(ctx, &ctx->v));
    const long long nb = std::max<long long>(
        {(long long)simple_blocks(ctx, 0, g.L) + 4 * simple_blocks(ctx, 0, g.e),
         (long long)ceil_div(g.nz, 56) * ceil_div(g.ny, 32) * std::min(g.L, 64),  // TMA one-step kernel: tiles x chunks
         (long long)ceil_div(g.nz, SW_BX) * ceil_div(g.ny, SW_BY) * ceil_div(g.L, SW_XCH), (long long)ctx->sm_count * 8});
    ctx->partials_cap = nb * 8;  // up to 1 + 4 fused running sums per CTA (sweep_tma1.cuh NRED), 4 for the observables
    CK(cudaMalloc(&ctx->partials, ctx->partials_cap * sizeof(double)));
    CK(cudaMalloc(&ctx->scal, SL_COUNT * sizeof(double)));
    CK(cudaMemsetAsync(ctx->scal, 0, SL_COUNT * sizeof(double), ctx->s_main));
    CK(cudaMallocHost(&ctx->h_scal, SL_COUNT * sizeof(double)));
    CK(cudaMalloc(&ctx->ring_flag, sizeof(int)));
    ctx->den_ok = den_in_fast_window(denominator(ctx));
    TRY(init_tb(ctx));
    TRY(init_t1(ctx));

    if (ctx->world > 1) {
        if (!p.nccl_id) { ctx->err = "world > 1 needs the 128-byte nccl_id of rank 0"; return WAFER_ERR_INVALID; }
        if (const char* why = nccl_api().load()) { ctx->err = why; return WAFER_ERR_NCCL; }
        NcclUniqueId id;
        memcpy(id.internal, p.nccl_id, sizeof(id.internal));
        NK(nccl_api().CommInitRank(&ctx->comm, ctx->world, id, ctx->rank));
    }
    CK(cudaStreamSynchronize(ctx->s_main));
    return WAFER_OK;
}

}  // namespace

// =============================================================================================================
extern "C" {

const char* wafer_version(void) { return "wafer_b200 0.1 (sm_100a)"; }

int wafer_create(const wafer_params* params, wafer_ctx** out) {
    if (!params || !out) { g_create_error = "NULL argument"; return WAFER_ERR_INVALID; }
    *out = nullptr;
    wafer_ctx* ctx = new (std::nothrow) wafer_ctx();
    if (!ctx) { g_create_error = "out of host memory"; return WAFER_ERR_INVALID; }
    int rc;
    try {
        rc = create_impl(params, ctx);
    } catch (const std::exception& e) {
        ctx->err = std::string("wafer_create: ") + e.what();
        rc = WAFER_ERR_INVALID;
    }
    if (rc != WAFER_OK) {
        g_create_error = ctx->err;
        wafer_destroy(ctx);
        return rc;
    }
    *out = ctx;
    return WAFER_OK;
}

int wafer_destroy(wafer_ctx* ctx) {
    if (!ctx) return WAFER_OK;
    if (ctx->s_main) cudaStreamSynchronize(ctx->s_main);
    if (ctx->s_halo) cudaStreamSynchronize(ctx->s_halo);
    drop_step_graphs(ctx);
    if (ctx->comm) nccl_api().CommDestroy(ctx->comm);
    for (int n = 0; n < 2; ++n) {
        if (ctx->peer_psi[n][0]) cudaIpcCloseMemHandle(ctx->peer_psi[n][0]);
        if (ctx->peer_psi[n][1]) cudaIpcCloseMemHandle(ctx->peer_psi[n][1]);
        if (ctx->peer_flags[n]) cudaIpcCloseMemHandle(ctx->peer_flags[n]);
    }
    cudaFree(ctx->flags); cudaFree(ctx->p2p_timeout);
    for (double* q : ctx->lowers) cudaFree(q);
    cudaFree(ctx->hfield);
    cudaFree(ctx->psi[0]); cudaFree(ctx->psi[1]); cudaFree(ctx->v); cudaFree(ctx->a); cudaFree(ctx->b);
    ring_free(ctx->ring, true);
    cudaFree(ctx->pow10);
    cudaFree(ctx->wr_btot); cudaFree(ctx->wr_boff); cudaFree(ctx->wr_flags); cudaFree(ctx->wr_txt); cudaFree(ctx->wr_count);
    cudaFree(ctx->wr_red);
    for (int b = 0; b < 2; ++b) {
        cudaFree(ctx->rd_bcount[b]); cudaFree(ctx->rd_boff[b]); cudaFree(ctx->rd_flags[b]);
    }
    cudaFree(ctx->rd_st);
    if (ctx->rd_hst) cudaFreeHost(ctx->rd_hst);
    cudaFree(ctx->d_cksum); cudaFree(ctx->gram);
    for (auto& kv : ctx->tb2_sched) {
        cudaFree(kv.second.bulk); cudaFree(kv.second.segs); cudaFree(kv.second.first); cudaFree(kv.second.counters);
    }
    cudaFree(ctx->potsub_arr); cudaFree(ctx->partials); cudaFree(ctx->scal); cudaFree(ctx->ring_flag);
    if (ctx->h_scal) cudaFreeHost(ctx->h_scal);
    if (ctx->ev_t0) cudaEventDestroy(ctx->ev_t0);
    if (ctx->ev_t1) cudaEventDestroy(ctx->ev_t1);
    if (ctx->ev_main) cudaEventDestroy(ctx->ev_main);
    if (ctx->ev_halo) cudaEventDestroy(ctx->ev_halo);
    if (ctx->s_main) cudaStreamDestroy(ctx->s_main);
    if (ctx->s_halo) cudaStreamDestroy(ctx->s_halo);
    delete ctx;
    return WAFER_OK;
}

const char* wafer_last_error(const wafer_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int wafer_nccl_unique_id(uint8_t out[128]) {
    if (!out) return WAFER_ERR_INVALID;
    if (const char* why = nccl_api().load()) { g_create_error = why; return WAFER_ERR_NCCL; }
    NcclUniqueId id;
    if (nccl_api().GetUniqueId(&id) != kNcclSuccess) { g_create_error = "ncclGetUniqueId failed"; return WAFER_ERR_NCCL; }
    memcpy(out, id.internal, 128);
    return WAFER_OK;
}

int wafer_slab_partition(uint64_t nx, uint32_t world, uint32_t rank, uint64_t* x0, uint64_t* x1) {
    if (world == 0) world = 1;
    if (rank >= world || !x0 || !x1) return WAFER_ERR_INVALID;
    const uint64_t base = nx / world, rem = nx % world;
    *x0 = rank * base + std::min<uint64_t>(rank, rem);
    *x1 = *x0 + base + (rank < rem ? 1 : 0);
    return WAFER_OK;
}

int wafer_tb2_plan(uint32_t ny, uint32_t nz, int32_t xb, int32_t xe, uint32_t slots, int32_t* segments, uint64_t cap, uint64_t* n) {
    if (!n || ny == 0 || nz == 0 || xe <= xb || slots == 0) return WAFER_ERR_INVALID;
    try {
        const Tb2Plan pl = tb2_plan((int)ny, (int)nz, xb, xe, (int)slots);
        uint64_t k = 0;
        auto put = [&](int owner, const tb::Segment& sg) {
            if (segments && k < cap) {
                int32_t* o = segments + 5 * k;
                o[0] = owner; o[1] = sg.y0; o[2] = sg.z0; o[3] = sg.xa; o[4] = sg.xz;
            }
            ++k;
        };
        for (const auto& sg : pl.bulk) put(-1, sg);
        for (size_t c = 0; c < pl.per.size(); ++c)
            for (const auto& sg : pl.per[c]) put((int)c, sg);
        *n = k;
        return WAFER_OK;
    } catch (const std::exception&) {
        return WAFER_ERR_INVALID;
    }
}

int wafer_slab(const wafer_ctx* ctx, uint64_t* x0, uint64_t* x1) {
    if (!ctx) return WAFER_ERR_INVALID;
    if (x0) *x0 = (uint64_t)ctx->g.x0;
    if (x1) *x1 = (uint64_t)(ctx->g.x0 + ctx->g.L);
    return WAFER_OK;
}

// ---- state in / out ------------------------------------------------------------------------------------------
int wafer_set_potential(wafer_ctx* ctx, const double* v_padded) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(v_padded, "v_padded is NULL");
    CK(cudaSetDevice(ctx->dev));
    return set_input(ctx, RS_POTENTIAL, [&](double* dst) { return upload_global(ctx, v_padded, dst, false, false); });
}

int wafer_get_potential(wafer_ctx* ctx, double* v_padded) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(v_padded, "v_padded is NULL");
    if (!ctx->have_v) { ctx->err = "potential not set"; return WAFER_ERR_NOT_READY; }
    CK(cudaSetDevice(ctx->dev));
    return download_global(ctx, ctx->v, v_padded);
}

int wafer_set_pot_sub_scalar(wafer_ctx* ctx, double c) {
    if (!ctx) return WAFER_ERR_INVALID;
    ctx->chk_valid = false;  // psi (or what the check sums depend on) changes
    // potential.rs:148-152: (None, Some(c)) only when c > 0, else (None, None)
    ctx->potsub_mode = c > 0.0 ? 1 : 0;
    ctx->potsub_scalar = c > 0.0 ? c : 0.0;
    return WAFER_OK;
}

int wafer_set_pot_sub_array(wafer_ctx* ctx, const double* work) {
    if (!ctx) return WAFER_ERR_INVALID;
    ctx->chk_valid = false;  // psi (or what the check sums depend on) changes
    REQUIRE(work, "pot_sub array is NULL");
    CK(cudaSetDevice(ctx->dev));
    if (!ctx->potsub_arr) TRY(alloc_field(ctx, &ctx->potsub_arr));
    TRY(upload_global(ctx, work, ctx->potsub_arr, true, false));
    ctx->potsub_mode = 2;
    return WAFER_OK;
}

int wafer_set_phi(wafer_ctx* ctx, const double* phi_padded) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(phi_padded, "phi_padded is NULL");
    CK(cudaSetDevice(ctx->dev));
    return set_input(ctx, RS_PHI, [&](double* dst) { return upload_global(ctx, phi_padded, dst, false, true); });
}

int wafer_get_phi(wafer_ctx* ctx, double* phi_padded) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(phi_padded, "phi_padded is NULL");
    if (!ctx->have_phi) { ctx->err = "phi not set"; return WAFER_ERR_NOT_READY; }
    CK(cudaSetDevice(ctx->dev));
    return download_global(ctx, ctx->psi[ctx->cur], phi_padded);
}

int wafer_slab_planes(const wafer_ctx* ctx, int32_t which, uint64_t* p0, uint64_t* p1) {
    if (!ctx) return WAFER_ERR_INVALID;
    long long a, b;
    if (which == 0) chunk_range(ctx, false, &a, &b);
    else owned_range(ctx, &a, &b);
    if (p0) *p0 = (uint64_t)a;
    if (p1) *p1 = (uint64_t)b;
    return WAFER_OK;
}

int wafer_set_phi_slab(wafer_ctx* ctx, const double* chunk) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(chunk, "chunk is NULL");
    CK(cudaSetDevice(ctx->dev));
    long long hp0, hp1;
    chunk_range(ctx, false, &hp0, &hp1);
    return set_input(ctx, RS_PHI, [&](double* dst) { return upload(ctx, chunk, hp0, hp0, hp1, dst, false, true); });
}

int wafer_set_phi_owned(wafer_ctx* ctx, const double* chunk) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(chunk, "chunk is NULL");
    CK(cudaSetDevice(ctx->dev));
    long long hp0, hp1;
    owned_range(ctx, &hp0, &hp1);
    TRY(set_input(ctx, RS_PHI, [&](double* dst) { return upload(ctx, chunk, hp0, hp0, hp1, dst, false, true); }));
    return exchange(ctx, ctx->psi[ctx->cur], ctx->s_main);  // ghost planes come from the neighbours (collective)
}

int wafer_get_phi_slab(wafer_ctx* ctx, double* chunk) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(chunk, "chunk is NULL");
    if (!ctx->have_phi) { ctx->err = "phi not set"; return WAFER_ERR_NOT_READY; }
    CK(cudaSetDevice(ctx->dev));
    long long hp0, hp1;
    owned_range(ctx, &hp0, &hp1);
    return download(ctx, ctx->psi[ctx->cur], chunk, hp0, hp0, hp1);
}

static int wafer_push_lower_impl(wafer_ctx* ctx, const double* q_padded) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(q_padded, "q_padded is NULL");
    CK(cudaSetDevice(ctx->dev));
    return set_input(ctx, RS_LOWER, [&](double* dst) { return upload_global(ctx, q_padded, dst, false, true); });
}

static int wafer_push_lower_from_phi_impl(wafer_ctx* ctx) {
    if (!ctx) return WAFER_ERR_INVALID;
    if (!ctx->have_phi) { ctx->err = "phi not set"; return WAFER_ERR_NOT_READY; }
    REQUIRE(ctx->lowers.size() < 255, "at most 255 lower states (wavenum is a u8, config.rs:308)");
    CK(cudaSetDevice(ctx->dev));
    double* q = nullptr;
    CK(cudaMalloc(&q, ctx->bytes()));
    CK(cudaMemcpyAsync(q, ctx->psi[ctx->cur], ctx->bytes(), cudaMemcpyDeviceToDevice, ctx->s_main));
    const int rc = register_lower(ctx, q);
    if (rc != WAFER_OK) cudaFree(q);
    return rc;
}

int wafer_get_lower(wafer_ctx* ctx, uint32_t idx, double* q_padded) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(q_padded && idx < ctx->lowers.size(), "no such lower state");
    CK(cudaSetDevice(ctx->dev));
    return download_global(ctx, ctx->lowers[idx], q_padded);
}

int wafer_phi_from_lower(wafer_ctx* ctx, uint32_t idx) {
    if (!ctx) return WAFER_ERR_INVALID;
    ctx->chk_valid = false;  // psi (or what the check sums depend on) changes
    REQUIRE(idx < ctx->lowers.size(), "no such lower state");
    CK(cudaSetDevice(ctx->dev));
    CK(cudaMemcpyAsync(ctx->psi[ctx->cur], ctx->lowers[idx], ctx->bytes(), cudaMemcpyDeviceToDevice, ctx->s_main));
    ctx->have_phi = true;
    return WAFER_OK;
}

int wafer_phi_seed_from_lower(wafer_ctx* ctx, uint32_t idx) {
    if (!ctx) return WAFER_ERR_INVALID;
    ctx->chk_valid = false;  // psi (or what the check sums depend on) changes
    REQUIRE(idx < ctx->lowers.size(), "no such lower state");
    CK(cudaSetDevice(ctx->dev));
    const long long rows = (long long)(ctx->g.L + 2 * ctx->g.gx) * ctx->g.ny;
    seed_from_state_kernel<<<(int)std::min<long long>(rows, (long long)ctx->sm_count * 32), 128, 0, ctx->s_main>>>(
        ctx->psi[ctx->cur], ctx->lowers[idx], ctx->g);
    TRY(post_launch(ctx));
    ctx->have_phi = true;
    return WAFER_OK;
}

int wafer_clear_lowers(wafer_ctx* ctx) {
    if (!ctx) return WAFER_ERR_INVALID;
    CK(cudaSetDevice(ctx->dev));
    CK(cudaStreamSynchronize(ctx->s_main));
    for (double* q : ctx->lowers) cudaFree(q);
    ctx->lowers.clear();
    drop_step_graphs(ctx);  // they hold the freed pointers
    return WAFER_OK;
}

uint32_t wafer_num_lowers(const wafer_ctx* ctx) { return ctx ? (uint32_t)ctx->lowers.size() : 0; }

int wafer_generate_potential(wafer_ctx* ctx, int32_t kind, double sig) {
    if (!ctx) return WAFER_ERR_INVALID;
    CK(cudaSetDevice(ctx->dev));
    GenParams gp = make_gen_params(ctx->p.dn, ctx->p.mass, sig);
    REQUIRE(potential_kind_supported(kind), "PotentialNotAvailable: no formula for this potential kind (potential.rs:315-317)");
    const long long rows = (long long)(ctx->g.L + 2 * ctx->g.gx) * ctx->g.ny;
    return set_input(ctx, RS_POTENTIAL, [&](double* dst) {
        gen_potential_kernel<<<(int)std::min<long long>(rows, (long long)ctx->sm_count * 32), 128, 0, ctx->s_main>>>(dst, ctx->g, kind, gp);
        return post_launch(ctx);
    });
}

int wafer_generate_initial_condition(wafer_ctx* ctx, int32_t kind) {
    if (!ctx) return WAFER_ERR_INVALID;
    ctx->chk_valid = false;  // psi (or what the check sums depend on) changes
    REQUIRE(kind >= 2 && kind <= 4, "only Coulomb (2), Constant (3) and Boolean (4) can be generated on the device");
    CK(cudaSetDevice(ctx->dev));
    GenParams gp = make_gen_params(ctx->p.dn, ctx->p.mass, 0.0);
    const long long rows = (long long)(ctx->g.L + 2 * ctx->g.gx) * ctx->g.ny;
    gen_ic_kernel<<<(int)std::min<long long>(rows, (long long)ctx->sm_count * 32), 128, 0, ctx->s_main>>>(ctx->psi[ctx->cur], ctx->g, kind, gp);
    TRY(post_launch(ctx));
    ctx->have_phi = true;
    return WAFER_OK;
}

int wafer_generate_gaussian(wafer_ctx* ctx, double sig, uint64_t seed) {
    if (!ctx) return WAFER_ERR_INVALID;
    ctx->chk_valid = false;  // psi (or what the check sums depend on) changes
    REQUIRE(std::isfinite(sig) && sig >= 0., "Gaussian initial condition: sig must be finite and >= 0");
    CK(cudaSetDevice(ctx->dev));
    const long long rows = (long long)(ctx->g.L + 2 * ctx->g.gx) * ctx->g.ny;
    gen_gaussian_kernel<<<(int)std::min<long long>(rows, (long long)ctx->sm_count * 32), 128, 0, ctx->s_main>>>(
        ctx->psi[ctx->cur], ctx->g, sig, (unsigned long long)seed);
    TRY(post_launch(ctx));
    ctx->have_phi = true;
    return WAFER_OK;
}

int wafer_symmetrise(wafer_ctx* ctx, int32_t kind) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(kind >= SYM_NONE && kind <= SYM_ANTI_Y,
            "init_symmetry: kind must be 0 NotConstrained, 1 AboutZ, 2 AntisymAboutZ, 3 AboutY or 4 AntisymAboutY");
    if (!ctx->have_phi) { ctx->err = "phi not set (wafer_set_phi / wafer_generate_initial_condition)"; return WAFER_ERR_NOT_READY; }
    if (kind == SYM_NONE) return WAFER_OK;
    ctx->chk_valid = false;  // psi (or what the check sums depend on) changes
    CK(cudaSetDevice(ctx->dev));
    const Geom& g = ctx->g;
    const double s = (kind == SYM_ANTI_Z || kind == SYM_ANTI_Y) ? -1. : 1.;
    const long long planes = (long long)(g.L + 2 * g.gx);
    if (kind == SYM_ABOUT_Z || kind == SYM_ANTI_Z) {
        symmetrise_z_kernel<<<(int)std::min<long long>(planes * g.ny, (long long)ctx->sm_count * 32), 128, 0, ctx->s_main>>>(
            ctx->psi[ctx->cur], g, s);
    } else {
        symmetrise_y_kernel<<<(int)std::min<long long>(planes * (g.ny - g.ny / 2), (long long)ctx->sm_count * 32), 128, 0,
                              ctx->s_main>>>(ctx->psi[ctx->cur], g, s);
    }
    return post_launch(ctx);
}

// ---- input files resampled on the device (resample.cuh) -------------------------------------------------------
static int resampled_impl(wafer_ctx* ctx, int which, const double* src, uint64_t sx, uint64_t sy, uint64_t sz,
                          uint32_t from_csv) {
    if (!ctx) return WAFER_ERR_INVALID;
    RsPlan pl;
    TRY(resample_args(ctx, src, sx, sy, sz, from_csv, &pl));  // before anything is allocated or written
    CK(cudaSetDevice(ctx->dev));
    return set_input(ctx, which, [&](double* dst) { return resample_into(ctx, pl, src, sx, sy, sz, dst); });
}

static int resampled(wafer_ctx* ctx, int which, const char* name, const double* src, uint64_t sx, uint64_t sy,
                     uint64_t sz, uint32_t from_csv) {
    try {
        return resampled_impl(ctx, which, src, sx, sy, sz, from_csv);
    } catch (const std::exception& e) {  // host-side allocation failures must not unwind through the C ABI
        if (ctx) ctx->err = std::string(name) + ": " + e.what();
        return WAFER_ERR_INVALID;
    }
}

int wafer_set_phi_resampled(wafer_ctx* ctx, const double* src, uint64_t sx, uint64_t sy, uint64_t sz, uint32_t from_csv) {
    return resampled(ctx, RS_PHI, "wafer_set_phi_resampled", src, sx, sy, sz, from_csv);
}

int wafer_set_potential_resampled(wafer_ctx* ctx, const double* src, uint64_t sx, uint64_t sy, uint64_t sz,
                                  uint32_t from_csv) {
    return resampled(ctx, RS_POTENTIAL, "wafer_set_potential_resampled", src, sx, sy, sz, from_csv);
}

int wafer_push_lower_resampled(wafer_ctx* ctx, const double* src, uint64_t sx, uint64_t sy, uint64_t sz, uint32_t from_csv) {
    return resampled(ctx, RS_LOWER, "wafer_push_lower_resampled", src, sx, sy, sz, from_csv);
}

// ---- the hot path --------------------------------------------------------------------------------------------
static int ready(wafer_ctx* ctx, bool need_v) {
    if (!ctx->have_phi) { ctx->err = "phi not set (wafer_set_phi / wafer_generate_initial_condition)"; return WAFER_ERR_NOT_READY; }
    if (need_v && !ctx->have_v) { ctx->err = "potential not set (wafer_set_potential / wafer_generate_potential)"; return WAFER_ERR_NOT_READY; }
    return WAFER_OK;
}

// ---- array files encoded on the device (encode.cuh) -------------------------------------------------------------
// Two passes over this rank's work sites.  Pass 1 measures: block totals of the certified sites, the refused sites
// formatted on the host (their lengths added), an exclusive scan into block offsets.  The ranks then exchange their
// byte counts in one all-reduce, so each knows where its planes start in the file.  Pass 2 encodes chunk after
// chunk into a slot of the staging ring (as many whole blocks as fit), copies it to the slot's pinned half and writes
// it with pwrite while the next chunk is encoded.  Refused sites are collected again per piece of a chunk (a run of
// blocks with at most ENC_FLAG_CAP of them) rather than kept from pass 1: host memory stays bounded whatever the field.
// the ring's slots for the array files, written or read: at least two blocks of the longest Csv rows
static constexpr size_t FILE_MIN_STG = 2 * (size_t)ENC_BS * enc::SITE_MAX;

// the 128-bit power table of encode.cuh / decode.cuh
static int pow10_table(wafer_ctx* ctx) {
    if (ctx->pow10) return WAFER_OK;
    EncTable h;
    const enc::Pow10 t = enc::host_pow10();
    memcpy(h.hilo, t.hilo, sizeof h.hilo);
    memcpy(h.shift, t.shift, sizeof h.shift);
    EncTable* p = nullptr;
    CK(cudaMalloc(&p, sizeof(EncTable)));
    CK(cudaMemcpy(p, &h, sizeof(EncTable), cudaMemcpyHostToDevice));
    ctx->pow10 = p;
    return WAFER_OK;
}

static int wr_buffers(wafer_ctx* ctx, long long nblocks) {
    TRY(ring_reserve(ctx, FILE_MIN_STG, true));
    TRY(pow10_table(ctx));
    if (ctx->wr_blocks < nblocks) {
        cudaFree(ctx->wr_btot);
        cudaFree(ctx->wr_boff);
        ctx->wr_btot = nullptr;
        ctx->wr_boff = nullptr;
        ctx->wr_blocks = 0;
        CK(cudaMalloc(&ctx->wr_btot, (size_t)nblocks * sizeof(unsigned int)));
        CK(cudaMalloc(&ctx->wr_boff, (size_t)(nblocks + 1) * sizeof(unsigned long long)));
        ctx->wr_blocks = nblocks;
    }
    if (!ctx->wr_count) {
        CK(cudaMalloc(&ctx->wr_flags, ENC_FLAG_CAP * sizeof(EncFlagIn)));
        CK(cudaMalloc(&ctx->wr_txt, ENC_FLAG_CAP * sizeof(EncFlagStr)));
        CK(cudaMalloc(&ctx->wr_count, 2 * sizeof(unsigned long long)));
    }
    if (ctx->world > 1 && !ctx->wr_red) CK(cudaMalloc(&ctx->wr_red, (size_t)(ctx->world + 1) * sizeof(unsigned long long)));
    return WAFER_OK;
}

static void wr_host_site(const Geom& g, unsigned long long s, unsigned long long* gi, unsigned long long* j,
                         unsigned long long* k) {
    const unsigned long long plane = (unsigned long long)g.ny * (unsigned long long)g.nz, li = s / plane, r = s % plane;
    *gi = (unsigned long long)g.x0 + li;
    *j = r / (unsigned long long)g.nz;
    *k = r % (unsigned long long)g.nz;
}

struct WrJob {
    const double* f;
    int fmt;
    unsigned long long nsites;
    long long nblocks;
    std::vector<unsigned long long> btot;  // bytes of each block
    std::vector<unsigned int> bflag;       // refused sites in each block
    unsigned long long host_formatted = 0;
};

// refused sites of blocks [b0, b1) with their %.17g text, sorted by site; *n = how many the launch met (more than
// ENC_FLAG_CAP: the list is incomplete and the caller splits the range).  bt: the blocks' certified bytes.
static int wr_collect(wafer_ctx* ctx, const WrJob& job, long long b0, long long b1, std::vector<EncFlagStr>* txt,
                      unsigned long long* n, std::vector<unsigned int>* bt) {
    const Geom& g = ctx->g;
    CK(cudaMemsetAsync(ctx->wr_count, 0, sizeof(unsigned long long), ctx->s_main));
    const unsigned grid = (unsigned)(b1 - b0);
    if (job.fmt == enc::FMT_CSV)
        encode_len_kernel<enc::FMT_CSV><<<grid, ENC_THREADS, 0, ctx->s_main>>>(job.f, g, b0, job.nsites, ctx->pow10, ctx->wr_btot, ctx->wr_flags, ctx->wr_count);
    else
        encode_len_kernel<enc::FMT_JSON><<<grid, ENC_THREADS, 0, ctx->s_main>>>(job.f, g, b0, job.nsites, ctx->pow10, ctx->wr_btot, ctx->wr_flags, ctx->wr_count);
    TRY(post_launch(ctx));
    CK(cudaMemcpyAsync(n, ctx->wr_count, sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->s_main));
    if (bt) {
        bt->resize(grid);
        CK(cudaMemcpyAsync(bt->data(), ctx->wr_btot + b0, grid * sizeof(unsigned int), cudaMemcpyDeviceToHost, ctx->s_main));
    }
    CK(cudaStreamSynchronize(ctx->s_main));
    txt->clear();
    if (*n == 0 || *n > ENC_FLAG_CAP) return WAFER_OK;
    std::vector<EncFlagIn> in(*n);
    CK(cudaMemcpyAsync(in.data(), ctx->wr_flags, *n * sizeof(EncFlagIn), cudaMemcpyDeviceToHost, ctx->s_main));
    CK(cudaStreamSynchronize(ctx->s_main));
    std::sort(in.begin(), in.end(), [](const EncFlagIn& a, const EncFlagIn& b) { return a.site < b.site; });
    txt->resize(*n);
    for (size_t i = 0; i < in.size(); ++i) {
        EncFlagStr& e = (*txt)[i];
        e.site = in[i].site;
        e.len = (unsigned int)snprintf(e.s, sizeof e.s, "%.17g", in[i].v);
    }
    return WAFER_OK;
}

// pass 1 over blocks [b0, b1): job.btot / job.bflag
static int wr_measure(wafer_ctx* ctx, WrJob& job, long long b0, long long b1) {
    std::vector<EncFlagStr> txt;
    std::vector<unsigned int> bt;
    unsigned long long n = 0;
    TRY(wr_collect(ctx, job, b0, b1, &txt, &n, &bt));
    if (n > ENC_FLAG_CAP) {  // pieces of ENC_FLAG_CAP sites cannot overflow the list
        for (long long p = b0; p < b1; p += ENC_FLAG_CAP / ENC_BS)
            TRY(wr_measure(ctx, job, p, std::min<long long>(b1, p + ENC_FLAG_CAP / ENC_BS)));
        return WAFER_OK;
    }
    for (long long b = b0; b < b1; ++b) job.btot[b] = bt[b - b0];
    const enc::Pow10 t = enc::host_pow10();
    for (const EncFlagStr& e : txt) {
        unsigned long long gi, j, k;
        wr_host_site(ctx->g, e.site, &gi, &j, &k);
        char buf[enc::SITE_MAX];
        const int len = enc::encode_site(job.fmt, 0.0, gi, j, k, ctx->g.x0 == 0 && e.site == 0, e.s, (int)e.len, buf, t);
        job.btot[e.site / ENC_BS] += (unsigned long long)len;
        job.bflag[e.site / ENC_BS] += 1;
        job.host_formatted += 1;
    }
    return WAFER_OK;
}

static int wr_allreduce(wafer_ctx* ctx, std::vector<unsigned long long>& v) {
    if (ctx->world == 1) return WAFER_OK;
    CK(cudaMemcpyAsync(ctx->wr_red, v.data(), v.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice, ctx->s_main));
    NK(nccl_api().AllReduce(ctx->wr_red, ctx->wr_red, v.size(), kNcclUint64, kNcclSum, ctx->comm, ctx->s_main));
    CK(cudaMemcpyAsync(v.data(), ctx->wr_red, v.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->s_main));
    CK(cudaStreamSynchronize(ctx->s_main));
    return WAFER_OK;
}

static bool wr_pwrite(int fd, const void* p, size_t n, unsigned long long off, std::string* err) {
    const char* c = (const char*)p;
    while (n > 0) {
        const ssize_t w = pwrite(fd, c, n, (off_t)off);
        if (w < 0 && errno == EINTR) continue;
        if (w <= 0) {
            *err = std::string("write failed: ") + (w < 0 ? strerror(errno) : "no progress");
            return false;
        }
        c += w;
        n -= (size_t)w;
        off += (unsigned long long)w;
    }
    return true;
}

// pass 2: encode, copy and write every chunk; `ok` / `io_err` report the first failed write (the GPU work is still
// drained so that the buffers are free on return)
static int wr_emit(wafer_ctx* ctx, const WrJob& job, const std::vector<unsigned long long>& boff, int fd,
                   unsigned long long data_off, bool* ok, std::string* io_err) {
    const Geom& g = ctx->g;
    CK(cudaMemsetAsync(ctx->wr_count + 1, 0, sizeof(unsigned long long), ctx->s_main));
    const size_t cap = ctx->ring.bytes;
    TRY(ring_start(ctx));
    unsigned long long pend_bytes = 0, pend_off = 0;
    int k = 0;
    for (long long cb = 0; cb < job.nblocks; ++k) {
        long long ce = cb + 1;
        while (ce < job.nblocks && boff[ce + 1] - boff[cb] <= cap) ++ce;
        const int buf = k & 1;
        const unsigned long long bytes = boff[ce] - boff[cb];
        TRY(ring_out(ctx, buf, ctx->ring.host[buf], bytes, [&](void* slot) -> int {
            unsigned char* out = (unsigned char*)slot;
            for (long long pb = cb; pb < ce;) {
                long long pe = pb;
                unsigned long long nf = 0;
                while (pe < ce && nf + job.bflag[pe] <= ENC_FLAG_CAP) nf += job.bflag[pe++];
                int ntxt = 0;
                if (nf > 0) {
                    std::vector<EncFlagStr> txt;
                    unsigned long long n = 0;
                    TRY(wr_collect(ctx, job, pb, pe, &txt, &n, nullptr));
                    if (n != nf) { ctx->err = "wafer_write_array: the refused sites differ between the passes"; return WAFER_ERR_CUDA; }
                    CK(cudaMemcpyAsync(ctx->wr_txt, txt.data(), txt.size() * sizeof(EncFlagStr), cudaMemcpyHostToDevice, ctx->s_main));
                    CK(cudaStreamSynchronize(ctx->s_main));
                    ntxt = (int)n;
                }
                const unsigned grid = (unsigned)(pe - pb);
                switch (job.fmt) {
                    case enc::FMT_MPK: encode_emit_kernel<enc::FMT_MPK><<<grid, ENC_THREADS, 0, ctx->s_main>>>(job.f, g, pb, job.nsites, ctx->pow10, ctx->wr_boff, boff[cb], ctx->wr_txt, ntxt, out, ctx->wr_count + 1); break;
                    case enc::FMT_CSV: encode_emit_kernel<enc::FMT_CSV><<<grid, ENC_THREADS, 0, ctx->s_main>>>(job.f, g, pb, job.nsites, ctx->pow10, ctx->wr_boff, boff[cb], ctx->wr_txt, ntxt, out, ctx->wr_count + 1); break;
                    default: encode_emit_kernel<enc::FMT_JSON><<<grid, ENC_THREADS, 0, ctx->s_main>>>(job.f, g, pb, job.nsites, ctx->pow10, ctx->wr_boff, boff[cb], ctx->wr_txt, ntxt, out, ctx->wr_count + 1); break;
                }
                TRY(post_launch(ctx));
                pb = pe;
            }
            return WAFER_OK;
        }));
        if (k > 0) {  // chunk k - 1 is written while chunk k is encoded and copied
            TRY(ring_wait(ctx, buf ^ 1));
            if (*ok) *ok = wr_pwrite(fd, ctx->ring.host[buf ^ 1], pend_bytes, data_off + pend_off, io_err);
        }
        pend_bytes = bytes;
        pend_off = boff[cb];
        cb = ce;
    }
    TRY(ring_wait(ctx, (k - 1) & 1));
    if (*ok) *ok = wr_pwrite(fd, ctx->ring.host[(k - 1) & 1], pend_bytes, data_off + pend_off, io_err);
    unsigned long long missing = 0;
    CK(cudaMemcpyAsync(&missing, ctx->wr_count + 1, sizeof(missing), cudaMemcpyDeviceToHost, ctx->s_main));
    CK(cudaStreamSynchronize(ctx->s_main));
    if (missing) { ctx->err = "wafer_write_array: a refused site had no host text"; return WAFER_ERR_CUDA; }
    return WAFER_OK;
}

namespace {
struct FdGuard {
    int fd = -1;
    ~FdGuard() {
        if (fd >= 0) close(fd);
    }
};
}  // namespace

static int write_array_impl(wafer_ctx* ctx, int32_t what, int32_t file_type, const char* path, wafer_write_stats* stats) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(what == 0 || what == 1, "what must be 0 (psi) or 1 (V)");
    REQUIRE(file_type >= 0 && file_type <= 2,
            "file_type must be 0 (Messagepack), 1 (Csv) or 2 (Json); Yaml and Ron files are not supported");
    REQUIRE(path, "path is NULL");
    const Geom& g = ctx->g;
    char pre[96];
    int npre = 0;
    if (file_type == enc::FMT_MPK) {
        npre = enc::mpk_preamble((uint64_t)g.gnx, (uint64_t)g.gny, (uint64_t)g.gnz, (unsigned char*)pre);
        REQUIRE(npre >= 0, "Messagepack: an array of more than 2^32-1 elements cannot be written (array32 limit)");
    } else if (file_type == enc::FMT_JSON) {
        npre = enc::json_preamble((uint64_t)g.gnx, (uint64_t)g.gny, (uint64_t)g.gnz, pre);
    }
    if (what == 0) TRY(ready(ctx, false));
    else if (!ctx->have_v) { ctx->err = "potential not set (wafer_set_potential / wafer_generate_potential)"; return WAFER_ERR_NOT_READY; }
    CK(cudaSetDevice(ctx->dev));
    const int rank = ctx->rank, world = ctx->world;

    WrJob job;
    job.f = what == 0 ? ctx->psi[ctx->cur] : ctx->v;
    job.fmt = file_type;
    job.nsites = (unsigned long long)g.L * (unsigned long long)g.ny * (unsigned long long)g.nz;
    job.nblocks = (long long)((job.nsites + ENC_BS - 1) / ENC_BS);
    job.btot.assign(job.nblocks, 0);
    job.bflag.assign(job.nblocks, 0);
    TRY(wr_buffers(ctx, job.nblocks));
    if (file_type == enc::FMT_MPK) {
        for (long long b = 0; b < job.nblocks; ++b)
            job.btot[b] = 9ull * (std::min<unsigned long long>(job.nsites, (unsigned long long)(b + 1) * ENC_BS) - (unsigned long long)b * ENC_BS);
    } else {
        for (long long b = 0; b < job.nblocks; b += 4096) TRY(wr_measure(ctx, job, b, std::min<long long>(job.nblocks, b + 4096)));
    }
    std::vector<unsigned long long> boff(job.nblocks + 1, 0);
    for (long long b = 0; b < job.nblocks; ++b) boff[b + 1] = boff[b] + job.btot[b];
    CK(cudaMemcpyAsync(ctx->wr_boff, boff.data(), boff.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice, ctx->s_main));

    // every rank opens the one file; no rank writes unless all could
    FdGuard fd;
    fd.fd = open(path, O_WRONLY | O_CREAT | O_CLOEXEC, 0666);
    std::string io_err = fd.fd < 0 ? std::string("cannot create ") + path + ": " + strerror(errno) : std::string();
    std::vector<unsigned long long> red(world + 1, 0);
    red[rank] = boff[job.nblocks];
    red[world] = fd.fd < 0 ? 1 : 0;
    TRY(wr_allreduce(ctx, red));
    if (red[world]) {
        ctx->err = io_err.empty() ? std::string("another rank cannot create ") + path : io_err;
        return WAFER_ERR_IO;
    }
    unsigned long long before = 0, all = 0;
    for (int q = 0; q < world; ++q) {
        if (q < rank) before += red[q];
        all += red[q];
    }
    const unsigned long long trailer = file_type == enc::FMT_JSON ? 2 : 0;
    const unsigned long long file_bytes = (unsigned long long)npre + all + trailer;
    bool ok = true;
    if (rank == 0) {  // a longer file of the same name loses its tail; the ranks write every byte below file_bytes
        if (ftruncate(fd.fd, (off_t)file_bytes) != 0) {
            io_err = std::string("cannot truncate ") + path + ": " + strerror(errno);
            ok = false;
        }
        if (ok && npre) ok = wr_pwrite(fd.fd, pre, (size_t)npre, 0, &io_err);
    }
    if (ok && rank == world - 1 && trailer) ok = wr_pwrite(fd.fd, "]}", 2, (unsigned long long)npre + all, &io_err);
    if (ok) TRY(wr_emit(ctx, job, boff, fd.fd, (unsigned long long)npre + before, &ok, &io_err));
    if (close(fd.fd) != 0 && ok) {
        io_err = std::string("close failed: ") + strerror(errno);
        ok = false;
    }
    fd.fd = -1;
    std::vector<unsigned long long> agree(1, ok ? 0 : 1);  // every rank returns the same status
    TRY(wr_allreduce(ctx, agree));
    if (agree[0]) {
        ctx->err = io_err.empty() ? std::string("another rank could not write ") + path : path + std::string(": ") + io_err;
        return WAFER_ERR_IO;
    }
    if (stats) {
        stats->bytes = boff[job.nblocks] + (rank == 0 ? (unsigned long long)npre : 0) + (rank == world - 1 ? trailer : 0);
        stats->file_bytes = file_bytes;
        stats->host_formatted = job.host_formatted;
    }
    return WAFER_OK;
}

int wafer_write_array(wafer_ctx* ctx, int32_t what, int32_t file_type, const char* path, wafer_write_stats* stats) {
    try {
        return write_array_impl(ctx, what, file_type, path, stats);
    } catch (const std::exception& e) {  // host-side allocation failures must not unwind through the C ABI
        if (ctx) ctx->err = std::string("wafer_write_array: ") + e.what();
        return WAFER_ERR_INVALID;
    }
}

// ---- array files decoded on the device (decode.cuh) -----------------------------------------------------------
// The preamble (and Json's trailer, a Csv file's last record) is read on the host; the shape rules give the source
// planes this rank needs, converted into one device buffer.  The body is then read with pread into the two pinned
// halves of the staging ring, chunk after chunk; each goes to the device through its slot and is decoded on s_main
// while the next one is read.  A chunk ends after its last separator, the rest is carried into the next.  Once a
// chunk's kernels are done its uncertified numbers are converted with strtod from the pinned buffer it is still in.
// The field changes only after the whole file has been read and found canonical: then resample_kernel reads the
// buffer.
static int dec_buffers(wafer_ctx* ctx) {
    TRY(ring_reserve(ctx, FILE_MIN_STG, true));
    TRY(pow10_table(ctx));
    const long long nb = (long long)(ctx->ring.bytes / DEC_SEG) + 1;
    if (ctx->rd_blocks < nb) {
        for (int b = 0; b < 2; ++b) {
            cudaFree(ctx->rd_bcount[b]);
            cudaFree(ctx->rd_boff[b]);
            ctx->rd_bcount[b] = nullptr;
            ctx->rd_boff[b] = nullptr;
        }
        ctx->rd_blocks = 0;
        for (int b = 0; b < 2; ++b) {
            CK(cudaMalloc(&ctx->rd_bcount[b], (size_t)nb * sizeof(unsigned int)));
            CK(cudaMalloc(&ctx->rd_boff[b], (size_t)nb * sizeof(unsigned long long)));
        }
        ctx->rd_blocks = nb;
    }
    if (!ctx->rd_st) {
        for (int b = 0; b < 2; ++b) CK(cudaMalloc(&ctx->rd_flags[b], DEC_FLAG_CAP * sizeof(DecFlag)));
        CK(cudaMalloc(&ctx->rd_st, (2 * DEC_WORDS + 1) * sizeof(unsigned long long)));
        CK(cudaMallocHost(&ctx->rd_hst, 2 * DEC_WORDS * sizeof(unsigned long long)));
    }
    return WAFER_OK;
}

static bool rd_pread(int fd, void* p, size_t n, unsigned long long off, std::string* err) {
    char* c = (char*)p;
    while (n > 0) {
        const ssize_t r = pread(fd, c, n, (off_t)off);
        if (r < 0 && errno == EINTR) continue;
        if (r <= 0) {
            *err = std::string("read failed: ") + (r < 0 ? strerror(errno) : "unexpected end of file");
            return false;
        }
        c += r;
        n -= (size_t)r;
        off += (unsigned long long)r;
    }
    return true;
}

struct RdChunk {
    int buf;
    const unsigned char* c;  // the slot it was copied to
    unsigned long long len;  // bytes of whole records
    long long nblocks;
};

struct RdJob {
    int fmt;
    DecDst d;
    unsigned long long host_converted = 0;
};

static int rd_launch_text(wafer_ctx* ctx, const RdJob& job, const RdChunk& ch, long long b0, long long b1) {
    unsigned long long* st = ctx->rd_st + DEC_WORDS * ch.buf;
    CK(cudaMemsetAsync(st + DEC_NFLAG, 0, sizeof(unsigned long long), ctx->s_main));
    if (job.fmt == enc::FMT_CSV)
        dec_text_kernel<enc::FMT_CSV><<<(unsigned)(b1 - b0), DEC_THREADS, 0, ctx->s_main>>>(ch.c, ch.len, b0, ctx->rd_boff[ch.buf], ctx->pow10, job.d, ctx->rd_flags[ch.buf], st);
    else
        dec_text_kernel<enc::FMT_JSON><<<(unsigned)(b1 - b0), DEC_THREADS, 0, ctx->s_main>>>(ch.c, ch.len, b0, ctx->rd_boff[ch.buf], ctx->pow10, job.d, ctx->rd_flags[ch.buf], st);
    TRY(post_launch(ctx));
    CK(cudaMemcpyAsync(ctx->rd_hst + DEC_WORDS * ch.buf, st, DEC_WORDS * sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                       ctx->s_main));
    return WAFER_OK;
}

// convert the listed numbers of blocks [b0, b1) of the chunk (its kernels done) with strtod and store them
static int rd_host_convert(wafer_ctx* ctx, RdJob& job, const RdChunk& ch, long long b0, long long b1) {
    const unsigned long long* hst = ctx->rd_hst + DEC_WORDS * ch.buf;
    if (hst[DEC_ERR]) return WAFER_ERR_FORMAT;
    const unsigned long long n = hst[DEC_NFLAG];
    if (n == 0) return WAFER_OK;
    if (n > DEC_FLAG_CAP) {  // the list overflowed: again in pieces of 16 blocks, which cannot overflow it
        for (long long p = b0; p < b1; p += DEC_FLAG_CAP / DEC_SEG) {
            const long long pe = std::min<long long>(b1, p + DEC_FLAG_CAP / DEC_SEG);
            TRY(rd_launch_text(ctx, job, ch, p, pe));
            CK(cudaStreamSynchronize(ctx->s_main));
            TRY(rd_host_convert(ctx, job, ch, p, pe));
        }
        return WAFER_OK;
    }
    std::vector<DecFlag> list(n);
    CK(cudaMemcpyAsync(list.data(), ctx->rd_flags[ch.buf], n * sizeof(DecFlag), cudaMemcpyDeviceToHost, ctx->s_main));
    CK(cudaStreamSynchronize(ctx->s_main));
    const char* hb = (const char*)ctx->ring.host[ch.buf];
    std::string tok;
    for (DecFlag& f : list) {
        if ((unsigned long long)f.at + f.len > ch.len) { ctx->err = "wafer_load_array: a listed number lies outside its chunk"; return WAFER_ERR_CUDA; }
        tok.assign(hb + f.at, f.len);  // the grammar of parse_f64 is a subset of strtod's: it takes the whole token
        char* end = nullptr;
        f.v = strtod(tok.c_str(), &end);
        if (end != tok.c_str() + tok.size()) return WAFER_ERR_FORMAT;
    }
    CK(cudaMemcpyAsync(ctx->rd_flags[ch.buf], list.data(), n * sizeof(DecFlag), cudaMemcpyHostToDevice, ctx->s_main));
    dec_scatter_kernel<<<(unsigned)std::min<unsigned long long>((n + 255) / 256, 1024), 256, 0, ctx->s_main>>>(job.d, ctx->rd_flags[ch.buf], (int)n);
    TRY(post_launch(ctx));
    CK(cudaStreamSynchronize(ctx->s_main));  // `list` is freed on return
    job.host_converted += n;
    return WAFER_OK;
}

// a chunk whose kernels are queued: wait for them, then its status and its uncertified numbers
static int rd_finish(wafer_ctx* ctx, RdJob& job, const RdChunk& ch) {
    TRY(ring_wait(ctx, ch.buf));
    if (ctx->rd_hst[DEC_WORDS * ch.buf + DEC_ERR]) return WAFER_ERR_FORMAT;
    if (job.fmt == enc::FMT_MPK) return WAFER_OK;
    return rd_host_convert(ctx, job, ch, 0, ch.nblocks);
}

// bytes [b0, b1) of the file: every chunk decoded into job.d
static int rd_stream(wafer_ctx* ctx, RdJob& job, int fd, unsigned long long b0, unsigned long long b1, std::string* io) {
    const unsigned char sep = job.fmt == enc::FMT_CSV ? '\n' : ',';
    const unsigned long long cap = job.fmt == enc::FMT_MPK ? ctx->ring.bytes / 9 * 9 : ctx->ring.bytes;
    unsigned long long off = b0, carry = 0;
    RdChunk prev{0, nullptr, 0, 0};
    CK(cudaMemsetAsync(ctx->rd_st, 0, (2 * DEC_WORDS + 1) * sizeof(unsigned long long), ctx->s_main));
    TRY(ring_start(ctx));
    for (int k = 0; off < b1; ++k) {
        const int buf = k & 1;
        unsigned char* hb = ctx->ring.host[buf];
        const unsigned long long e0 = (off - b0) / 9;  // Messagepack: the chunk's first element
        if (carry) memcpy(hb, ctx->ring.host[buf ^ 1] + prev.len, carry);  // chunk k - 1's split record
        const unsigned long long n = std::min(cap - carry, b1 - off);
        if (!rd_pread(fd, hb + carry, n, off, io)) return WAFER_ERR_IO;
        off += n;
        unsigned long long len = carry + n;
        carry = 0;
        if (off < b1 && job.fmt != enc::FMT_MPK) {  // end the chunk after its last separator
            unsigned long long cut = len;
            while (cut > 0 && hb[cut - 1] != sep) --cut;
            if (cut == 0) return WAFER_ERR_FORMAT;  // a record longer than a slot
            carry = len - cut;
            len = cut;
        }
        RdChunk ch{buf, nullptr, len, (long long)((len + DEC_SEG - 1) / DEC_SEG)};
        TRY(ring_in(ctx, buf, hb, len, [&](void* slot) -> int {
            ch.c = (const unsigned char*)slot;
            unsigned long long* st = ctx->rd_st + DEC_WORDS * buf;
            if (job.fmt == enc::FMT_MPK) {
                const unsigned long long nel = len / 9;
                dec_mpk_kernel<<<(unsigned)std::min<unsigned long long>((nel + DEC_THREADS - 1) / DEC_THREADS, (unsigned long long)ctx->sm_count * 16),
                                 DEC_THREADS, 0, ctx->s_main>>>(ch.c, nel, e0, job.d, st);
                TRY(post_launch(ctx));
                CK(cudaMemcpyAsync(ctx->rd_hst + DEC_WORDS * buf, st, DEC_WORDS * sizeof(unsigned long long), cudaMemcpyDeviceToHost,
                                   ctx->s_main));
                return WAFER_OK;
            }
            dec_count_kernel<<<(unsigned)ch.nblocks, DEC_THREADS, 0, ctx->s_main>>>(ch.c, len, sep, ctx->rd_bcount[buf]);
            dec_offsets_kernel<<<1, 1024, 0, ctx->s_main>>>(ctx->rd_bcount[buf], (int)ch.nblocks, ctx->rd_boff[buf],
                                                            ctx->rd_st + 2 * DEC_WORDS);
            TRY(post_launch(ctx, 2));
            return rd_launch_text(ctx, job, ch, 0, ch.nblocks);
        }));
        if (k > 0) TRY(rd_finish(ctx, job, prev));  // chunk k - 1, while chunk k is decoded
        prev = ch;
    }
    if (off > b0) TRY(rd_finish(ctx, job, prev));
    if (job.fmt != enc::FMT_MPK) {  // every site had its record
        unsigned long long recs = 0;
        CK(cudaMemcpyAsync(&recs, ctx->rd_st + 2 * DEC_WORDS, sizeof(recs), cudaMemcpyDeviceToHost, ctx->s_main));
        CK(cudaStreamSynchronize(ctx->s_main));
        if (recs != job.d.n) return WAFER_ERR_FORMAT;
    }
    return WAFER_OK;
}

namespace {
struct DevBuf {  // the converted source planes; freed once the work queued on them is done
    wafer_ctx* ctx;
    double* p = nullptr;
    ~DevBuf() {
        ring_drain(ctx);
        cudaFree(p);
    }
};
}  // namespace

static int load_array_impl(wafer_ctx* ctx, int32_t what, int32_t file_type, const char* path, wafer_load_stats* stats) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(what >= 0 && what <= 2, "what must be 0 (psi), 1 (V) or 2 (push a lower state)");
    REQUIRE(file_type >= 0 && file_type <= 2,
            "file_type must be 0 (Messagepack), 1 (Csv) or 2 (Json); Yaml and Ron files are not supported");
    REQUIRE(path, "path is NULL");
    CK(cudaSetDevice(ctx->dev));
    FdGuard fd;
    fd.fd = open(path, O_RDONLY | O_CLOEXEC);
    std::string io;
    struct stat sb;
    if (fd.fd < 0 || fstat(fd.fd, &sb) != 0) {
        ctx->err = std::string("wafer_load_array: cannot open ") + path + ": " + strerror(errno);
        return WAFER_ERR_IO;
    }
    const unsigned long long size = (unsigned long long)sb.st_size;
    auto not_canonical = [&](const char* why) {
        ctx->err = std::string("wafer_load_array: ") + path + ": " + why + " (not a layout the device decoder reads)";
        return WAFER_ERR_FORMAT;
    };
    auto io_error = [&]() {
        ctx->err = std::string("wafer_load_array: ") + path + ": " + io;
        return WAFER_ERR_IO;
    };
    // preamble, trailer, dims: the body [b0, b1) holds the records
    uint64_t dims[3] = {0, 0, 0};
    unsigned long long b0 = 0, b1 = size;
    unsigned char head[128], tail[4096];
    const unsigned long long nh = std::min<unsigned long long>(size, sizeof head);
    if (!rd_pread(fd.fd, head, nh, 0, &io)) return io_error();
    if (file_type == enc::FMT_MPK) {
        uint64_t count = 0;
        const int h = dec::mpk_header(head, nh, dims, &count);
        if (h < 0) return not_canonical("Messagepack preamble");
        b0 = (unsigned long long)h;
    } else if (file_type == enc::FMT_JSON) {
        const int h = dec::json_header(head, nh, dims);
        if (h < 0) return not_canonical("Json preamble");
        const unsigned long long nt = std::min<unsigned long long>(size - (unsigned long long)h, 8);
        if (!rd_pread(fd.fd, tail, nt, size - nt, &io)) return io_error();
        const int tl = dec::json_trailer(tail, nt);
        if (tl < 0) return not_canonical("Json trailer");
        b0 = (unsigned long long)h;
        b1 = size - (unsigned long long)tl;
    } else {
        const unsigned long long nt = std::min<unsigned long long>(size, sizeof tail);
        if (!rd_pread(fd.fd, tail, nt, size - nt, &io)) return io_error();
        if (!dec::csv_dims(tail, nt, nt == size, dims)) return not_canonical("Csv last record");
    }
    if (!dec::body_fits(file_type, dims[0] * dims[1] * dims[2], b1 - b0))
        return not_canonical("the file is too short for its dims");
    RsPlan pl;
    TRY(resample_shape(ctx, dims[0], dims[1], dims[2], file_type == enc::FMT_CSV ? 1 : 0, &pl));
    TRY(dec_buffers(ctx));
    RdJob job;
    job.fmt = file_type;
    job.d.n = dims[0] * dims[1] * dims[2];
    job.d.plane = dims[1] * dims[2];
    job.d.sz = dims[2];
    job.d.p0 = (unsigned long long)pl.sp0;
    job.d.p1 = (unsigned long long)pl.sp1;
    DevBuf src{ctx};
    const unsigned long long nsrc = (unsigned long long)(pl.sp1 - pl.sp0) * job.d.plane;  // <= n <= file bytes
    if (nsrc > SIZE_MAX / sizeof(double) || cudaMalloc(&src.p, (size_t)nsrc * sizeof(double)) != cudaSuccess) {
        cudaGetLastError();
        src.p = nullptr;
        return not_canonical("the source planes do not fit the device");
    }
    job.d.dst = src.p;
    const int rc = rd_stream(ctx, job, fd.fd, b0, b1, &io);
    if (rc == WAFER_ERR_IO) return io_error();
    if (rc == WAFER_ERR_FORMAT) return not_canonical(file_type == enc::FMT_MPK ? "an element is not a float 64" : "a record is not canonical");
    TRY(rc);
    TRY(set_input(ctx, what, [&](double* dst) -> int {
        rs_launch(ctx, pl, dst, src.p, pl.sp0, dims[0], dims[1], dims[2], pl.ga, pl.gb);
        TRY(post_launch(ctx));
        CK(cudaStreamSynchronize(ctx->s_main));
        return WAFER_OK;
    }));
    if (stats) {
        stats->sx = dims[0];
        stats->sy = dims[1];
        stats->sz = dims[2];
        stats->bytes_read = size;
        stats->sites_converted = nsrc;
        stats->host_converted = job.host_converted;
    }
    return WAFER_OK;
}

int wafer_load_array(wafer_ctx* ctx, int32_t what, int32_t file_type, const char* path, wafer_load_stats* stats) {
    try {
        return load_array_impl(ctx, what, file_type, path, stats);
    } catch (const std::exception& e) {  // host-side allocation failures must not unwind through the C ABI
        if (ctx) ctx->err = std::string("wafer_load_array: ") + e.what();
        return WAFER_ERR_INVALID;
    }
}

int wafer_observables_compute(wafer_ctx* ctx, wafer_observables* out) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(out, "out is NULL");
    TRY(ready(ctx, true));
    CK(cudaSetDevice(ctx->dev));
    TRY(observables_device(ctx));
    double s[4];
    TRY(read_scalars(ctx, SL_OBS, 4, s));
    out->energy = s[0]; out->norm2 = s[1]; out->v_infinity = s[2]; out->r2 = s[3];
    return WAFER_OK;
}

int wafer_norm2(wafer_ctx* ctx, double* out) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(out, "out is NULL");
    TRY(ready(ctx, false));
    CK(cudaSetDevice(ctx->dev));
    const Geom& g = ctx->g;
    const long long ob = (long long)g.gx * g.plane / 2, oe = (long long)(g.gx + g.L) * g.plane / 2;
    const int grid = ew_grid(ctx, oe - ob);
    norm2_kernel<<<grid, EW_THREADS, 0, ctx->s_main>>>(ctx->psi[ctx->cur], ob, oe, ctx->partials);
    TRY(post_launch(ctx));
    TRY(finalize(ctx, 1, grid, SL_TMP, ctx->s_main));
    return read_scalars(ctx, SL_TMP, 1, out);
}

int wafer_normalise(wafer_ctx* ctx, double norm2) {
    if (!ctx) return WAFER_ERR_INVALID;
    ctx->chk_valid = false;  // psi (or what the check sums depend on) changes
    TRY(ready(ctx, false));
    CK(cudaSetDevice(ctx->dev));
    set_scalar_kernel<<<1, 1, 0, ctx->s_main>>>(ctx->scal + SL_TMP, norm2);
    TRY(post_launch(ctx));
    return gs_apply(ctx, ctx->psi[ctx->cur], ctx->scal + SL_TMP, 0);
}

int wafer_orthogonalise(wafer_ctx* ctx, uint8_t wnum) {
    if (!ctx) return WAFER_ERR_INVALID;
    ctx->chk_valid = false;  // psi (or what the check sums depend on) changes
    TRY(ready(ctx, false));
    // grid.rs:478: w_store.iter().take(wnum) — silently clamps to the stored count
    const int n = std::min<int>(wnum, (int)ctx->lowers.size());
    if (n == 0) return WAFER_OK;
    CK(cudaSetDevice(ctx->dev));
    return gs_apply(ctx, ctx->psi[ctx->cur], nullptr, n);
}

// one excited-state step on a single rank (grid.rs:567-681): sweep with the fused sums, then normalise + Gram-Schmidt
static int excited_step(wafer_ctx* ctx, int wnum) {
    const Geom& g = ctx->g;
    const int src = ctx->cur;
    const int nred = ctx->use_t1 ? 1 + std::min(wnum, t1::MAX_FUSED_LOWERS) : 1;
    TRY(launch_sweep(ctx, ctx->psi[src], ctx->psi[src ^ 1], 0, g.L, nred, 0, ctx->s_main));
    ctx->cur ^= 1;
    return gs_apply(ctx, ctx->psi[src ^ 1], ctx->scal + SL_RAW, wnum, nred, sweep_blocks(ctx, 0, g.L));
}


// `pairs` times two excited-state steps through a captured graph.  Returns WAFER_OK with *ran = false when graphs are not
// to be used (several ranks, or the capture failed: the caller then steps the ordinary way).
static int excited_pairs_graph(wafer_ctx* ctx, int wnum, uint64_t pairs, bool* ran) {
    *ran = false;
    if (ctx->world != 1 || pairs == 0) return WAFER_OK;
    const std::pair<int, int> key{wnum, ctx->cur};
    auto it = ctx->step_graphs.find(key);
    if (it == ctx->step_graphs.end()) {
        cudaGraph_t graph = nullptr;
        cudaGraphExec_t exec = nullptr;
        const uint64_t launches0 = ctx->launches;
        const int cur0 = ctx->cur;
        if (cudaStreamBeginCapture(ctx->s_main, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); return WAFER_OK; }
        int rc = excited_step(ctx, wnum);
        if (rc == WAFER_OK) rc = excited_step(ctx, wnum);
        const cudaError_t ce = cudaStreamEndCapture(ctx->s_main, &graph);
        const int per_pair = (int)(ctx->launches - launches0);
        ctx->launches = launches0;  // nothing ran yet
        ctx->cur = cur0;
        if (rc != WAFER_OK || ce != cudaSuccess || !graph || cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) {
            if (graph) cudaGraphDestroy(graph);
            cudaGetLastError();
            return WAFER_OK;
        }
        cudaGraphDestroy(graph);
        it = ctx->step_graphs.emplace(key, std::make_pair(exec, per_pair)).first;
    }
    for (uint64_t i = 0; i < pairs; ++i) CK(cudaGraphLaunch(it->second.first, ctx->s_main));
    ctx->launches += pairs * (uint64_t)it->second.second;
    *ran = true;
    return WAFER_OK;
}

static int wafer_evolve_impl(wafer_ctx* ctx, uint8_t wnum_in, uint64_t steps) {
    if (!ctx) return WAFER_ERR_INVALID;
    TRY(ready(ctx, true));
    CK(cudaSetDevice(ctx->dev));
    const Geom& g = ctx->g;
    const int wnum = std::min<int>(wnum_in, (int)ctx->lowers.size());
    const bool excited = wnum_in > 0;  // grid.rs:674: norm/normalise run for wnum > 0 even with an empty w_store
    // every rank must take the same branch (one side calling NCCL while the other stores through peer memory would
    // hang): decide from the smallest slab of the decomposition, not from this rank's own L
    const bool overlap = ctx->world > 1 && !excited && ctx->min_L > 2 * g.gx;
    // (before the events below: the halo stream's launches must come after the build of h as well)
    if (((ctx->use_tb && !excited) || (ctx->use_t1 && t1_reads_h())) && steps >= 4)
        TRY(ensure_hfield(ctx));  // one 16 B/site pass: pays for itself after two sweep pairs
    if (overlap) {
        CK(cudaEventRecord(ctx->ev_main, ctx->s_main));
        CK(cudaEventRecord(ctx->ev_halo, ctx->s_main));
    }
    const uint64_t total = steps == 0 ? 1 : steps;  // grid.rs:562-686 is a do-while: steps == 0 still sweeps once
    const bool fused = overlap && ctx->p2p;  // halo stores fused into the boundary kernels (peer memory), no NCCL
    // North-star "block reductions fused into the final sweep before each check": the LAST step of a ground-state evolve
    // runs as a one-step sweep that also accumulates sum psi^2, sum psi^2 pot_sub and sum psi^2 r2 of its output; the
    // check that follows then only needs the energy pass.  Worth one non-time-tiled pass only on long calls.
    const bool fuse_chk = ctx->use_t1 && !excited && total >= 64 && !(ctx->p.flags & WAFER_FLAG_NO_FUSED_CHECK);
    ctx->chk_valid = false;
    int chk_nb = 0;
    const int has_lo = ctx->rank > 0, has_hi = ctx->rank < ctx->world - 1;
    uint64_t done = 0;
    if (excited && ctx->world == 1 && wnum <= t1::MAX_FUSED_LOWERS && total >= 8) {
        bool ran = false;
        TRY(excited_pairs_graph(ctx, wnum, total / 2, &ran));
        if (ran) done = (total / 2) * 2;
    }
    while (done < total) {
        // ground state: two steps per HBM pass with the time-tiled TMA kernel whenever two steps remain;
        // excited states need a global norm / Gram-Schmidt after EVERY step (grid.rs:674-681): one step per pass
        const bool last = total - done == 1;
        const bool two = ctx->use_tb && !excited && total - done >= 2 && !(fuse_chk && total - done == 2);
        const int chk_mode = (fuse_chk && last) ? t1::MODE_CHK + ctx->potsub_mode : 0;
        const int b = g.gx;  // boundary planes = ghost depth the neighbours keep (2 for ThreePoint, else ext)
        const int src = ctx->cur;
        const double* cur = ctx->psi[src];
        double* nxt = ctx->psi[src ^ 1];
        // Fused halos, two-step pass, "whole column" form: ONE launch on the main stream sweeps all owned planes and
        // stores its first / last two output planes into the neighbours' ghost planes as it produces them; the neighbours'
        // pass counters are awaited before it and published after it.  No separate boundary launches: those produce 2 planes
        // for 6 plane-iterations of pipeline (140 instead of 132 iterations per tile column at 128 planes per rank, and four
        // small launches that the persistent interior kernel serialises behind itself anyway — 0.894 parallel efficiency at
        // N = 8, profiles/scaling_r2).  The price is a per-pass handshake between neighbours instead of a pass of slack.
        if (fused && two) {
            CK(cudaStreamWaitEvent(ctx->s_main, ctx->ev_halo, 0));  // an earlier pass may have used the halo stream
            if (ctx->dbg_halo_delay_ns) {
                spin_kernel<<<1, 1, 0, ctx->s_main>>>(ctx->dbg_halo_delay_ns);
                TRY(post_launch(ctx));
            }
            // counter >= P: the neighbours have finished pass P-1 — their stores into my ghost planes of `cur` have landed,
            // and they no longer read the ghost planes (of their `nxt`) that this pass overwrites
            p2p_wait_kernel<<<1, 1, 0, ctx->s_main>>>(ctx->flags, ctx->pass, has_lo, has_hi, ctx->p2p_timeout);
            TRY(post_launch(ctx));
            // my planes [0,b) are the lower neighbour's ghost planes [L_lo, L_lo+b); my [L-b,L) the upper one's [-b,0)
            tb::PeerStores pr{0, 0, INT_MIN, INT_MAX};
            if (has_lo) { pr.delta_lo = (ctx->peer_psi[0][src ^ 1] - nxt) + (long long)ctx->peer_L[0] * g.plane; pr.lo_end = b; }
            if (has_hi) { pr.delta_hi = (ctx->peer_psi[1][src ^ 1] - nxt) - (long long)g.L * g.plane; pr.hi_begin = g.L - b; }
            TRY(launch_sweep_tb2(ctx, src, 0, g.L, ctx->s_main, &pr));
            ctx->pass += 1;
            p2p_signal_kernel<<<1, 1, 0, ctx->s_main>>>(has_lo ? ctx->peer_flags[0] : nullptr, has_hi ? ctx->peer_flags[1] : nullptr, ctx->pass);
            TRY(post_launch(ctx));
            CK(cudaEventRecord(ctx->ev_main, ctx->s_main));
            CK(cudaEventRecord(ctx->ev_halo, ctx->s_main));
        } else if (overlap) {
            // boundary planes + halo on the high-priority stream, interior on the main stream (a two-step pass gets here only
            // with the NCCL halo: with fused halos it takes the branch above)
            CK(cudaStreamWaitEvent(ctx->s_halo, ctx->ev_main, 0));
            CK(cudaStreamWaitEvent(ctx->s_main, ctx->ev_halo, 0));
            if (ctx->dbg_halo_delay_ns) {
                spin_kernel<<<1, 1, 0, ctx->s_halo>>>(ctx->dbg_halo_delay_ns);
                TRY(post_launch(ctx));
            }
            if (fused) {
                // my ghost planes of `cur` hold the neighbours' pass-(n-1) boundary planes once their flag says so;
                // the same flag says they are done reading the ghost planes (of their `nxt`) that I overwrite now
                p2p_wait_kernel<<<1, 1, 0, ctx->s_halo>>>(ctx->flags, ctx->pass, has_lo, has_hi, ctx->p2p_timeout);
                TRY(post_launch(ctx));
            }
            if (two) {
                TRY(launch_sweep_tb2(ctx, src, 0, b, ctx->s_halo));
                TRY(launch_sweep_tb2(ctx, src, g.L - b, g.L, ctx->s_halo));
            } else {
                // (final step with fused check sums: the three launches share one row of per-CTA partial sums)
                const int nb_lo = sweep_blocks(ctx, 0, b), nb_hi = sweep_blocks(ctx, g.L - b, g.L);
                chk_nb = chk_mode ? nb_lo + nb_hi + sweep_blocks(ctx, b, g.L - b) : 0;
                TRY(launch_sweep(ctx, cur, nxt, 0, b, chk_mode, 0, ctx->s_halo, chk_nb, 0));
                TRY(launch_sweep(ctx, cur, nxt, g.L - b, g.L, chk_mode, 0, ctx->s_halo, chk_nb, nb_lo));
                if (fused) {  // rare odd tail step: plain peer copies of the boundary planes
                    const size_t bytes = (size_t)b * g.plane * sizeof(double);
                    if (has_lo) CK(cudaMemcpyAsync(ctx->peer_psi[0][src ^ 1] + g.off(ctx->peer_L[0], -g.e, 0), nxt + g.off(0, -g.e, 0), bytes, cudaMemcpyDeviceToDevice, ctx->s_halo));
                    if (has_hi) CK(cudaMemcpyAsync(ctx->peer_psi[1][src ^ 1] + g.off(-b, -g.e, 0), nxt + g.off(g.L - b, -g.e, 0), bytes, cudaMemcpyDeviceToDevice, ctx->s_halo));
                }
            }
            if (fused) {
                ctx->pass += 1;
                p2p_signal_kernel<<<1, 1, 0, ctx->s_halo>>>(has_lo ? ctx->peer_flags[0] : nullptr, has_hi ? ctx->peer_flags[1] : nullptr, ctx->pass);
                TRY(post_launch(ctx));
            } else {
                TRY(exchange(ctx, nxt, ctx->s_halo));
            }
            CK(cudaEventRecord(ctx->ev_halo, ctx->s_halo));
            if (two) TRY(launch_sweep_tb2(ctx, src, b, g.L - b, ctx->s_main));
            else TRY(launch_sweep(ctx, cur, nxt, b, g.L - b, chk_mode, 0, ctx->s_main, chk_nb, chk_nb - sweep_blocks(ctx, b, g.L - b)));
            CK(cudaEventRecord(ctx->ev_main, ctx->s_main));
        } else {
            // excited states: sum psi'^2 and (TMA kernel) the overlaps with up to four stored states ride on the sweep
            const int nred = !excited ? chk_mode : (ctx->use_t1 ? 1 + std::min(wnum, t1::MAX_FUSED_LOWERS) : 1);
            if (chk_mode) chk_nb = sweep_blocks(ctx, 0, g.L);
            if (two) TRY(launch_sweep_tb2(ctx, src, 0, g.L, ctx->s_main));
            else TRY(launch_sweep(ctx, cur, nxt, 0, g.L, nred, 0, ctx->s_main));
            TRY(exchange(ctx, nxt, ctx->s_main));
            ctx->cur ^= 1;
            // grid.rs:674-681: norm2 -> normalise -> orthogonalise, every step
            if (excited) TRY(gs_apply(ctx, nxt, ctx->scal + SL_RAW, wnum, nred, sweep_blocks(ctx, 0, g.L)));
        }
        if (overlap) ctx->cur ^= 1;
        done += two ? 2 : 1;
    }
    if (overlap) {
        if (fused) {
            // The neighbours' boundary stores of the LAST pass must have landed in my ghost planes before anything
            // that follows on the main stream reads them (observables, Gram-Schmidt, downloads, w_store.push) or
            // overwrites them (normalise, uploads): wait for their pass counter to reach mine.  Without this a rank
            // that runs ahead returns with ghost planes that are one same-buffer pass (4 steps) old.
            p2p_wait_kernel<<<1, 1, 0, ctx->s_halo>>>(ctx->flags, ctx->pass, has_lo, has_hi, ctx->p2p_timeout);
            TRY(post_launch(ctx));
            CK(cudaEventRecord(ctx->ev_halo, ctx->s_halo));
        }
        CK(cudaStreamWaitEvent(ctx->s_main, ctx->ev_halo, 0));
    }
    if (fuse_chk && chk_nb > 0) {
        gs_coeff_kernel<true, false><<<1, 1024, 0, ctx->s_main>>>(ctx->partials, chk_nb, 3, ctx->scal + SL_CHK, 0, nullptr, nullptr,
                                                                    nullptr, 0, nullptr);
        TRY(post_launch(ctx));
        ctx->chk_valid = true;
    }
    return WAFER_OK;
}

int wafer_push_lower(wafer_ctx* ctx, const double* q_padded) {
    try {
        return wafer_push_lower_impl(ctx, q_padded);
    } catch (const std::exception& e) {  // host-side allocation failures must not unwind through the C ABI
        if (ctx) ctx->err = std::string("wafer_push_lower: ") + e.what();
        return WAFER_ERR_INVALID;
    }
}

int wafer_push_lower_from_phi(wafer_ctx* ctx) {
    try {
        return wafer_push_lower_from_phi_impl(ctx);
    } catch (const std::exception& e) {  // host-side allocation failures must not unwind through the C ABI
        if (ctx) ctx->err = std::string("wafer_push_lower_from_phi: ") + e.what();
        return WAFER_ERR_INVALID;
    }
}

int wafer_evolve(wafer_ctx* ctx, uint8_t wnum_in, uint64_t steps) {
    try {
        return wafer_evolve_impl(ctx, wnum_in, steps);
    } catch (const std::exception& e) {  // host-side allocation failures must not unwind through the C ABI
        if (ctx) ctx->err = std::string("wafer_evolve: ") + e.what();
        return WAFER_ERR_INVALID;
    }
}

int wafer_check(wafer_ctx* ctx, uint8_t wnum_in, wafer_observables* out) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(out, "out is NULL");
    TRY(ready(ctx, true));
    CK(cudaSetDevice(ctx->dev));
    const int wnum = std::min<int>(wnum_in, (int)ctx->lowers.size());
    TRY(observables_device(ctx));                // grid.rs:127
    TRY(gs_apply(ctx, ctx->psi[ctx->cur], ctx->scal + SL_OBS + 1, wnum));  // grid.rs:130 normalise(norm2), 133-135 orthogonalise
    ctx->chk_valid = false;
    double s[4];
    TRY(read_scalars(ctx, SL_OBS, 4, s));
    out->energy = s[0]; out->norm2 = s[1]; out->v_infinity = s[2]; out->r2 = s[3];
    return WAFER_OK;
}

// grid.rs:50-246
int wafer_solve(wafer_ctx* ctx, uint8_t wnum, double tolerance, int64_t max_steps, uint64_t screen_update,
                uint64_t snap_update, wafer_record* records, uint64_t max_records, uint64_t* n_records) {
    if (!ctx) return WAFER_ERR_INVALID;
    TRY(ready(ctx, true));
    uint64_t step = 0, nrec = 0;
    double last_energy = 1.7976931348623157e308;  // f64::MAX (grid.rs:124)
    bool converged = false;
    for (;;) {
        wafer_observables obs;
        TRY(wafer_check(ctx, wnum, &obs));                                  // grid.rs:127-135
        if (!std::isfinite(obs.energy) || !std::isfinite(obs.norm2) || obs.norm2 == 0.0) {
            ctx->err = "non-finite observables (the reference's R64 would panic here)";
            return WAFER_ERR_NONFINITE;
        }
        const double norm_energy = obs.energy / obs.norm2;                  // grid.rs:128
        const double tau = (double)step * ctx->p.dt;                        // grid.rs:129
        if (snap_update != 0 && step % snap_update == 0)                    // grid.rs:137-139 (NotConstrained):
            TRY(wafer_normalise(ctx, obs.norm2));                           // second division by sqrt(norm2)
        const double diff = std::fabs(norm_energy - last_energy);           // grid.rs:161
        if (records && nrec < max_records) {
            records[nrec].step = step; records[nrec].tau = tau; records[nrec].diff = diff; records[nrec].obs = obs;
        }
        nrec++;
        if (diff < tolerance) { converged = true; break; }                  // grid.rs:162-192
        last_energy = norm_energy;                                          // grid.rs:194
        if (max_steps >= 0 && step > (uint64_t)max_steps) break;            // grid.rs:211-213 (strict >)
        TRY(wafer_evolve(ctx, wnum, screen_update));                        // grid.rs:216
        step += screen_update;                                              // grid.rs:220
    }
    if (n_records) *n_records = nrec;
    if (converged) {
        TRY(wafer_push_lower_from_phi(ctx));                                // grid.rs:241
        return WAFER_OK;
    }
    ctx->err = "Maximum step limit reached before convergence (ErrorKind::MaxStep)";
    return WAFER_ERR_MAX_STEP;
}

// ---- plumbing ----------------------------------------------------------------------------------------------
int wafer_synchronize(wafer_ctx* ctx) {
    if (!ctx) return WAFER_ERR_INVALID;
    CK(cudaSetDevice(ctx->dev));
    CK(cudaStreamSynchronize(ctx->s_halo));
    CK(cudaStreamSynchronize(ctx->s_main));
    return check_p2p_timeout(ctx);
}

int wafer_timer_begin(wafer_ctx* ctx) {
    if (!ctx) return WAFER_ERR_INVALID;
    CK(cudaSetDevice(ctx->dev));
    CK(cudaEventRecord(ctx->ev_t0, ctx->s_main));
    return WAFER_OK;
}

int wafer_timer_end(wafer_ctx* ctx, double* ms) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(ms, "ms is NULL");
    CK(cudaSetDevice(ctx->dev));
    CK(cudaEventRecord(ctx->ev_t1, ctx->s_main));
    CK(cudaEventSynchronize(ctx->ev_t1));
    float f = 0.f;
    CK(cudaEventElapsedTime(&f, ctx->ev_t0, ctx->ev_t1));
    *ms = (double)f;
    return WAFER_OK;
}

uint64_t wafer_kernel_launches(const wafer_ctx* ctx) { return ctx ? ctx->launches : 0; }

int wafer_host_alloc(void** ptr, size_t bytes) {
    if (!ptr) return WAFER_ERR_INVALID;
    return cudaMallocHost(ptr, bytes) == cudaSuccess ? WAFER_OK : WAFER_ERR_CUDA;
}

int wafer_host_free(void* ptr) { return cudaFreeHost(ptr) == cudaSuccess ? WAFER_OK : WAFER_ERR_CUDA; }

int wafer_host_register(void* ptr, size_t bytes) {
    if (!ptr || !bytes) return WAFER_ERR_INVALID;
    return cudaHostRegister(ptr, bytes, cudaHostRegisterDefault) == cudaSuccess ? WAFER_OK : WAFER_ERR_CUDA;
}

int wafer_host_unregister(void* ptr) { return cudaHostUnregister(ptr) == cudaSuccess ? WAFER_OK : WAFER_ERR_CUDA; }

int wafer_device_info(const wafer_ctx* ctx, char* name, size_t name_len, int32_t* sm_count, int32_t* cc_major,
                      int32_t* cc_minor, uint64_t* mem_bytes) {
    if (!ctx) return WAFER_ERR_INVALID;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, ctx->dev) != cudaSuccess) return WAFER_ERR_CUDA;
    if (name && name_len) { strncpy(name, prop.name, name_len - 1); name[name_len - 1] = 0; }
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    if (mem_bytes) *mem_bytes = prop.totalGlobalMem;
    return WAFER_OK;
}

// ---- fused halo over peer memory: export / import CUDA IPC handles of the psi buffers and the flag words ------
int wafer_p2p_export(wafer_ctx* ctx, uint8_t out[192]) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(out, "out is NULL");
    CK(cudaSetDevice(ctx->dev));
    if (!ctx->flags) {
        CK(cudaMalloc(&ctx->flags, 2 * sizeof(unsigned long long)));
        CK(cudaMemset(ctx->flags, 0, 2 * sizeof(unsigned long long)));
        CK(cudaMalloc(&ctx->p2p_timeout, sizeof(int)));
        CK(cudaMemset(ctx->p2p_timeout, 0, sizeof(int)));
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t h[3];
    CK(cudaIpcGetMemHandle(&h[0], ctx->psi[0]));
    CK(cudaIpcGetMemHandle(&h[1], ctx->psi[1]));
    CK(cudaIpcGetMemHandle(&h[2], ctx->flags));
    memcpy(out, h, 192);
    return WAFER_OK;
}

int wafer_p2p_connect(wafer_ctx* ctx, const uint8_t* lower, const uint8_t* upper) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(ctx->world > 1, "wafer_p2p_connect needs world > 1");
    REQUIRE(ctx->flags, "call wafer_p2p_export first");
    REQUIRE((ctx->rank == 0) == (lower == nullptr) && (ctx->rank == ctx->world - 1) == (upper == nullptr),
            "pass the export blobs of rank-1 and rank+1 (NULL at the ends of the chain)");
    CK(cudaSetDevice(ctx->dev));
    REQUIRE(!ctx->p2p, "wafer_p2p_connect was already called on this context");
    const uint8_t* blobs[2] = {lower, upper};
    for (int n = 0; n < 2; ++n) {
        if (!blobs[n]) continue;
        cudaIpcMemHandle_t h[3];
        memcpy(h, blobs[n], 192);
        void* p[3];
        for (int k = 0; k < 3; ++k) CK(cudaIpcOpenMemHandle(&p[k], h[k], cudaIpcMemLazyEnablePeerAccess));
        ctx->peer_psi[n][0] = (double*)p[0];
        ctx->peer_psi[n][1] = (double*)p[1];
        ctx->peer_flags[n] = (unsigned long long*)p[2];
        uint64_t x0, x1;
        wafer_slab_partition(ctx->p.nx, (uint32_t)ctx->world, (uint32_t)(ctx->rank + (n == 0 ? -1 : 1)), &x0, &x1);
        ctx->peer_L[n] = (int)(x1 - x0);
    }
    ctx->p2p = true;
    ctx->pass = 0;
    return WAFER_OK;
}

int wafer_selftest_division(wafer_ctx* ctx, double den, uint64_t n, uint64_t seed, uint64_t* mismatches) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(mismatches, "mismatches is NULL");
    CK(cudaSetDevice(ctx->dev));
    unsigned long long* d = nullptr;
    CK(cudaMalloc(&d, sizeof(unsigned long long)));
    CK(cudaMemsetAsync(d, 0, sizeof(unsigned long long), ctx->s_main));
    tb::div_selftest_kernel<<<ctx->sm_count * 8, 256, 0, ctx->s_main>>>(den, den_in_fast_window(den), n, seed, d);
    TRY(post_launch(ctx));
    unsigned long long h = 0;
    CK(cudaMemcpyAsync(&h, d, sizeof(h), cudaMemcpyDeviceToHost, ctx->s_main));
    CK(cudaStreamSynchronize(ctx->s_main));
    cudaFree(d);
    *mismatches = h;
    return WAFER_OK;
}

int wafer_phi_checksum(wafer_ctx* ctx, uint64_t x_begin, uint64_t x_end, uint64_t out[2]) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(out, "out is NULL");
    TRY(ready(ctx, false));
    CK(cudaSetDevice(ctx->dev));
    const Geom& g = ctx->g;
    if (!ctx->d_cksum) CK(cudaMalloc(&ctx->d_cksum, 2 * sizeof(unsigned long long)));
    CK(cudaMemsetAsync(ctx->d_cksum, 0, 2 * sizeof(unsigned long long), ctx->s_main));
    const long long xb = std::max<long long>((long long)x_begin, g.x0) - g.x0;
    const long long xe = std::min<long long>((long long)std::min<uint64_t>(x_end, (uint64_t)g.gnx), g.x0 + g.L) - g.x0;
    if (xe > xb) {
        const int grid = (int)std::min<long long>((xe - xb) * g.ny, (long long)ctx->sm_count * 16);
        checksum_kernel<<<grid, 256, 0, ctx->s_main>>>(ctx->psi[ctx->cur], g, (int)xb, (int)xe, ctx->d_cksum);
        TRY(post_launch(ctx));
    }
    unsigned long long h[2] = {0, 0};
    CK(cudaMemcpyAsync(h, ctx->d_cksum, sizeof(h), cudaMemcpyDeviceToHost, ctx->s_main));
    CK(cudaStreamSynchronize(ctx->s_main));
    out[0] = h[0]; out[1] = h[1];
    return check_p2p_timeout(ctx);
}

int wafer_debug_halo_delay(wafer_ctx* ctx, uint64_t nanoseconds) {
    if (!ctx) return WAFER_ERR_INVALID;
    REQUIRE(nanoseconds <= 1000000000ull, "delay is capped at one second per pass");
    ctx->dbg_halo_delay_ns = nanoseconds;
    return WAFER_OK;
}

const char* wafer_sweep_variant(const wafer_ctx* ctx) {
    if (!ctx) return "";
    if (ctx->use_tb) return ctx->p2p ? "tb2-tma/V-onfly+p2p-halo" : (ctx->use_t1 ? "tb2-tma/V-onfly+tma1" : "tb2-tma/V-onfly");
    if (ctx->use_t1) return "tma1/V-onfly";
    return ctx->onfly ? "simple-regqueue/V-onfly" : "simple-regqueue/AB-arrays";
}

}  // extern "C"
