// mt19937.cu -- NumPy's legacy MT19937 Gaussian stream drawn on the device, bit for bit.
//
// The word stream of each seed is cut into segments of J = 624 * 2^JUMP_Q words (whole twist blocks,
// whole 4-word attempts).  Segment start states come from F2-polynomial jump-ahead: the state after
// t words is g(T) s0 with g = x^t mod phi, phi the degree-19937 characteristic polynomial of
// MT19937 (found once per process by Berlekamp-Massey on 2 * 19937 output bits).  The polynomials
// x^(J 2^i) mod phi depend on nothing but J and are obtained by squaring only; they are cached.
//   plan:    level i of mt_jump_kernel applies x^(J 2^i) to the 2^i known start states (one warp
//            per jump, Horner: 19937 steps of "advance one word, XOR in the source state when the
//            coefficient is 1"), log2(S) launches for S segments; mt_count_kernel counts the
//            accepted attempts of every segment; the host scans the counts (one synchronisation).
//   execute: mt_write_kernel regenerates the segments that overlap the requested ranges, gives
//            each accepted attempt its pair index (warp ballot + the segment's base), computes f
//            with the extended log of mt19937.cuh and writes the outputs in range.  Pairs whose log
//            lies within w ulp of a rounding midpoint are listed; the host computes libm's log for
//            them (several threads) and mt_fixup_kernel finishes them with the same IEEE steps.
// Compiled with --fmad=false (see _build.py): no contraction anywhere in this file.
#include "common.cuh"
#include "mt19937.cuh"

#include <math.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <thread>
#include <vector>

namespace {

using namespace rla::mt;

constexpr int JUMP_Q = 9;                                 // J = 624 * 512 = 319488 words per segment
constexpr int64_t SEG_WORDS = int64_t(N) << JUMP_Q;
constexpr int SEG_BLOCKS = 1 << JUMP_Q;                   // twist blocks per segment
constexpr int PW = (DEG + 63) / 64;                       // 64-bit words of a reduced polynomial
constexpr int WARPS = 4;                                  // warps per CTA in every kernel here

// ---------------------------------------------------------------- host: F2 polynomials
using Poly = std::vector<uint64_t>;                       // bit i = coefficient of x^i

inline int get_bit(const uint64_t *p, int64_t i) { return int((p[i >> 6] >> (i & 63)) & 1u); }

// a ^= b << sh   (a has na words, bits shifted past the end are dropped)
void xor_shifted(uint64_t *a, int64_t na, const uint64_t *b, int64_t nb, int64_t sh) {
    const int64_t q = sh >> 6;
    const int r = int(sh & 63);
    for (int64_t k = 0; k < nb && k + q < na; ++k) {
        a[k + q] ^= b[k] << r;
        if (r && k + q + 1 < na) a[k + q + 1] ^= b[k] >> (64 - r);
    }
}

void twist_block(uint32_t *mt) {
    for (int i = 0; i < N; ++i) mt[i] = twist(mt[i], mt[(i + 1) % N], mt[(i + M) % N]);
}

// phi from Berlekamp-Massey on bit 0 of 2 * DEG outputs of a nonzero state: that bit sequence
// is a nonzero linear functional of the state, and phi is irreducible, so phi is its minimal
// polynomial
Poly compute_phi() {
    const int64_t nb = 2 * int64_t(DEG);
    const int64_t W = (nb + 63) / 64 + 2;
    uint32_t mt[N];
    mt[0] = 5489u;                                        // init_genrand(5489), the reference seed of MT19937
    for (int i = 1; i < N; ++i) mt[i] = 1812433253u * (mt[i - 1] ^ (mt[i - 1] >> 30)) + uint32_t(i);
    std::vector<uint64_t> rs(W, 0);                       // reversed sequence: rs bit j = s[nb - 1 - j]
    int pos = N;
    for (int64_t n = 0; n < nb; ++n) {
        if (pos == N) { twist_block(mt); pos = 0; }
        if (temper(mt[pos++]) & 1u) { const int64_t j = nb - 1 - n; rs[j >> 6] |= uint64_t(1) << (j & 63); }
    }
    std::vector<uint64_t> C(W, 0), B(W, 0), T;
    C[0] = B[0] = 1;
    int64_t L = 0, m = 1;
    for (int64_t n = 0; n < nb; ++n) {
        // discrepancy sum_{i=0..L} c_i s_{n-i}; s_{n-i} = rs bit (nb - 1 - n + i)
        const int64_t base = nb - 1 - n;
        uint64_t acc = 0;
        for (int64_t k = 0; k <= L / 64; ++k) {            // deg C <= L; bits past the sequence are 0
            const int64_t bit = base + 64 * k, q = bit >> 6;
            if (q >= W) break;
            const int r = int(bit & 63);
            uint64_t v = rs[q] >> r;
            if (r && q + 1 < W) v |= rs[q + 1] << (64 - r);
            acc ^= C[k] & v;
        }
        if (!(__builtin_popcountll(acc) & 1)) { ++m; continue; }
        if (2 * L <= n) {
            T = C;
            xor_shifted(C.data(), W, B.data(), W, m);
            L = n + 1 - L;
            B = T;
            m = 1;
        } else {
            xor_shifted(C.data(), W, B.data(), W, m);
            ++m;
        }
    }
    Poly phi(PW + 1, 0);                                  // phi_k = c_{L-k}, degree DEG
    if (L != DEG) return Poly();
    for (int64_t k = 0; k <= L; ++k)
        if (get_bit(C.data(), L - k)) phi[k >> 6] |= uint64_t(1) << (k & 63);
    return phi;
}

std::mutex g_poly_mu;
Poly g_phi;
std::vector<Poly> g_levels;                               // g_levels[i] = x^(J 2^i) mod phi

// reduce a polynomial of degree < 2 DEG (2 PW + 1 words) mod phi into PW words
Poly reduce(std::vector<uint64_t> &a) {
    const int64_t na = int64_t(a.size());
    for (int64_t j = 64 * na - 1; j >= DEG; --j)
        if (get_bit(a.data(), j)) xor_shifted(a.data(), na, g_phi.data(), PW + 1, j - DEG);
    return Poly(a.begin(), a.begin() + PW);
}

inline uint64_t spread32(uint32_t x) {
    uint64_t v = x;
    v = (v | (v << 16)) & 0x0000FFFF0000FFFFull;
    v = (v | (v << 8)) & 0x00FF00FF00FF00FFull;
    v = (v | (v << 4)) & 0x0F0F0F0F0F0F0F0Full;
    v = (v | (v << 2)) & 0x3333333333333333ull;
    v = (v | (v << 1)) & 0x5555555555555555ull;
    return v;
}

Poly sqr_mod(const Poly &p) {                             // squaring over F2 spreads the bits
    std::vector<uint64_t> a(2 * PW + 1, 0);
    for (int k = 0; k < PW; ++k) {
        a[2 * k] = spread32(uint32_t(p[k]));
        a[2 * k + 1] = spread32(uint32_t(p[k] >> 32));
    }
    return reduce(a);
}

Poly mulx_mod(const Poly &p) {
    std::vector<uint64_t> a(PW + 1, 0);
    for (int k = 0; k < PW; ++k) {
        a[k] |= p[k] << 1;
        a[k + 1] |= p[k] >> 63;
    }
    return reduce(a);
}

// phi and the level polynomials 0 .. nlev-1 (computed once, extended on demand)
bool ensure_levels(int nlev) {
    std::lock_guard<std::mutex> lk(g_poly_mu);
    if (g_phi.empty()) {
        g_phi = compute_phi();
        if (g_phi.empty()) return false;
    }
    if (g_levels.empty()) {
        Poly g(PW, 0);
        g[N / 64] = uint64_t(1) << (N % 64);              // x^624, already reduced
        for (int i = 0; i < JUMP_Q; ++i) g = sqr_mod(g);
        g_levels.push_back(g);
    }
    while (int(g_levels.size()) < nlev) g_levels.push_back(sqr_mod(g_levels.back()));
    return true;
}

Poly x_pow_mod(uint64_t t) {                              // x^t mod phi, left-to-right binary powering
    Poly r(PW, 0);
    r[0] = 1;
    for (int b = 63; b >= 0; --b) {
        r = sqr_mod(r);
        if ((t >> b) & 1u) r = mulx_mod(r);
    }
    return r;
}

// g(T) applied to a window state (the 624 raw words before the next output, oldest first)
void horner_host(const Poly &g, const uint32_t *src, uint32_t *dst) {
    std::vector<uint32_t> acc(N, 0);
    int h = 0;
    for (int j = DEG - 1; j >= 0; --j) {
        acc[h] = twist(acc[h], acc[(h + 1) % N], acc[(h + M) % N]);
        h = (h + 1) % N;
        if (get_bit(g.data(), j))
            for (int k = 0; k < N; ++k) acc[(h + k) % N] ^= src[k];
    }
    for (int k = 0; k < N; ++k) dst[k] = acc[(h + k) % N];
}

// ---------------------------------------------------------------- device
// one warp twists the 624-word block in shared memory in place, NumPy's order: word i needs the
// new word i - 227 (an earlier chunk of 32), the old word i + 1 (this chunk or the next) and, for
// i = 623, the new word 0
__device__ __forceinline__ void warp_twist(uint32_t *mt, int lane) {
#pragma unroll 1
    for (int base = 0; base < N; base += 32) {
        const int i = base + lane;
        uint32_t v = 0;
        if (i < N) v = twist(mt[i], mt[i + 1 < N ? i + 1 : 0], mt[i + M < N ? i + M : i + M - N]);
        __syncwarp();
        if (i < N) mt[i] = v;
        __syncwarp();
    }
}

struct StreamDesc {            // per stream of a plan (device copy)
    int64_t seg_begin, nseg;
};
struct ExecDesc {              // per stream of an execute call
    int64_t first, count, offset;
};

// level `lev` of the doubling: segment 2^lev + j <- x^(J 2^lev)(T) segment j
__global__ void __launch_bounds__(32 * WARPS) mt_jump_kernel(uint32_t *states, const StreamDesc *streams,
                                                             const uint64_t *poly, int lev) {
    __shared__ uint32_t sm[WARPS][2][N];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const StreamDesc sd = streams[blockIdx.y];
    const int64_t half = int64_t(1) << lev;
    const int64_t j = int64_t(blockIdx.x) * WARPS + warp;
    if (j >= half || half + j >= sd.nseg) return;
    uint32_t *acc = sm[warp][0], *src = sm[warp][1];
    const uint32_t *s = states + (sd.seg_begin + j) * N;
    for (int k = lane; k < N; k += 32) { src[k] = s[k]; acc[k] = 0; }
    __syncwarp();
    int h = 0;
#pragma unroll 1
    for (int jj = DEG - 1; jj >= 0; --jj) {
        if (lane == 0) {
            const int h1 = h + 1 < N ? h + 1 : 0, hm = h + M < N ? h + M : h + M - N;
            acc[h] = twist(acc[h], acc[h1], acc[hm]);
        }
        h = h + 1 < N ? h + 1 : 0;
        __syncwarp();
        if ((poly[jj >> 6] >> (jj & 63)) & 1u) {
            int idx = h + lane;
            if (idx >= N) idx -= N;
            for (int k = lane; k < N; k += 32) {
                acc[idx] ^= src[k];
                idx += 32;
                if (idx >= N) idx -= N;
            }
            __syncwarp();
        }
    }
    uint32_t *d = states + (sd.seg_begin + half + j) * N;
    int idx = h + lane;
    if (idx >= N) idx -= N;
    for (int k = lane; k < N; k += 32) {
        d[k] = acc[idx];
        idx += 32;
        if (idx >= N) idx -= N;
    }
}

// accepted attempts of every segment (no log here)
__global__ void __launch_bounds__(32 * WARPS) mt_count_kernel(const uint32_t *states, int64_t total_seg,
                                                              int64_t *counts) {
    __shared__ __align__(16) uint32_t sm[WARPS][N];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t seg = int64_t(blockIdx.x) * WARPS + warp;
    if (seg >= total_seg) return;
    uint32_t *mt = sm[warp];
    for (int k = lane; k < N; k += 32) mt[k] = states[seg * N + k];
    __syncwarp();
    int64_t cnt = 0;
#pragma unroll 1
    for (int blk = 0; blk < SEG_BLOCKS; ++blk) {
        warp_twist(mt, lane);
#pragma unroll
        for (int r = 0; r < 5; ++r) {
            const int a = 32 * r + lane;
            if (a < N / 4) {
                const uint4 q = reinterpret_cast<const uint4 *>(mt)[a];
                cnt += attempt(temper(q.x), temper(q.y), temper(q.z), temper(q.w)).accept;
            }
        }
        __syncwarp();
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (lane == 0) counts[seg] = cnt;
}

__device__ __forceinline__ int find_stream(const StreamDesc *streams, int nstreams, int64_t seg) {
    int lo = 0, hi = nstreams - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (streams[mid].seg_begin <= seg) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// outputs [first, first + count) of each stream at out + offset.  A flagged pair writes its raw
// x2 / x1 into its slots and lists (slot << 2 | mask, r2); mask bit 0: the x2 slot (output 2p) is
// in range at `slot`, bit 1: the x1 slot (2p + 1) is in range at slot + (mask & 1).
__global__ void __launch_bounds__(32 * WARPS) mt_write_kernel(const uint32_t *states, const int64_t *base,
                                                              const StreamDesc *streams, int nstreams,
                                                              const ExecDesc *exec, int64_t total_seg,
                                                              double scale, double w, double *out,
                                                              unsigned long long *nflag, int64_t cap,
                                                              int64_t *flag_code, double *flag_r2) {
    __shared__ __align__(16) uint32_t sm[WARPS][N];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t seg = int64_t(blockIdx.x) * WARPS + warp;
    if (seg >= total_seg) return;
    const int st = find_stream(streams, nstreams, seg);
    const ExecDesc ex = exec[st];
    if (ex.count <= 0) return;
    const int64_t p_lo = ex.first >> 1, p_hi = (ex.first + ex.count - 1) >> 1;
    int64_t run = base[seg];
    if (run > p_hi) return;
    if (seg + 1 < streams[st].seg_begin + streams[st].nseg && base[seg + 1] <= p_lo) return;
    uint32_t *mt = sm[warp];
    for (int k = lane; k < N; k += 32) mt[k] = states[seg * N + k];
    __syncwarp();
    const int64_t o_end = ex.first + ex.count;
    const unsigned lt = (1u << lane) - 1u;
#pragma unroll 1
    for (int blk = 0; blk < SEG_BLOCKS && run <= p_hi; ++blk) {
        warp_twist(mt, lane);
#pragma unroll 1
        for (int r = 0; r < 5; ++r) {
            const int a = 32 * r + lane;
            Attempt at;
            at.accept = false;
            if (a < N / 4) {
                const uint4 q = reinterpret_cast<const uint4 *>(mt)[a];
                at = attempt(temper(q.x), temper(q.y), temper(q.z), temper(q.w));
            }
            const unsigned bal = __ballot_sync(0xffffffffu, at.accept);
            const int64_t p = run + __popc(bal & lt);
            run += __popc(bal);
            if (!at.accept || p < p_lo || p > p_hi) continue;
            const int64_t o2 = 2 * p, o1 = 2 * p + 1;
            const bool in2 = o2 >= ex.first && o2 < o_end, in1 = o1 >= ex.first && o1 < o_end;
            const DD lg = ext_log(at.r2);
            if (near_midpoint(lg, w)) {
                const int mask = (in2 ? 1 : 0) | (in1 ? 2 : 0);
                const int64_t slot = ex.offset + ((in2 ? o2 : o1) - ex.first);
                if (in2) out[slot] = at.x2;
                if (in1) out[slot + (in2 ? 1 : 0)] = at.x1;
                const unsigned long long i = atomicAdd(nflag, 1ull);
                if ((int64_t)i < cap) {
                    flag_code[i] = (slot << 2) | mask;
                    flag_r2[i] = at.r2;
                }
            } else {
                const double f = gauss_f(lg.hi, at.r2);
                if (in2) out[ex.offset + (o2 - ex.first)] = gauss_out(scale, f, at.x2);
                if (in1) out[ex.offset + (o1 - ex.first)] = gauss_out(scale, f, at.x1);
            }
        }
        __syncwarp();
    }
}

__global__ void mt_fixup_kernel(const int64_t *flag_code, const double *flag_r2, const double *flag_log,
                                int64_t n, double scale, double *out) {
    const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t code = flag_code[i];
    const int mask = int(code & 3);
    const int64_t slot = code >> 2;
    const double f = gauss_f(flag_log[i], flag_r2[i]);
    if (mask & 1) out[slot] = gauss_out(scale, f, out[slot]);
    if (mask & 2) out[slot + (mask & 1)] = gauss_out(scale, f, out[slot + (mask & 1)]);
}

// ---------------------------------------------------------------- host: libm log
// log() of the C library, called through a volatile pointer: no vector math library (libmvec) and no
// compiler rewrite of the call, the same function the reference's NumPy calls in legacy_gauss
double (*volatile g_libm_log)(double) = ::log;

void libm_log_batch(const double *x, int64_t n, double *out) {
    if (n <= 0) return;
    const int64_t per = 1 << 16;
    int nt = int(std::min<int64_t>((n + per - 1) / per, std::max(1u, std::thread::hardware_concurrency())));
    nt = std::min(nt, 64);
    auto work = [&](int t) {
        const int64_t lo = n * t / nt, hi = n * (t + 1) / nt;
        double (*fn)(double) = g_libm_log;
        for (int64_t i = lo; i < hi; ++i) out[i] = fn(x[i]);
    };
    if (nt <= 1) { work(0); return; }
    std::vector<std::thread> th;
    for (int t = 1; t < nt; ++t) th.emplace_back(work, t);
    work(0);
    for (auto &t : th) t.join();
}

size_t align256(size_t b) { return (b + 255) & ~size_t(255); }

}  // namespace

struct rla_mt19937_plan {
    int64_t nstreams = 0, total_seg = 0, nlev = 0;
    std::vector<uint32_t> keys;                           // nstreams x 624
    std::vector<StreamDesc> streams;
    std::vector<int64_t> base;                            // per segment: pairs before it in its stream
    std::vector<int64_t> pairs;                           // per stream: pairs of all its segments
    void *ws = nullptr;                                   // device workspace given to rla_mt19937_plan_build
    // workspace layout
    size_t off_states = 0, off_base = 0, off_streams = 0, off_poly = 0, bytes = 0;
};

extern "C" int64_t rla_mt19937_segment_words(void) { return SEG_WORDS; }

extern "C" int rla_mt19937_plan_create(rla_mt19937_plan **plan, const uint32_t *keys, const int64_t *nseg,
                                       int64_t nstreams) {
    RLA_REQUIRE(plan && keys && nseg, "rla_mt19937_plan_create: null pointer");
    RLA_REQUIRE(nstreams >= 1 && nstreams <= 65535, "rla_mt19937_plan_create: nstreams must be in [1, 65535]");
    auto *p = new rla_mt19937_plan();
    p->nstreams = nstreams;
    p->keys.assign(keys, keys + nstreams * N);
    int64_t maxseg = 1;
    for (int64_t i = 0; i < nstreams; ++i) {
        if (nseg[i] < 1 || nseg[i] > (int64_t(1) << 30)) {
            delete p;
            return rla::fail(RLA_ERR_INVALID, "rla_mt19937_plan_create: nseg[%lld] = %lld out of [1, 2^30]",
                             (long long)i, (long long)nseg[i]);
        }
        p->streams.push_back(StreamDesc{p->total_seg, nseg[i]});
        p->total_seg += nseg[i];
        maxseg = std::max(maxseg, nseg[i]);
    }
    while ((int64_t(1) << p->nlev) < maxseg) ++p->nlev;
    p->off_states = 0;
    p->off_base = align256(size_t(p->total_seg) * N * 4);
    p->off_streams = p->off_base + align256(size_t(p->total_seg) * 8);
    p->off_poly = p->off_streams + align256(size_t(nstreams) * sizeof(StreamDesc));
    p->bytes = p->off_poly + size_t(std::max<int64_t>(p->nlev, 1)) * PW * 8;
    *plan = p;
    return RLA_OK;
}

extern "C" void rla_mt19937_plan_destroy(rla_mt19937_plan *plan) { delete plan; }

extern "C" size_t rla_mt19937_plan_workspace_bytes(const rla_mt19937_plan *plan) { return plan ? plan->bytes : 0; }

extern "C" int rla_mt19937_plan_build(rla_mt19937_plan *plan, void *ws_dev, size_t ws_bytes, void *stream) {
    RLA_REQUIRE(plan && ws_dev, "rla_mt19937_plan_build: null pointer");
    if (ws_bytes < plan->bytes)
        return rla::fail(RLA_ERR_WORKSPACE, "rla_mt19937_plan_build: workspace %zu < %zu bytes", ws_bytes, plan->bytes);
    if (!ensure_levels(int(plan->nlev)))
        return rla::fail(RLA_ERR_UNSUPPORTED, "rla_mt19937_plan_build: Berlekamp-Massey did not find degree 19937");
    cudaStream_t s = (cudaStream_t)stream;
    char *ws = (char *)ws_dev;
    uint32_t *states = (uint32_t *)(ws + plan->off_states);
    int64_t *base = (int64_t *)(ws + plan->off_base);
    StreamDesc *streams = (StreamDesc *)(ws + plan->off_streams);
    uint64_t *poly = (uint64_t *)(ws + plan->off_poly);
    for (int64_t i = 0; i < plan->nstreams; ++i)
        RLA_CUDA_CHECK(cudaMemcpyAsync(states + plan->streams[i].seg_begin * N, plan->keys.data() + i * N, N * 4,
                                       cudaMemcpyHostToDevice, s));
    RLA_CUDA_CHECK(cudaMemcpyAsync(streams, plan->streams.data(), plan->nstreams * sizeof(StreamDesc),
                                   cudaMemcpyHostToDevice, s));
    for (int64_t l = 0; l < plan->nlev; ++l)
        RLA_CUDA_CHECK(cudaMemcpyAsync(poly + l * PW, g_levels[l].data(), PW * 8, cudaMemcpyHostToDevice, s));
    int64_t maxseg = 0;
    for (auto &sd : plan->streams) maxseg = std::max(maxseg, sd.nseg);
    for (int64_t l = 0; l < plan->nlev; ++l) {
        const int64_t half = int64_t(1) << l;
        const int64_t jobs = std::min(half, maxseg - half);
        dim3 grid(unsigned((jobs + WARPS - 1) / WARPS), unsigned(plan->nstreams));
        mt_jump_kernel<<<grid, 32 * WARPS, 0, s>>>(states, streams, poly + l * PW, int(l));
        RLA_CUDA_CHECK(cudaGetLastError());
        rla::count_launch();
    }
    mt_count_kernel<<<unsigned((plan->total_seg + WARPS - 1) / WARPS), 32 * WARPS, 0, s>>>(states, plan->total_seg, base);
    RLA_CUDA_CHECK(cudaGetLastError());
    rla::count_launch();
    plan->base.assign(plan->total_seg, 0);
    RLA_CUDA_CHECK(cudaMemcpyAsync(plan->base.data(), base, plan->total_seg * 8, cudaMemcpyDeviceToHost, s));
    RLA_CUDA_CHECK(cudaStreamSynchronize(s));
    plan->pairs.assign(plan->nstreams, 0);
    for (int64_t i = 0; i < plan->nstreams; ++i) {
        int64_t run = 0;
        for (int64_t k = 0; k < plan->streams[i].nseg; ++k) {
            const int64_t c = plan->base[plan->streams[i].seg_begin + k];
            plan->base[plan->streams[i].seg_begin + k] = run;
            run += c;
        }
        plan->pairs[i] = run;
    }
    RLA_CUDA_CHECK(cudaMemcpyAsync(base, plan->base.data(), plan->total_seg * 8, cudaMemcpyHostToDevice, s));
    RLA_CUDA_CHECK(cudaStreamSynchronize(s));              // plan->base is pageable host memory
    plan->ws = ws_dev;
    return RLA_OK;
}

extern "C" int64_t rla_mt19937_plan_pairs(const rla_mt19937_plan *plan, int64_t i) {
    if (!plan || i < 0 || i >= plan->nstreams || plan->pairs.empty()) return -1;
    return plan->pairs[i];
}

extern "C" size_t rla_mt19937_execute_workspace_bytes(const rla_mt19937_plan *plan, int64_t flag_cap) {
    if (!plan || flag_cap < 0) return 0;
    return align256(size_t(plan->nstreams) * sizeof(ExecDesc)) + 256 + size_t(flag_cap) * 24;
}

extern "C" int rla_mt19937_normal_f64(const rla_mt19937_plan *plan, const int64_t *first, const int64_t *count,
                                      const int64_t *offset, double scale, double w, double *out_dev,
                                      int64_t out_len, void *ws_dev, size_t ws_bytes, int64_t flag_cap,
                                      double *staging_host, int64_t *nflagged, void *stream) {
    RLA_REQUIRE(plan && first && count && offset && nflagged, "rla_mt19937_normal_f64: null pointer");
    RLA_REQUIRE(plan->ws, "rla_mt19937_normal_f64: the plan has not been built");
    RLA_REQUIRE(w >= 0.0 && w <= 0.5, "rla_mt19937_normal_f64: w = %g outside [0, 0.5]", w);
    RLA_REQUIRE(flag_cap >= 0, "rla_mt19937_normal_f64: negative flag capacity");
    *nflagged = 0;
    int64_t total = 0;
    for (int64_t i = 0; i < plan->nstreams; ++i) {
        RLA_REQUIRE(first[i] >= 0 && count[i] >= 0 && offset[i] >= 0 && offset[i] + count[i] <= out_len,
                    "rla_mt19937_normal_f64: range of stream %lld outside the output", (long long)i);
        RLA_REQUIRE(first[i] + count[i] <= 2 * plan->pairs[i],
                    "rla_mt19937_normal_f64: stream %lld has %lld normals in its plan, %lld requested",
                    (long long)i, (long long)(2 * plan->pairs[i]), (long long)(first[i] + count[i]));
        total += count[i];
    }
    if (total == 0) return RLA_OK;
    RLA_REQUIRE(out_dev && ws_dev, "rla_mt19937_normal_f64: null pointer");
    const size_t need = rla_mt19937_execute_workspace_bytes(plan, flag_cap);
    if (ws_bytes < need)
        return rla::fail(RLA_ERR_WORKSPACE, "rla_mt19937_normal_f64: workspace %zu < %zu bytes", ws_bytes, need);
    cudaStream_t s = (cudaStream_t)stream;
    char *ws = (char *)ws_dev;
    ExecDesc *exec = (ExecDesc *)ws;
    const size_t off_cnt = align256(size_t(plan->nstreams) * sizeof(ExecDesc));
    unsigned long long *nflag = (unsigned long long *)(ws + off_cnt);
    int64_t *flag_code = (int64_t *)(ws + off_cnt + 256);
    double *flag_r2 = (double *)(flag_code + flag_cap);
    double *flag_log = flag_r2 + flag_cap;
    std::vector<ExecDesc> ed(plan->nstreams);
    for (int64_t i = 0; i < plan->nstreams; ++i) ed[i] = ExecDesc{first[i], count[i], offset[i]};
    RLA_CUDA_CHECK(cudaMemcpyAsync(exec, ed.data(), ed.size() * sizeof(ExecDesc), cudaMemcpyHostToDevice, s));
    RLA_CUDA_CHECK(cudaMemsetAsync(nflag, 0, 8, s));
    const char *pw = (const char *)plan->ws;
    mt_write_kernel<<<unsigned((plan->total_seg + WARPS - 1) / WARPS), 32 * WARPS, 0, s>>>(
        (const uint32_t *)(pw + plan->off_states), (const int64_t *)(pw + plan->off_base),
        (const StreamDesc *)(pw + plan->off_streams), int(plan->nstreams), exec, plan->total_seg, scale, w,
        out_dev, nflag, flag_cap, flag_code, flag_r2);
    RLA_CUDA_CHECK(cudaGetLastError());
    rla::count_launch();
    unsigned long long nf = 0;
    RLA_CUDA_CHECK(cudaMemcpyAsync(&nf, nflag, 8, cudaMemcpyDeviceToHost, s));
    RLA_CUDA_CHECK(cudaStreamSynchronize(s));
    *nflagged = int64_t(nf);
    if (nf == 0) return RLA_OK;
    if (int64_t(nf) > flag_cap)
        return rla::fail(RLA_ERR_WORKSPACE, "rla_mt19937_normal_f64: %llu flagged pairs, capacity %lld", nf,
                         (long long)flag_cap);
    RLA_REQUIRE(staging_host, "rla_mt19937_normal_f64: flagged pairs need host staging");
    RLA_CUDA_CHECK(cudaMemcpyAsync(staging_host, flag_r2, nf * 8, cudaMemcpyDeviceToHost, s));
    RLA_CUDA_CHECK(cudaStreamSynchronize(s));
    libm_log_batch(staging_host, int64_t(nf), staging_host);
    RLA_CUDA_CHECK(cudaMemcpyAsync(flag_log, staging_host, nf * 8, cudaMemcpyHostToDevice, s));
    mt_fixup_kernel<<<unsigned((nf + 255) / 256), 256, 0, s>>>(flag_code, flag_r2, flag_log, int64_t(nf), scale, out_dev);
    RLA_CUDA_CHECK(cudaGetLastError());
    rla::count_launch();
    RLA_CUDA_CHECK(cudaStreamSynchronize(s));              // the staging buffer is free again on return
    return RLA_OK;
}

// ---------------------------------------------------------------- host hooks (tests)
extern "C" int rla_mt19937_jump_host(const uint32_t *key_in, uint64_t steps, uint32_t *key_out) {
    RLA_REQUIRE(key_in && key_out, "rla_mt19937_jump_host: null pointer");
    if (!ensure_levels(1)) return rla::fail(RLA_ERR_UNSUPPORTED, "rla_mt19937_jump_host: no characteristic polynomial");
    Poly g;
    {
        std::lock_guard<std::mutex> lk(g_poly_mu);
        g = x_pow_mod(steps);
    }
    horner_host(g, key_in, key_out);
    return RLA_OK;
}

extern "C" int rla_mt19937_attempts_host(const uint32_t *words, int64_t n, double *x1, double *x2, double *r2,
                                         int8_t *accept) {
    RLA_REQUIRE(n >= 0 && (n == 0 || (words && x1 && x2 && r2 && accept)), "rla_mt19937_attempts_host: bad arguments");
    for (int64_t i = 0; i < n; ++i) {
        const Attempt a = attempt(words[4 * i], words[4 * i + 1], words[4 * i + 2], words[4 * i + 3]);
        x1[i] = a.x1;
        x2[i] = a.x2;
        r2[i] = a.r2;
        accept[i] = a.accept ? 1 : 0;
    }
    return RLA_OK;
}

extern "C" int rla_mt19937_ext_log_host(const double *x, int64_t n, double w, double *hi, double *lo, int8_t *flag) {
    RLA_REQUIRE(n >= 0 && (n == 0 || (x && hi && lo && flag)), "rla_mt19937_ext_log_host: bad arguments");
    for (int64_t i = 0; i < n; ++i) {
        RLA_REQUIRE(x[i] > 0.0 && x[i] < 1.0, "rla_mt19937_ext_log_host: x outside (0, 1)");
        const DD v = ext_log(x[i]);
        hi[i] = v.hi;
        lo[i] = v.lo;
        flag[i] = near_midpoint(v, w) ? 1 : 0;
    }
    return RLA_OK;
}

extern "C" int rla_libm_log_host(const double *x, int64_t n, double *out) {
    RLA_REQUIRE(n >= 0 && (n == 0 || (x && out)), "rla_libm_log_host: bad arguments");
    libm_log_batch(x, n, out);
    return RLA_OK;
}
