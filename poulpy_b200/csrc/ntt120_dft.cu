// ntt120_dft.cu -- batched forward / inverse negacyclic NTT of the NTT120 flavour (K1 / K2 of SURVEY.md 2.8).
//
// What is computed (reference: poulpy-cpu-ref/src/reference/ntt120/ntt.rs:558-684, vec_znx_dft.rs:177-409):
//   forward : i64 limb -> four planes of canonical residues, out_k[p] = sum_i a_i * psi_k^(i * (2*bitrev(p) + 1)),
//             i.e. the reference's bit-reversed frequency order (its DIF network after the psi^i twist);
//   inverse : planes -> centred i128 via CRT (arithmetic.rs:119-140), 1/n folded into the CRT constant.
// How: one CTA per limb (all four primes), the polynomial lives in padded shared memory, radix-8 register passes
// (three butterfly levels per shared-memory round trip) in the twist-free "block twiddle" Cooley-Tukey form
// (forward) / Gentleman-Sande form (inverse), Shoup multiplication with Harvey lazy reduction.  Global loads and
// stores are fused into the first / last pass and are fully coalesced (i64 in: 8 B/thread contiguous per warp;
// planes out: 32 B/thread; i128 out: 16 B/thread contiguous per warp).
#include <stdlib.h>

#include "internal.h"
#include "ntt120.cuh"

using namespace n120;

__constant__ CrtConsts c_crt;

// conflict-free padding for strides 1 (128-bit), 8, 64, 512: 4 extra words per 32
__device__ __forceinline__ int PAD(int idx) { return idx + ((idx >> 5) << 2); }
template <int L> struct Geo {
    static constexpr int NB = 1 << L;
    static constexpr int T = NB >= 8 ? NB / 8 : 1;         // threads per limb, 8 coefficients each
    static constexpr int R0 = (L % 3 == 0) ? 3 : (L % 3);  // levels of the (possibly short) top pass
    static constexpr int PLANE = NB + (NB >> 5) * 4 + 4;   // padded words per prime plane
};

// resident CTAs the register budget of the stand-alone transforms is sized for: two CTAs of 512 threads at n = 4096 (one CTA of 16 warps per SM
// at 100 registers left the passes latency bound), unconstrained below
#ifndef NTT_MINB
#define NTT_MINB(threads) (((threads) >= 128 && (threads) <= 512) ? 1024 / (threads) : 1)
#endif
template <int K, int NLEV> __device__ __forceinline__ void ct_radix8(uint32_t (&x)[8], const uint2 *__restrict__ tw, uint32_t hi) {
    constexpr uint32_t q = Prime<K>::q;
    {
        uint2 w = __ldg(tw + hi);
#pragma unroll
        for (int j = 0; j < 4; j++) ct_bf(x[j], x[j + 4], w, q);
    }
    if (NLEV >= 2) {
        const uint4 ww = __ldg(reinterpret_cast<const uint4 *>(tw + 2 * hi));
        const uint2 w0 = make_uint2(ww.x, ww.y), w1 = make_uint2(ww.z, ww.w);
        ct_bf(x[0], x[2], w0, q);
        ct_bf(x[1], x[3], w0, q);
        ct_bf(x[4], x[6], w1, q);
        ct_bf(x[5], x[7], w1, q);
    }
    if (NLEV >= 3) {
        const uint4 wa = __ldg(reinterpret_cast<const uint4 *>(tw + 4 * hi)), wb = __ldg(reinterpret_cast<const uint4 *>(tw + 4 * hi + 2));
        ct_bf(x[0], x[1], make_uint2(wa.x, wa.y), q);
        ct_bf(x[2], x[3], make_uint2(wa.z, wa.w), q);
        ct_bf(x[4], x[5], make_uint2(wb.x, wb.y), q);
        ct_bf(x[6], x[7], make_uint2(wb.z, wb.w), q);
    }
}
template <int K, int NLEV> __device__ __forceinline__ void gs_radix8(uint32_t (&x)[8], const uint2 *__restrict__ tw, uint32_t hi) {
    constexpr uint32_t q = Prime<K>::q;
    if (NLEV >= 3) {
        const uint4 wa = __ldg(reinterpret_cast<const uint4 *>(tw + 4 * hi)), wb = __ldg(reinterpret_cast<const uint4 *>(tw + 4 * hi + 2));
        gs_bf(x[0], x[1], make_uint2(wa.x, wa.y), q);
        gs_bf(x[2], x[3], make_uint2(wa.z, wa.w), q);
        gs_bf(x[4], x[5], make_uint2(wb.x, wb.y), q);
        gs_bf(x[6], x[7], make_uint2(wb.z, wb.w), q);
    }
    if (NLEV >= 2) {
        const uint4 ww = __ldg(reinterpret_cast<const uint4 *>(tw + 2 * hi));
        const uint2 w0 = make_uint2(ww.x, ww.y), w1 = make_uint2(ww.z, ww.w);
        gs_bf(x[0], x[2], w0, q);
        gs_bf(x[1], x[3], w0, q);
        gs_bf(x[4], x[6], w1, q);
        gs_bf(x[5], x[7], w1, q);
    }
    {
        uint2 w = __ldg(tw + hi);
#pragma unroll
        for (int j = 0; j < 4; j++) gs_bf(x[j], x[j + 4], w, q);
    }
}

struct NttJobs {
    LimbSet in, out;
    int jobs_per_batch;
    int total_jobs;
    const int *skip; // optional, per batch item: non-zero = leave this item alone (forward kernel only)
    int skip_list;   // skip[] is followed by a count and a compacted list of the items that are NOT skipped: skip[batch] = count,
                     // skip[batch + 1 ..] = their indices (written by the gadget kernel); the grid then strides over that list only
    long long and_mask; // i64 inputs are ANDed with this before the residue map (cnv_prepare's masked last limb); -1 = none
};

// ---------------------------------------------------------------------------------------------- forward
template <int K, int L> __device__ __forceinline__ void fwd_prime(const long long (&v)[8], uint32_t *__restrict__ plane,
                                                                 uint32_t *__restrict__ gout, const uint2 *__restrict__ tw,
                                                                 int t, bool active) {
    typedef Geo<L> G;
    constexpr uint32_t q = Prime<K>::q;
    uint32_t x[8];
#pragma unroll
    for (int j = 0; j < 8; j++) x[j] = from_i64<K>(v[j]);
    ct_radix8<K, G::R0>(x, tw, 1u);
    if (L == G::R0) { // n == 8: the top pass is the whole transform
        if (active) {
#pragma unroll
            for (int j = 0; j < 8; j++) gout[j] = csub(csub(x[j], 2 * q), q);
        }
        return;
    }
#pragma unroll
    for (int j = 0; j < 8; j++) plane[PAD(t + j * G::T)] = x[j];
}

template <int K, int L, int L0> __device__ __forceinline__ void fwd_mid(uint32_t *__restrict__ plane, uint32_t *__restrict__ gout,
                                                                       const uint2 *__restrict__ tw, int t, bool active, uint32_t root) {
    constexpr uint32_t q = Prime<K>::q;
    constexpr int SL = L - L0 - 3; // log2 of the in-group stride
    const int a = t >> SL, b = t & ((1 << SL) - 1);
    const int base = (a << (SL + 3)) | b;
    const uint32_t hi = (root << L0) | (uint32_t)a;
    uint32_t x[8];
    if (SL == 0) {
        const uint4 *p = reinterpret_cast<const uint4 *>(plane + PAD(base));
        uint4 u0 = p[0], u1 = p[1];
        x[0] = u0.x; x[1] = u0.y; x[2] = u0.z; x[3] = u0.w;
        x[4] = u1.x; x[5] = u1.y; x[6] = u1.z; x[7] = u1.w;
    } else {
#pragma unroll
        for (int j = 0; j < 8; j++) x[j] = plane[PAD(base + (j << SL))];
    }
    ct_radix8<K, 3>(x, tw, hi);
    if (SL == 0) {
        if (active) {
#pragma unroll
            for (int j = 0; j < 8; j++) x[j] = csub(csub(x[j], 2 * q), q);
            uint4 *o = reinterpret_cast<uint4 *>(gout + base);
            o[0] = make_uint4(x[0], x[1], x[2], x[3]);
            o[1] = make_uint4(x[4], x[5], x[6], x[7]);
        }
    } else {
#pragma unroll
        for (int j = 0; j < 8; j++) plane[PAD(base + (j << SL))] = x[j];
    }
}

template <int L, int L0> struct FwdMid {
    static __device__ __forceinline__ void run(uint32_t *sm, uint32_t *gout, const uint2 *tw, int n, int t, bool active,
                                               uint32_t root = 1u) {
        typedef Geo<L> G;
        fwd_mid<0, L, L0>(sm + 0 * G::PLANE, gout + 0 * n, tw + 0 * n, t, active, root);
        fwd_mid<1, L, L0>(sm + 1 * G::PLANE, gout + 1 * n, tw + 1 * n, t, active, root);
        fwd_mid<2, L, L0>(sm + 2 * G::PLANE, gout + 2 * n, tw + 2 * n, t, active, root);
        fwd_mid<3, L, L0>(sm + 3 * G::PLANE, gout + 3 * n, tw + 3 * n, t, active, root);
        if (L0 + 3 < L) __syncthreads();
        FwdMid<L, (L0 + 3 < L) ? L0 + 3 : L>::run(sm, gout, tw, n, t, active, root);
    }
};
template <int L> struct FwdMid<L, L> {
    static __device__ __forceinline__ void run(uint32_t *, uint32_t *, const uint2 *, int, int, bool, uint32_t = 1u) {}
};

template <int L, int LPC> __device__ __forceinline__ void ntt120_fwd_job(const NttJobs &jb, const uint2 *__restrict__ tw, uint32_t *smem, int b, int j,
                                                                         bool active, int slot, int t) {
    typedef Geo<L> G;
    const long long *gin = reinterpret_cast<const long long *>(jb.in.base + (size_t)b * jb.in.batch_stride + (size_t)j * jb.in.limb_stride);
    uint32_t *gout = reinterpret_cast<uint32_t *>(jb.out.base + (size_t)b * jb.out.batch_stride + (size_t)j * jb.out.limb_stride);
    uint32_t *sm = smem + slot * 4 * G::PLANE;
    constexpr int n = G::NB;

    long long v[8];
#pragma unroll
    for (int jj = 0; jj < 8; jj++) v[jj] = active ? (__ldg(gin + t + jj * G::T) & jb.and_mask) : 0;
    fwd_prime<0, L>(v, sm + 0 * G::PLANE, gout + 0 * n, tw + 0 * n, t, active);
    fwd_prime<1, L>(v, sm + 1 * G::PLANE, gout + 1 * n, tw + 1 * n, t, active);
    fwd_prime<2, L>(v, sm + 2 * G::PLANE, gout + 2 * n, tw + 2 * n, t, active);
    fwd_prime<3, L>(v, sm + 3 * G::PLANE, gout + 3 * n, tw + 3 * n, t, active);
    if (L > G::R0) {
        __syncthreads();
        FwdMid<L, (L > G::R0) ? G::R0 : L>::run(sm, gout, tw, n, t, active);
    }
}

template <int L, int LPC> __global__ void __launch_bounds__(Geo<L>::T *LPC, NTT_MINB(Geo<L>::T *LPC)) ntt120_fwd_kernel(NttJobs jb, const uint2 *__restrict__ tw) {
    typedef Geo<L> G;
    extern __shared__ __align__(16) uint32_t smem[];
    const int slot = threadIdx.x / G::T, t = threadIdx.x % G::T;
    if (jb.skip && jb.skip_list) { // the per-limb route of the gadget product: normally an empty list, the few CTAs leave at once
        const int batch = jb.total_jobs / jb.jobs_per_batch;
        const int nwork = __ldg(jb.skip + batch) * jb.jobs_per_batch;
        for (int base = blockIdx.x * LPC; base < nwork; base += gridDim.x * LPC) {
            const int job = base + slot;
            const bool active = job < nwork;
            const int b = active ? __ldg(jb.skip + batch + 1 + job / jb.jobs_per_batch) : 0, j = active ? job % jb.jobs_per_batch : 0;
            ntt120_fwd_job<L, LPC>(jb, tw, smem, b, j, active, slot, t);
            __syncthreads(); // the planes are reused by the next job
        }
        return;
    }
    const int job = blockIdx.x * LPC + slot;
    bool active = job < jb.total_jobs;
    const int b = active ? job / jb.jobs_per_batch : 0, j = active ? job % jb.jobs_per_batch : 0;
    if (jb.skip) {
        if (LPC == 1) {
            if (__ldg(jb.skip + b)) return; // CTA-uniform
        } else {
            active = active && !__ldg(jb.skip + b);
        }
    }
    ntt120_fwd_job<L, LPC>(jb, tw, smem, b, j, active, slot, t);
}

// ---------------------------------------------------------------------------------------------- inverse
// bottom pass: levels L-3..L-1 on 8 consecutive residues per thread, results to shared memory
template <int K, int L> __device__ __forceinline__ void inv_bottom_core(uint32_t (&x)[8], uint32_t *__restrict__ plane,
                                                                       const uint2 *__restrict__ tw, int t, uint32_t root = 1u) {
    constexpr int L0 = L - 3;
    const uint32_t hi = (root << L0) | (uint32_t)t;
    gs_radix8<K, 3>(x, tw, hi);
    uint4 *o = reinterpret_cast<uint4 *>(plane + PAD(8 * t));
    o[0] = make_uint4(x[0], x[1], x[2], x[3]);
    o[1] = make_uint4(x[4], x[5], x[6], x[7]);
}
// inputs read from global planes
template <int K, int L> __device__ __forceinline__ void inv_bottom(uint32_t *__restrict__ plane, const uint32_t *__restrict__ gin,
                                                                  const uint2 *__restrict__ tw, int t, bool active, uint32_t root = 1u) {
    uint32_t x[8];
    uint4 u0 = make_uint4(0, 0, 0, 0), u1 = u0;
    if (active) {
        const uint4 *p = reinterpret_cast<const uint4 *>(gin + 8 * t);
        u0 = __ldg(p);
        u1 = __ldg(p + 1);
    }
    x[0] = u0.x; x[1] = u0.y; x[2] = u0.z; x[3] = u0.w;
    x[4] = u1.x; x[5] = u1.y; x[6] = u1.z; x[7] = u1.w;
    inv_bottom_core<K, L>(x, plane, tw, t, root);
}
template <int K, int L, int L0> __device__ __forceinline__ void inv_mid(uint32_t *__restrict__ plane, const uint2 *__restrict__ tw, int t,
                                                                       uint32_t root) {
    constexpr int SL = L - L0 - 3;
    const int a = t >> SL, b = t & ((1 << SL) - 1);
    const int base = (a << (SL + 3)) | b;
    const uint32_t hi = (root << L0) | (uint32_t)a;
    uint32_t x[8];
#pragma unroll
    for (int j = 0; j < 8; j++) x[j] = plane[PAD(base + (j << SL))];
    gs_radix8<K, 3>(x, tw, hi);
#pragma unroll
    for (int j = 0; j < 8; j++) plane[PAD(base + (j << SL))] = x[j];
}
// passes from l0 = L-6 down to R0 (exclusive of the top pass)
template <int L, int L0> struct InvMid {
    static __device__ __forceinline__ void run(uint32_t *sm, const uint2 *tw, int n, int t, uint32_t root = 1u) {
        typedef Geo<L> G;
        inv_mid<0, L, L0>(sm + 0 * G::PLANE, tw + 0 * n, t, root);
        inv_mid<1, L, L0>(sm + 1 * G::PLANE, tw + 1 * n, t, root);
        inv_mid<2, L, L0>(sm + 2 * G::PLANE, tw + 2 * n, t, root);
        inv_mid<3, L, L0>(sm + 3 * G::PLANE, tw + 3 * n, t, root);
        __syncthreads();
        InvMid<L, (L0 - 3 >= G::R0) ? L0 - 3 : -1>::run(sm, tw, n, t, root);
    }
};
template <int L> struct InvMid<L, -1> {
    static __device__ __forceinline__ void run(uint32_t *, const uint2 *, int, int, uint32_t = 1u) {}
};

// top pass for one prime: R0 levels, then t_k = x * CRT_k / n and accumulation of t_k * (Q / Q_k)
template <int K, int L> __device__ __forceinline__ void inv_top(const uint32_t *__restrict__ plane, const uint32_t *__restrict__ gin,
                                                               const uint2 *__restrict__ tw, int t, bool active,
                                                               const Ntt120Consts &nc, u128 (&acc)[8]) {
    typedef Geo<L> G;
    constexpr uint32_t q = Prime<K>::q;
    uint32_t x[8];
    if (L == G::R0) {
#pragma unroll
        for (int j = 0; j < 8; j++) x[j] = active ? __ldg(gin + j) : 0;
    } else {
#pragma unroll
        for (int j = 0; j < 8; j++) x[j] = plane[PAD(t + j * G::T)];
    }
    gs_radix8<K, G::R0>(x, tw, 1u);
    const unsigned long long mlo = c_crt.m_lo[K], mhi = c_crt.m_hi[K];
#pragma unroll
    for (int j = 0; j < 8; j++) {
        uint32_t tk = csub(mul_shoup(x[j], nc.crt_ninv[K], nc.crt_ninv_sh[K], q), q);
        u128 p = (u128)tk * mlo + ((u128)((unsigned long long)tk * mhi) << 64);
        acc[j] += p;
    }
}

__device__ __forceinline__ i128 crt_finish(u128 v) {
    const u128 Q = ((u128)c_crt.q_hi << 64) | c_crt.q_lo;
    const u128 H = ((u128)c_crt.half_hi << 64) | c_crt.half_lo;
    unsigned qa = (unsigned)(v >> 120);
    v -= (u128)qa * Q;
    if (v >= Q) v -= Q;
    return v >= H ? (i128)v - (i128)Q : (i128)v;
}

// OUT_I128 = true : write centred i128 coefficients (VecZnxBig of the NTT120 flavour)
template <int L, int LPC> __global__ void __launch_bounds__(Geo<L>::T *LPC, NTT_MINB(Geo<L>::T *LPC)) ntt120_inv_kernel(NttJobs jb, const uint2 *__restrict__ tw,
                                                                                             Ntt120Consts nc) {
    typedef Geo<L> G;
    extern __shared__ __align__(16) uint32_t smem[];
    const int slot = threadIdx.x / G::T, t = threadIdx.x % G::T;
    const int job = blockIdx.x * LPC + slot;
    const bool active = job < jb.total_jobs;
    const int b = active ? job / jb.jobs_per_batch : 0, j = active ? job % jb.jobs_per_batch : 0;
    const uint32_t *gin = reinterpret_cast<const uint32_t *>(jb.in.base + (size_t)b * jb.in.batch_stride + (size_t)j * jb.in.limb_stride);
    i128 *gout = reinterpret_cast<i128 *>(jb.out.base + (size_t)b * jb.out.batch_stride + (size_t)j * jb.out.limb_stride);
    uint32_t *sm = smem + slot * 4 * G::PLANE;
    constexpr int n = G::NB;

    if (L > G::R0) {
        inv_bottom<0, L>(sm + 0 * G::PLANE, gin + 0 * n, tw + 0 * n, t, active);
        inv_bottom<1, L>(sm + 1 * G::PLANE, gin + 1 * n, tw + 1 * n, t, active);
        inv_bottom<2, L>(sm + 2 * G::PLANE, gin + 2 * n, tw + 2 * n, t, active);
        inv_bottom<3, L>(sm + 3 * G::PLANE, gin + 3 * n, tw + 3 * n, t, active);
        __syncthreads();
        InvMid<L, (L - 6 >= G::R0) ? L - 6 : -1>::run(sm, tw, n, t);
    }
    u128 acc[8];
#pragma unroll
    for (int jj = 0; jj < 8; jj++) acc[jj] = 0;
    inv_top<0, L>(sm + 0 * G::PLANE, gin + 0 * n, tw + 0 * n, t, active, nc, acc);
    inv_top<1, L>(sm + 1 * G::PLANE, gin + 1 * n, tw + 1 * n, t, active, nc, acc);
    inv_top<2, L>(sm + 2 * G::PLANE, gin + 2 * n, tw + 2 * n, t, active, nc, acc);
    inv_top<3, L>(sm + 3 * G::PLANE, gin + 3 * n, tw + 3 * n, t, active, nc, acc);
    if (L == G::R0) __syncthreads(); // n == 8, in-place safety: every thread has read before anyone writes
    if (active) {
#pragma unroll
        for (int jj = 0; jj < 8; jj++) gout[t + jj * G::T] = crt_finish(acc[jj]);
    }
}

// ---------------------------------------------------------------------------------------------- n > 8192 (two kernels)
// n = 8 * NB: the three top levels run as a global radix-8 pass (stride n/8, fully coalesced), the remaining log2(NB) levels as
// eight independent size-NB sub-transforms in shared memory whose block twiddles start at root = 8 + sub-block index.
struct TopJobs {
    LimbSet in, out;
    int jobs_per_batch, total_jobs, n;
    long long and_mask;
};
__global__ void __launch_bounds__(256) ntt120_fwd_top8_kernel(TopJobs jb, const uint2 *__restrict__ tw) {
    const int n = jb.n, s = n >> 3;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= s) return;
    const int job = blockIdx.y, b = job / jb.jobs_per_batch, j = job % jb.jobs_per_batch;
    const long long *gin = reinterpret_cast<const long long *>(jb.in.base + (size_t)b * jb.in.batch_stride + (size_t)j * jb.in.limb_stride);
    uint32_t *gout = reinterpret_cast<uint32_t *>(jb.out.base + (size_t)b * jb.out.batch_stride + (size_t)j * jb.out.limb_stride);
    long long v[8];
#pragma unroll
    for (int jj = 0; jj < 8; jj++) v[jj] = __ldg(gin + i + jj * s) & jb.and_mask;
    uint32_t x[8];
#define TOP_FWD(K)                                                   \
    _Pragma("unroll") for (int jj = 0; jj < 8; jj++) x[jj] = from_i64<K>(v[jj]); \
    ct_radix8<K, 3>(x, tw + (size_t)K * n, 1u);                      \
    _Pragma("unroll") for (int jj = 0; jj < 8; jj++) gout[(size_t)K * n + i + jj * s] = x[jj];
    TOP_FWD(0) TOP_FWD(1) TOP_FWD(2) TOP_FWD(3)
#undef TOP_FWD
}

// sub-transform, forward: in place on the lazy residues left by the top pass; job = limb * 8 + sub-block
template <int L> __global__ void __launch_bounds__(Geo<L>::T) ntt120_fwd_sub_kernel(LimbSet out, int jobs_per_batch, int n_total,
                                                                                   const uint2 *__restrict__ tw) {
    typedef Geo<L> G;
    extern __shared__ __align__(16) uint32_t smem[];
    const int t = threadIdx.x;
    const int sb = blockIdx.x & 7, limb = blockIdx.x >> 3;
    const int b = limb / jobs_per_batch, j = limb % jobs_per_batch;
    uint32_t *g = reinterpret_cast<uint32_t *>(out.base + (size_t)b * out.batch_stride + (size_t)j * out.limb_stride) + (size_t)sb * G::NB;
    const uint32_t root = 8u | (uint32_t)sb;
#define SUB_FWD(K)                                                                                   \
    {                                                                                                \
        uint32_t x[8];                                                                               \
        _Pragma("unroll") for (int jj = 0; jj < 8; jj++) x[jj] = g[(size_t)K * n_total + t + jj * G::T]; \
        ct_radix8<K, G::R0>(x, tw + (size_t)K * n_total, root);                                      \
        _Pragma("unroll") for (int jj = 0; jj < 8; jj++) smem[K * G::PLANE + PAD(t + jj * G::T)] = x[jj]; \
    }
    SUB_FWD(0) SUB_FWD(1) SUB_FWD(2) SUB_FWD(3)
#undef SUB_FWD
    __syncthreads();
    FwdMid<L, G::R0>::run(smem, g, tw, n_total, t, true, root);
}

// sub-transform, inverse: reads canonical residues, writes lazy [0, 2q) residues to `out` (scratch), same plane layout
template <int L> __global__ void __launch_bounds__(Geo<L>::T) ntt120_inv_sub_kernel(LimbSet in, LimbSet out, int jobs_per_batch, int n_total,
                                                                                   const uint2 *__restrict__ tw) {
    typedef Geo<L> G;
    extern __shared__ __align__(16) uint32_t smem[];
    const int t = threadIdx.x;
    const int sb = blockIdx.x & 7, limb = blockIdx.x >> 3;
    const int b = limb / jobs_per_batch, j = limb % jobs_per_batch;
    const uint32_t *gi = reinterpret_cast<const uint32_t *>(in.base + (size_t)b * in.batch_stride + (size_t)j * in.limb_stride) + (size_t)sb * G::NB;
    uint32_t *go = reinterpret_cast<uint32_t *>(out.base + (size_t)b * out.batch_stride + (size_t)j * out.limb_stride) + (size_t)sb * G::NB;
    const uint32_t root = 8u | (uint32_t)sb;
    inv_bottom<0, L>(smem + 0 * G::PLANE, gi + (size_t)0 * n_total, tw + (size_t)0 * n_total, t, true, root);
    inv_bottom<1, L>(smem + 1 * G::PLANE, gi + (size_t)1 * n_total, tw + (size_t)1 * n_total, t, true, root);
    inv_bottom<2, L>(smem + 2 * G::PLANE, gi + (size_t)2 * n_total, tw + (size_t)2 * n_total, t, true, root);
    inv_bottom<3, L>(smem + 3 * G::PLANE, gi + (size_t)3 * n_total, tw + (size_t)3 * n_total, t, true, root);
    __syncthreads();
    InvMid<L, (L - 6 >= G::R0) ? L - 6 : -1>::run(smem, tw, n_total, t, root);
#define SUB_INV(K)                                                                                   \
    {                                                                                                \
        uint32_t x[8];                                                                               \
        _Pragma("unroll") for (int jj = 0; jj < 8; jj++) x[jj] = smem[K * G::PLANE + PAD(t + jj * G::T)]; \
        gs_radix8<K, G::R0>(x, tw + (size_t)K * n_total, root);                                      \
        _Pragma("unroll") for (int jj = 0; jj < 8; jj++) go[(size_t)K * n_total + t + jj * G::T] = x[jj]; \
    }
    SUB_INV(0) SUB_INV(1) SUB_INV(2) SUB_INV(3)
#undef SUB_INV
}

// top three inverse levels + CRT, out of place (scratch planes -> i128 limb)
__global__ void __launch_bounds__(256) ntt120_inv_top8_kernel(TopJobs jb, const uint2 *__restrict__ tw, Ntt120Consts nc) {
    const int n = jb.n, s = n >> 3;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= s) return;
    const int job = blockIdx.y, b = job / jb.jobs_per_batch, j = job % jb.jobs_per_batch;
    const uint32_t *gin = reinterpret_cast<const uint32_t *>(jb.in.base + (size_t)b * jb.in.batch_stride + (size_t)j * jb.in.limb_stride);
    i128 *gout = reinterpret_cast<i128 *>(jb.out.base + (size_t)b * jb.out.batch_stride + (size_t)j * jb.out.limb_stride);
    u128 acc[8];
#pragma unroll
    for (int jj = 0; jj < 8; jj++) acc[jj] = 0;
#define TOP_INV(K)                                                                                    \
    {                                                                                                 \
        constexpr uint32_t q = Prime<K>::q;                                                           \
        uint32_t x[8];                                                                                \
        _Pragma("unroll") for (int jj = 0; jj < 8; jj++) x[jj] = __ldg(gin + (size_t)K * n + i + jj * s); \
        gs_radix8<K, 3>(x, tw + (size_t)K * n, 1u);                                                   \
        const unsigned long long mlo = c_crt.m_lo[K], mhi = c_crt.m_hi[K];                            \
        _Pragma("unroll") for (int jj = 0; jj < 8; jj++) {                                            \
            uint32_t tk = csub(mul_shoup(x[jj], nc.crt_ninv[K], nc.crt_ninv_sh[K], q), q);            \
            acc[jj] += (u128)tk * mlo + ((u128)((unsigned long long)tk * mhi) << 64);                 \
        }                                                                                             \
    }
    TOP_INV(0) TOP_INV(1) TOP_INV(2) TOP_INV(3)
#undef TOP_INV
#pragma unroll
    for (int jj = 0; jj < 8; jj++) gout[i + jj * s] = crt_finish(acc[jj]);
}

// ---------------------------------------------------------------------------------------------- fused back end
// One CTA per (ciphertext, output column): for every limb from the least significant one
//     vmp on the fly (sum_r a[r] * M[r][c], loaded straight into the bottom pass)  ->  inverse NTT  ->  CRT
//     -> (+ small, the body column of the key-switch input)  ->  base-2^K carry step with the carry kept in registers
// so that res_dft / res_big / add_small / normalize never touch HBM.  Restates, per coefficient and limb by limb, the sequence
// vmp_apply_dft_to_dft + vec_znx_idft_apply_consume + vec_znx_big_add_small_assign + vec_znx_big_normalize of
// poulpy-core/src/keyswitching/glwe.rs:229-237,106-108 and external_product/glwe.rs:231-234,270,138-140 (same-base2k path of
// poulpy-cpu-ref/src/reference/ntt120/vec_znx_big.rs:367-446).
struct FusedArgs {
    const char *a_dft;  uint64_t a_bs;      // R polys (16n B each) per ciphertext
    const char *pmat;   uint64_t pmat_bs;   // [R][C] polys; item b's matrix at pmat + b * pmat_bs (0 = one matrix for the batch)
    const char *small;  uint64_t small_bs;  uint64_t small_limb_stride; int small_size; // i64 limbs added to column 0 (or null)
    char *res;          uint64_t res_bs;    uint64_t res_limb_stride;                    // i64 output, column c at + c*n*8
    int R, C, cols_out;
    int direct;         // 1: a_dft already holds the C product polys (limb-major, column-minor): no matrix, straight to the inverse transform
    int small_all_cols; // 1: `small` is added on every output column (column c at + c*n words), not only on column 0
    // same-base2k normalisation plan (big = C / cols_out limbs)
    int K, lsh, res_size, a_size, a_start, a_end, res_start, res_end;
};

__device__ __forceinline__ i128 nd_get_digit(int k, i128 x) { return (i128)((u128)x << (128 - k)) >> (128 - k); }
__device__ __forceinline__ i128 nd_get_carry(int k, i128 x, i128 d) { return (i128)((u128)x - (u128)d) >> k; }

// x[i] = sum_r a[r][8t+i] * m[r][8t+i] mod q, in [0, 2q)
template <int K> __device__ __forceinline__ void vmp_rows8(uint32_t (&x)[8], const uint32_t *__restrict__ a, size_t a_stride,
                                                           const uint32_t *__restrict__ mm, size_t m_stride, int R) {
    constexpr uint32_t q = Prime<K>::q;
    constexpr uint32_t c32 = (uint32_t)((1ull << 32) % q);
    constexpr uint32_t c32s = (uint32_t)(((unsigned long long)c32 << 32) / q);
    unsigned long long acc[8];
#pragma unroll
    for (int i = 0; i < 8; i++) acc[i] = 0;
    if (R == 3) { // the key-switch bench shape: all 12 loads in flight before the first MAC
        uint4 a0[3], a1[3], m0[3], m1[3];
#pragma unroll
        for (int r = 0; r < 3; r++) {
            const uint4 *pa = reinterpret_cast<const uint4 *>(a + (size_t)r * a_stride);
            const uint4 *pm = reinterpret_cast<const uint4 *>(mm + (size_t)r * m_stride);
            a0[r] = __ldg(pa); a1[r] = __ldg(pa + 1); m0[r] = __ldg(pm); m1[r] = __ldg(pm + 1);
        }
#pragma unroll
        for (int r = 0; r < 3; r++) {
            acc[0] += (unsigned long long)a0[r].x * m0[r].x; acc[1] += (unsigned long long)a0[r].y * m0[r].y;
            acc[2] += (unsigned long long)a0[r].z * m0[r].z; acc[3] += (unsigned long long)a0[r].w * m0[r].w;
            acc[4] += (unsigned long long)a1[r].x * m1[r].x; acc[5] += (unsigned long long)a1[r].y * m1[r].y;
            acc[6] += (unsigned long long)a1[r].z * m1[r].z; acc[7] += (unsigned long long)a1[r].w * m1[r].w;
        }
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const uint32_t hi = (uint32_t)(acc[i] >> 32), lo = (uint32_t)acc[i];
            acc[i] = csub(mul_shoup(hi, c32, c32s, q) + (lo - (lo >> 30) * q), 2 * q);
        }
    } else
    for (int r0 = 0; r0 < R; r0 += 16) {
        const int r1 = min(r0 + 16, R);
#pragma unroll 2
        for (int r = r0; r < r1; r++) {
            const uint4 *pa = reinterpret_cast<const uint4 *>(a + (size_t)r * a_stride);
            const uint4 *pm = reinterpret_cast<const uint4 *>(mm + (size_t)r * m_stride);
            const uint4 a0 = __ldg(pa), a1 = __ldg(pa + 1), m0 = __ldg(pm), m1 = __ldg(pm + 1);
            acc[0] += (unsigned long long)a0.x * m0.x; acc[1] += (unsigned long long)a0.y * m0.y;
            acc[2] += (unsigned long long)a0.z * m0.z; acc[3] += (unsigned long long)a0.w * m0.w;
            acc[4] += (unsigned long long)a1.x * m1.x; acc[5] += (unsigned long long)a1.y * m1.y;
            acc[6] += (unsigned long long)a1.z * m1.z; acc[7] += (unsigned long long)a1.w * m1.w;
        }
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const uint32_t hi = (uint32_t)(acc[i] >> 32), lo = (uint32_t)acc[i];
            const uint32_t r = csub(mul_shoup(hi, c32, c32s, q) + (lo - (lo >> 30) * q), 2 * q);
            acc[i] = r;
        }
    }
#pragma unroll
    for (int i = 0; i < 8; i++) x[i] = (uint32_t)acc[i];
}

// direct mode: the residues of one product poly come straight from global memory
template <int K, int L> __device__ __forceinline__ void fused_bottom_direct(uint32_t *__restrict__ plane, const uint32_t *__restrict__ src,
                                                                           const uint2 *__restrict__ tw, int t) {
    const uint4 *p4 = reinterpret_cast<const uint4 *>(src + 8 * t);
    const uint4 u0 = __ldg(p4), u1 = __ldg(p4 + 1);
    uint32_t x[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
    inv_bottom_core<K, L>(x, plane, tw, t);
}
template <int K, int L> __device__ __forceinline__ void fused_bottom(uint32_t *__restrict__ plane, const uint32_t *__restrict__ a,
                                                                    size_t a_stride, const uint32_t *__restrict__ mm, size_t m_stride,
                                                                    int R, const uint2 *__restrict__ tw, int t) {
    uint32_t x[8];
    vmp_rows8<K>(x, a + 8 * t, a_stride, mm + 8 * t, m_stride, R);
    inv_bottom_core<K, L>(x, plane, tw, t);
}

// top pass of the fused kernel for one prime: R0 levels, scale by CRT_k / n, leave the canonical residue in the plane
template <int K, int L> __device__ __forceinline__ void fused_top(uint32_t *__restrict__ plane, const uint2 *__restrict__ tw, int t,
                                                                 const Ntt120Consts &nc) {
    typedef Geo<L> G;
    constexpr uint32_t q = Prime<K>::q;
    uint32_t x[8];
#pragma unroll
    for (int j = 0; j < 8; j++) x[j] = plane[PAD(t + j * G::T)];
    gs_radix8<K, G::R0>(x, tw, 1u);
#pragma unroll
    for (int j = 0; j < 8; j++) plane[PAD(t + j * G::T)] = csub(mul_shoup(x[j], nc.crt_ninv[K], nc.crt_ninv_sh[K], q), q);
}

// Persistent CTAs (two per SM): each loops over (ciphertext, column) work items; the per-coefficient i128 carries of the
// normalisation live in a small L2-resident scratch indexed by CTA (16 B per coefficient), so the kernel fits in 64 registers.
template <int L> __global__ void __launch_bounds__(Geo<L>::T, 2) ntt120_fused_back_kernel(FusedArgs p, const uint2 *__restrict__ tw,
                                                                                         Ntt120Consts nc, int total_work,
                                                                                         i128 *__restrict__ carry_scratch,
                                                                                         const int *__restrict__ skip, int skip_list) {
    typedef Geo<L> G;
    static_assert(L > G::R0, "fused path needs at least two passes");
    extern __shared__ __align__(16) uint32_t smem[];
    constexpr int n = G::NB;
    const int t = threadIdx.x;
    const size_t poly = (size_t)4 * n; // u32 words per poly
    const size_t res_ls = p.res_limb_stride / 8, small_ls = p.small_limb_stride / 8;
    const int K = p.K, lsh = p.lsh, w = lsh == 0 ? K : K - lsh;
    i128 *carry = carry_scratch + (size_t)blockIdx.x * n;
    if (skip && skip_list && __ldg(skip + total_work / p.cols_out) == 0) return; // the gadget kernel flagged nothing (see NttJobs::skip_list)
    const size_t m_stride = (size_t)p.C * poly;
    const u128 M0 = ((u128)c_crt.m_hi[0] << 64) | c_crt.m_lo[0], M1 = ((u128)c_crt.m_hi[1] << 64) | c_crt.m_lo[1];
    const u128 M2 = ((u128)c_crt.m_hi[2] << 64) | c_crt.m_lo[2], M3 = ((u128)c_crt.m_hi[3] << 64) | c_crt.m_lo[3];

    for (int work = blockIdx.x; work < total_work; work += gridDim.x) {
        const int col = work % p.cols_out;
        const size_t b = work / p.cols_out;
        if (skip && skip[b]) continue; // handled by the collapsed-key kernel
        const uint32_t *a = reinterpret_cast<const uint32_t *>(p.a_dft + b * p.a_bs);
        const uint32_t *pm = reinterpret_cast<const uint32_t *>(p.pmat + b * p.pmat_bs);
        long long *res = reinterpret_cast<long long *>(p.res + b * p.res_bs) + (size_t)col * n;
        const long long *small = (p.small && (col == 0 || p.small_all_cols))
                                     ? reinterpret_cast<const long long *>(p.small + b * p.small_bs) + (p.small_all_cols ? (size_t)col * n : 0)
                                     : nullptr;

        for (int j = p.res_start; j < p.res_size; j++) {
#pragma unroll
            for (int jj = 0; jj < 8; jj++) res[(size_t)j * res_ls + t + jj * G::T] = 0;
        }
        for (int j = p.a_size - 1; j >= p.a_end; j--) {
            if (p.direct) {
                const uint32_t *src = a + ((size_t)j * p.cols_out + col) * poly;
                fused_bottom_direct<0, L>(smem + 0 * G::PLANE, src + 0 * n, tw + 0 * n, t);
                fused_bottom_direct<1, L>(smem + 1 * G::PLANE, src + 1 * n, tw + 1 * n, t);
                fused_bottom_direct<2, L>(smem + 2 * G::PLANE, src + 2 * n, tw + 2 * n, t);
                fused_bottom_direct<3, L>(smem + 3 * G::PLANE, src + 3 * n, tw + 3 * n, t);
            } else {
                const uint32_t *mc = pm + ((size_t)j * p.cols_out + col) * poly;
                fused_bottom<0, L>(smem + 0 * G::PLANE, a + 0 * n, poly, mc + 0 * n, m_stride, p.R, tw + 0 * n, t);
                fused_bottom<1, L>(smem + 1 * G::PLANE, a + 1 * n, poly, mc + 1 * n, m_stride, p.R, tw + 1 * n, t);
                fused_bottom<2, L>(smem + 2 * G::PLANE, a + 2 * n, poly, mc + 2 * n, m_stride, p.R, tw + 2 * n, t);
                fused_bottom<3, L>(smem + 3 * G::PLANE, a + 3 * n, poly, mc + 3 * n, m_stride, p.R, tw + 3 * n, t);
            }
            __syncthreads();
            InvMid<L, (L - 6 >= G::R0) ? L - 6 : -1>::run(smem, tw, n, t);
            fused_top<0, L>(smem + 0 * G::PLANE, tw + 0 * n, t, nc);
            fused_top<1, L>(smem + 1 * G::PLANE, tw + 1 * n, t, nc);
            fused_top<2, L>(smem + 2 * G::PLANE, tw + 2 * n, t, nc);
            fused_top<3, L>(smem + 3 * G::PLANE, tw + 3 * n, t, nc);
            // the residues of coefficient idx = t + jj*T sit at thread-private plane slots: no barrier needed here
            const bool carry_only = j >= p.a_start;
            const bool first = j == p.a_size - 1 && carry_only;
            const bool have_carry = j != p.a_size - 1;
            const int res_limb = j - p.a_start + p.res_start;
            const bool add_small = small && j < p.small_size;
#pragma unroll 2
            for (int jj = 0; jj < 8; jj++) {
                const int idx = t + jj * G::T;
                const int pi = PAD(idx);
                const u128 acc = (u128)smem[pi] * M0 + (u128)smem[G::PLANE + pi] * M1 + (u128)smem[2 * G::PLANE + pi] * M2 +
                                 (u128)smem[3 * G::PLANE + pi] * M3;
                i128 v = crt_finish(acc);
                if (add_small) v = (i128)((u128)v + (u128)(i128)small[(size_t)j * small_ls + idx]);
                if (lsh == 0) {
                    // Same-base2k step without an intra-limb shift collapses to one digit extraction of t = v + carry_in:
                    //   digit_K(digit_K(v) + c) = digit_K(t)   and   carry(v) + carry(digit_K(v) + c) = (t + 2^(K-1)) >> K
                    // (vec_znx_big.rs:120-133 with lsh == 0; t cannot overflow: |v| < 2^119, |c| < 2^(120-K)).
                    const i128 tt = (first || !have_carry) ? v : (i128)((u128)v + (u128)carry[idx]);
                    const long long out = ((long long)(unsigned long long)tt << (64 - K)) >> (64 - K);
                    carry[idx] = (i128)((u128)tt + ((u128)1 << (K - 1))) >> K;
                    if (!carry_only) res[(size_t)res_limb * res_ls + idx] = out;
                } else {
                    const i128 d = nd_get_digit(w, v);
                    const i128 co = nd_get_carry(w, v, d);
                    if (first) {
                        carry[idx] = co;
                    } else {
                        const i128 cin = have_carry ? carry[idx] : (i128)0;
                        const i128 s = (i128)(((u128)d << lsh) + (u128)cin);
                        const i128 out = nd_get_digit(K, s);
                        carry[idx] = (i128)((u128)co + (u128)nd_get_carry(K, s, out));
                        if (!carry_only) res[(size_t)res_limb * res_ls + idx] = (long long)out;
                    }
                }
            }
            __syncthreads(); // planes are rewritten by the next limb's bottom pass
        }
        const bool any = p.a_size - 1 >= p.a_end;
        for (int j = 0; j < p.res_end; j++) {
#pragma unroll
            for (int jj = 0; jj < 8; jj++) {
                const int idx = t + jj * G::T;
                const i128 c = any ? carry[idx] : (i128)0;
                const i128 out = nd_get_digit(K, c);
                res[(size_t)(p.res_end - j - 1) * res_ls + idx] = (long long)out;
                carry[idx] = nd_get_carry(K, c, out);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------- collapsed-key fast path
// The S output limbs of a gadget product are the base-2^K digits of ONE integer polynomial
//     V = sum_j 2^((S-1-j)K) * v_j ,  v_j = sum_r a_r (*) M[r][j]   (negacyclic convolutions over Z)
// because vec_znx_big_normalize (same base2k, offset 0) is exactly the balanced base-2^K expansion of V
// (reference/ntt120/vec_znx_big.rs:367-446: out_j = digit(v_j + c_{j+1}), c_j = (v_j + c_{j+1} - out_j) >> K).  By linearity of the
// NTT, V = sum_r a_r (*) M'[r] with the "collapsed" key M'[r] = sum_j 2^((S-1-j)K) M[r][j] (mod Q, computed in the DFT domain), so
// ONE inverse transform per output column replaces S of them.  This is bit-identical to the per-limb route iff every v_j and V
// stay inside (-Q/2, Q/2); that is decided per ciphertext on the device from max|a| and max|key coefficient| (both measured, not
// assumed), and ciphertexts that fail the bound take the per-limb kernel instead.
struct CollapseArgs {
    const char *pmat;
    char *out;
    int n4, R, C, cols_out, S;
    uint32_t c[32][4]; // 2^((S-1-j)K) mod Q[k]
};
__global__ void __launch_bounds__(256) ntt120_collapse_key_kernel(CollapseArgs p) {
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= 4u * p.n4) return;
    const int k = u / p.n4;
    const PrimeRt pr(k);
    const int r = blockIdx.y / p.cols_out, col = blockIdx.y % p.cols_out;
    const size_t poly = (size_t)4 * p.n4;
    const uint4 *src = reinterpret_cast<const uint4 *>(p.pmat) + ((size_t)r * p.C + col) * poly + u;
    unsigned long long acc[4] = {0, 0, 0, 0};
    for (int j0 = 0; j0 < p.S; j0 += 16) {
        const int j1 = min(j0 + 16, p.S);
        for (int j = j0; j < j1; j++) {
            const uint4 v = __ldg(src + (size_t)j * p.cols_out * poly);
            const unsigned long long cj = p.c[j][k];
            acc[0] += v.x * cj; acc[1] += v.y * cj; acc[2] += v.z * cj; acc[3] += v.w * cj;
        }
#pragma unroll
        for (int i = 0; i < 4; i++) acc[i] = pr.reduce(acc[i]);
    }
    reinterpret_cast<uint4 *>(p.out)[((size_t)r * p.cols_out + col) * poly + u] =
        make_uint4((uint32_t)acc[0], (uint32_t)acc[1], (uint32_t)acc[2], (uint32_t)acc[3]);
}

__device__ __forceinline__ int bitlen_u128(u128 x) {
    const unsigned long long hi = (unsigned long long)(x >> 64), lo = (unsigned long long)x;
    return hi ? 128 - __clzll((long long)hi) : (lo ? 64 - __clzll((long long)lo) : 0);
}
// bits[0] = max bit length of |x| over `count` i128 values
__global__ void __launch_bounds__(256) max_bits_i128_kernel(const i128 *__restrict__ x, size_t count, int *__restrict__ bits) {
    int mx = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
        const i128 v = x[i];
        mx = max(mx, bitlen_u128(v < 0 ? (u128)0 - (u128)v : (u128)v));
    }
    for (int o = 16; o; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) atomicMax(bits, mx);
}
// per ciphertext: ok[b] = 1 iff the integers behind the collapsed product provably stay below 2^118 in magnitude
struct GuardArgs {
    const char *a; uint64_t a_bs; uint64_t words; // i64 words per ciphertext (all columns and limbs of the GLWE)
    const int *key_bits;
    int base_bits; // ceil(log2(R * n)) + (S - 1) * K + 3
    int *ok;
};
__global__ void __launch_bounds__(256) ntt120_collapse_guard_kernel(GuardArgs p) {
    const long long *a = reinterpret_cast<const long long *>(p.a + (size_t)blockIdx.x * p.a_bs);
    int mx = 0;
    for (uint64_t i = threadIdx.x; i < p.words; i += blockDim.x) {
        const long long v = a[i];
        const unsigned long long m = v < 0 ? 0ull - (unsigned long long)v : (unsigned long long)v;
        mx = max(mx, m ? 64 - __clzll((long long)m) : 0);
    }
    __shared__ int smx;
    if (threadIdx.x == 0) smx = 0;
    __syncthreads();
    for (int o = 16; o; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) atomicMax(&smx, mx);
    __syncthreads();
    if (threadIdx.x == 0) p.ok[blockIdx.x] = (smx + *p.key_bits + p.base_bits <= 118) ? 1 : 0;
}

template <int L> __global__ void __launch_bounds__(Geo<L>::T, 2) ntt120_collapsed_back_kernel(FusedArgs p, const uint2 *__restrict__ tw,
                                                                                            Ntt120Consts nc, int total_work,
                                                                                            const int *__restrict__ ok) {
    typedef Geo<L> G;
    extern __shared__ __align__(16) uint32_t smem[];
    constexpr int n = G::NB;
    const int t = threadIdx.x;
    const uint32_t *pm = reinterpret_cast<const uint32_t *>(p.pmat); // collapsed key: [R][cols_out] polys
    const size_t poly = (size_t)4 * n;
    const size_t res_ls = p.res_limb_stride / 8, small_ls = p.small_limb_stride / 8;
    const int K = p.K, S = p.a_size;
    const size_t m_stride = (size_t)p.cols_out * poly;
    const u128 M0 = ((u128)c_crt.m_hi[0] << 64) | c_crt.m_lo[0], M1 = ((u128)c_crt.m_hi[1] << 64) | c_crt.m_lo[1];
    const u128 M2 = ((u128)c_crt.m_hi[2] << 64) | c_crt.m_lo[2], M3 = ((u128)c_crt.m_hi[3] << 64) | c_crt.m_lo[3];
    for (int work = blockIdx.x; work < total_work; work += gridDim.x) {
        const int col = work % p.cols_out;
        const size_t b = work / p.cols_out;
        if (!ok[b]) continue; // uniform per CTA: this ciphertext is handled by the per-limb kernel
        const uint32_t *a = reinterpret_cast<const uint32_t *>(p.a_dft + b * p.a_bs);
        long long *res = reinterpret_cast<long long *>(p.res + b * p.res_bs) + (size_t)col * n;
        const long long *small = (p.small && col == 0) ? reinterpret_cast<const long long *>(p.small + b * p.small_bs) : nullptr;
        const uint32_t *mc = pm + (size_t)col * poly;
        fused_bottom<0, L>(smem + 0 * G::PLANE, a + 0 * n, poly, mc + 0 * n, m_stride, p.R, tw + 0 * n, t);
        fused_bottom<1, L>(smem + 1 * G::PLANE, a + 1 * n, poly, mc + 1 * n, m_stride, p.R, tw + 1 * n, t);
        fused_bottom<2, L>(smem + 2 * G::PLANE, a + 2 * n, poly, mc + 2 * n, m_stride, p.R, tw + 2 * n, t);
        fused_bottom<3, L>(smem + 3 * G::PLANE, a + 3 * n, poly, mc + 3 * n, m_stride, p.R, tw + 3 * n, t);
        __syncthreads();
        InvMid<L, (L - 6 >= G::R0) ? L - 6 : -1>::run(smem, tw, n, t);
        fused_top<0, L>(smem + 0 * G::PLANE, tw + 0 * n, t, nc);
        fused_top<1, L>(smem + 1 * G::PLANE, tw + 1 * n, t, nc);
        fused_top<2, L>(smem + 2 * G::PLANE, tw + 2 * n, t, nc);
        fused_top<3, L>(smem + 3 * G::PLANE, tw + 3 * n, t, nc);
#pragma unroll 2
        for (int jj = 0; jj < 8; jj++) {
            const int idx = t + jj * G::T;
            const int pi = PAD(idx);
            const u128 acc = (u128)smem[pi] * M0 + (u128)smem[G::PLANE + pi] * M1 + (u128)smem[2 * G::PLANE + pi] * M2 +
                             (u128)smem[3 * G::PLANE + pi] * M3;
            i128 v = crt_finish(acc);
            if (small) {
                for (int j = 0; j < p.small_size; j++)
                    v = (i128)((u128)v + ((u128)(i128)small[(size_t)j * small_ls + idx] << ((S - 1 - j) * K)));
            }
            for (int j = S - 1; j >= 0; j--) { // balanced base-2^K digits, least significant limb first
                const long long out = ((long long)(unsigned long long)v << (64 - K)) >> (64 - K);
                v = (i128)((u128)v + ((u128)1 << (K - 1))) >> K;
                if (j < p.a_start) res[(size_t)(j - p.a_start + p.res_start) * res_ls + idx] = out;
            }
        }
        for (int j = p.res_start; j < p.res_size; j++) {
#pragma unroll
            for (int jj = 0; jj < 8; jj++) res[(size_t)j * res_ls + t + jj * G::T] = 0;
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------- host side
static uint32_t modpow(uint32_t x, uint64_t e, uint32_t q) {
    uint64_t r = 1, b = x;
    while (e) {
        if (e & 1) r = r * b % q;
        b = b * b % q;
        e >>= 1;
    }
    return (uint32_t)r;
}

int ntt120_module_init(pgb_module *m) {
    const uint64_t n = m->n;
    // block-twiddle exponents: E[1] = n/2, E[2i] = E[i]/2, E[2i+1] = E[i]/2 + n/2  (W[i] = psi^E[i], psi = 2n-th root)
    uint64_t *E = (uint64_t *)malloc(sizeof(uint64_t) * n);
    if (n >= 2) E[1] = n / 2;
    for (uint64_t i = 1; 2 * i + 1 < n; i++) {
        E[2 * i] = E[i] / 2;
        E[2 * i + 1] = E[i] / 2 + n / 2;
    }
    uint2 *hf = (uint2 *)calloc(4 * n, sizeof(uint2)), *hi = (uint2 *)calloc(4 * n, sizeof(uint2));
    for (int k = 0; k < 4; k++) {
        uint32_t q = qk(k);
        uint32_t psi = modpow(OMEGA[k], (1u << 16) / n, q); // ntt.rs:164-167
        for (uint64_t i = 1; i < n; i++) {
            uint32_t w = modpow(psi, E[i], q);
            uint32_t wi = modpow(psi, 2 * n - E[i], q);
            hf[k * n + i] = make_uint2(w, (uint32_t)(((uint64_t)w << 32) / q));
            hi[k * n + i] = make_uint2(wi, (uint32_t)(((uint64_t)wi << 32) / q));
            if (i < 16) {
                m->tw_top_f[k][i] = hf[k * n + i];
                m->tw_top_i[k][i] = hi[k * n + i];
            }
        }
        uint32_t ninv = modpow((uint32_t)(n % q), q - 2, q);
        uint32_t c = (uint32_t)((uint64_t)CRT_CST[k] * ninv % q);
        m->nc.crt_ninv[k] = c;
        m->nc.crt_ninv_sh[k] = (uint32_t)(((uint64_t)c << 32) / q);
    }
    free(E);
    PGB_CHECK_CUDA(cudaMalloc(&m->ntt_fwd, 4 * n * sizeof(uint2)));
    PGB_CHECK_CUDA(cudaMalloc(&m->ntt_inv, 4 * n * sizeof(uint2)));
    PGB_CHECK_CUDA(cudaMemcpy(m->ntt_fwd, hf, 4 * n * sizeof(uint2), cudaMemcpyHostToDevice));
    PGB_CHECK_CUDA(cudaMemcpy(m->ntt_inv, hi, 4 * n * sizeof(uint2), cudaMemcpyHostToDevice));
    m->ntt_last16_f = m->ntt_last16_i = nullptr;
    if (n >= 32) { // per-thread tables of the last radix-16 pass (common.cuh)
        const uint64_t T = n / 16;
        uint4 *lf = (uint4 *)calloc(4 * 8 * T, sizeof(uint4)), *li = (uint4 *)calloc(4 * 8 * T, sizeof(uint4));
        for (int k = 0; k < 4; k++)
            for (uint64_t t = 0; t < T; t++) {
                const uint64_t node = T + t;
                for (int dir = 0; dir < 2; dir++) {
                    const uint2 *src = (dir ? hi : hf) + (size_t)k * n;
                    uint4 *dst = (dir ? li : lf) + (size_t)k * 8 * T + t;
                    dst[0 * T] = make_uint4(src[node].x, src[node].y, 0u, 0u);
                    dst[1 * T] = make_uint4(src[2 * node].x, src[2 * node].y, src[2 * node + 1].x, src[2 * node + 1].y);
                    for (int j = 0; j < 2; j++)
                        dst[(2 + j) * T] = make_uint4(src[4 * node + 2 * j].x, src[4 * node + 2 * j].y, src[4 * node + 2 * j + 1].x, src[4 * node + 2 * j + 1].y);
                    for (int j = 0; j < 4; j++)
                        dst[(4 + j) * T] = make_uint4(src[8 * node + 2 * j].x, src[8 * node + 2 * j].y, src[8 * node + 2 * j + 1].x, src[8 * node + 2 * j + 1].y);
                }
            }
        PGB_CHECK_CUDA(cudaMalloc(&m->ntt_last16_f, 4 * 8 * T * sizeof(uint4)));
        PGB_CHECK_CUDA(cudaMalloc(&m->ntt_last16_i, 4 * 8 * T * sizeof(uint4)));
        PGB_CHECK_CUDA(cudaMemcpy(m->ntt_last16_f, lf, 4 * 8 * T * sizeof(uint4), cudaMemcpyHostToDevice));
        PGB_CHECK_CUDA(cudaMemcpy(m->ntt_last16_i, li, 4 * 8 * T * sizeof(uint4), cudaMemcpyHostToDevice));
        free(lf);
        free(li);
    }
    free(hf);
    free(hi);
    CrtConsts cc;
    u128 Q = 1;
    for (int k = 0; k < 4; k++) Q *= qk(k);
    for (int k = 0; k < 4; k++) {
        u128 mk = Q / qk(k);
        cc.m_lo[k] = (unsigned long long)mk;
        cc.m_hi[k] = (unsigned long long)(mk >> 64);
    }
    cc.q_lo = (unsigned long long)Q;
    cc.q_hi = (unsigned long long)(Q >> 64);
    u128 H = (Q + 1) / 2;
    cc.half_lo = (unsigned long long)H;
    cc.half_hi = (unsigned long long)(H >> 64);
    PGB_CHECK_CUDA(cudaMemcpyToSymbol(c_crt, &cc, sizeof cc));
    return PGB_OK;
}

template <int L> static constexpr int lpc_for() { return Geo<L>::T >= 128 ? 1 : (128 / Geo<L>::T > 16 ? 16 : 128 / Geo<L>::T); }

template <int L> static int launch_fwd(pgb_module *m, const NttJobs &jb) {
    constexpr int LPC = lpc_for<L>();
    typedef Geo<L> G;
    size_t smem = (size_t)LPC * 4 * G::PLANE * sizeof(uint32_t);
    static bool attr_set_dev[32] = {}; // per device: function attributes are per device
    bool &attr_set = attr_set_dev[m->device & 31];
    if (!attr_set) {
        PGB_CHECK_CUDA(cudaFuncSetAttribute(ntt120_fwd_kernel<L, LPC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    int grid = (jb.total_jobs + LPC - 1) / LPC;
    if (jb.skip && jb.skip_list && grid > 296) grid = 296;
    { ProfScope _ps(m, PROF_DFT_FWD);
    ntt120_fwd_kernel<L, LPC><<<grid, G::T * LPC, smem, m->stream>>>(jb, m->ntt_fwd);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}
template <int L> static int launch_inv(pgb_module *m, const NttJobs &jb) {
    constexpr int LPC = lpc_for<L>();
    typedef Geo<L> G;
    size_t smem = (size_t)LPC * 4 * G::PLANE * sizeof(uint32_t);
    static bool attr_set_dev[32] = {}; // per device: function attributes are per device
    bool &attr_set = attr_set_dev[m->device & 31];
    if (!attr_set) {
        PGB_CHECK_CUDA(cudaFuncSetAttribute(ntt120_inv_kernel<L, LPC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    int grid = (jb.total_jobs + LPC - 1) / LPC;
    { ProfScope _ps(m, PROF_DFT_INV);
    ntt120_inv_kernel<L, LPC><<<grid, G::T * LPC, smem, m->stream>>>(jb, m->ntt_inv, m->nc);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

#define NTT_DISPATCH(fn)                         \
    switch (m->log_n) {                          \
    case 3: return fn<3>(m, jb);                 \
    case 4: return fn<4>(m, jb);                 \
    case 5: return fn<5>(m, jb);                 \
    case 6: return fn<6>(m, jb);                 \
    case 7: return fn<7>(m, jb);                 \
    case 8: return fn<8>(m, jb);                 \
    case 9: return fn<9>(m, jb);                 \
    case 10: return fn<10>(m, jb);               \
    case 11: return fn<11>(m, jb);               \
    case 12: return fn<12>(m, jb);               \
    case 13: return fn<13>(m, jb);               \
    default:                                     \
        pgb_set_error("NTT120: n = 2^%d not supported by the single-CTA path (16 <= n <= 65536)", m->log_n); \
        return PGB_ERR_UNSUPPORTED;              \
    }

template <int L> static int launch_fwd_sub(pgb_module *m, LimbSet out, int jobs_per_batch, int total_jobs) {
    typedef Geo<L> G;
    size_t smem = (size_t)4 * G::PLANE * sizeof(uint32_t);
    static bool attr_set_dev[32] = {}; // per device: function attributes are per device
    bool &attr_set = attr_set_dev[m->device & 31];
    if (!attr_set) {
        PGB_CHECK_CUDA(cudaFuncSetAttribute(ntt120_fwd_sub_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    { ProfScope _ps(m, PROF_DFT_FWD);
    ntt120_fwd_sub_kernel<L><<<total_jobs * 8, G::T, smem, m->stream>>>(out, jobs_per_batch, (int)m->n, m->ntt_fwd);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}
template <int L> static int launch_inv_sub(pgb_module *m, LimbSet in, LimbSet out, int jobs_per_batch, int total_jobs) {
    typedef Geo<L> G;
    size_t smem = (size_t)4 * G::PLANE * sizeof(uint32_t);
    static bool attr_set_dev[32] = {}; // per device: function attributes are per device
    bool &attr_set = attr_set_dev[m->device & 31];
    if (!attr_set) {
        PGB_CHECK_CUDA(cudaFuncSetAttribute(ntt120_inv_sub_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    { ProfScope _ps(m, PROF_DFT_INV);
    ntt120_inv_sub_kernel<L><<<total_jobs * 8, G::T, smem, m->stream>>>(in, out, jobs_per_batch, (int)m->n, m->ntt_inv);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

static int ntt120_forward_large(pgb_module *m, LimbSet in, LimbSet out, int jobs_per_batch, int batch, long long and_mask) {
    const int total = jobs_per_batch * batch;
    for (int j0 = 0; j0 < total; j0 += 32768) { // gridDim.y limit
        // jobs are (batch, limb) pairs in batch-major order: split on whole batches when there are many, else on limbs
        const int cnt = total - j0 < 32768 ? total - j0 : 32768;
        PGB_REQUIRE(j0 == 0 && cnt == total, "NTT120 large-n path: more than 32768 limbs per call (split the batch)");
        TopJobs tj = {in, out, jobs_per_batch, total, (int)m->n, and_mask};
        dim3 grid(((unsigned)(m->n >> 3) + 255) / 256, cnt);
        { ProfScope _ps(m, PROF_DFT_FWD);
        ntt120_fwd_top8_kernel<<<grid, 256, 0, m->stream>>>(tj, m->ntt_fwd);
        }
        PGB_CHECK_CUDA(cudaGetLastError());
    }
    switch (m->log_n) {
    case 14: return launch_fwd_sub<11>(m, out, jobs_per_batch, total);
    case 15: return launch_fwd_sub<12>(m, out, jobs_per_batch, total);
    default: return launch_fwd_sub<13>(m, out, jobs_per_batch, total);
    }
}

// scratch for the out-of-place inverse of the large-n path: lazy residue planes of the limbs in flight
static int ensure_carry_ws(pgb_module *m, size_t need) {
    if (m->carry_len >= need) return PGB_OK;
    if (m->carry_ws) {
        PGB_CHECK_CUDA(cudaStreamSynchronize(m->stream));
        cudaFree(m->carry_ws);
    }
    m->carry_ws = nullptr;
    m->carry_len = 0;
    PGB_CHECK_CUDA(cudaMalloc(&m->carry_ws, need));
    m->carry_len = need;
    return PGB_OK;
}

static int ntt120_inverse_large(pgb_module *m, LimbSet in, LimbSet out, int jobs_per_batch, int batch) {
    const size_t limb_bytes = (size_t)16 * m->n;
    // process whole batch items per chunk so that the (batch, limb) addressing of the LimbSets stays valid
    const size_t max_ws = (size_t)512 << 20;
    int chunk_b = (int)(max_ws / (limb_bytes * jobs_per_batch));
    if (chunk_b < 1) chunk_b = 1;
    if (chunk_b > batch) chunk_b = batch;
    PGB_TRY(ensure_carry_ws(m, (size_t)chunk_b * jobs_per_batch * limb_bytes));
    for (int b0 = 0; b0 < batch; b0 += chunk_b) {
        const int nb = batch - b0 < chunk_b ? batch - b0 : chunk_b;
        const int total = nb * jobs_per_batch;
        PGB_REQUIRE(total <= 32768, "NTT120 large-n path: more than 32768 limbs per chunk");
        LimbSet cin = in, cout = out;
        cin.base += (size_t)b0 * in.batch_stride;
        cout.base += (size_t)b0 * out.batch_stride;
        LimbSet ws = {(char *)m->carry_ws, limb_bytes, limb_bytes * jobs_per_batch};
        switch (m->log_n) {
        case 14: PGB_TRY(launch_inv_sub<11>(m, cin, ws, jobs_per_batch, total)); break;
        case 15: PGB_TRY(launch_inv_sub<12>(m, cin, ws, jobs_per_batch, total)); break;
        default: PGB_TRY(launch_inv_sub<13>(m, cin, ws, jobs_per_batch, total)); break;
        }
        TopJobs tj = {ws, cout, jobs_per_batch, total, (int)m->n, -1};
        dim3 grid(((unsigned)(m->n >> 3) + 255) / 256, total);
        { ProfScope _ps(m, PROF_DFT_INV);
        ntt120_inv_top8_kernel<<<grid, 256, 0, m->stream>>>(tj, m->ntt_inv, m->nc);
        }
        PGB_CHECK_CUDA(cudaGetLastError());
    }
    return PGB_OK;
}

// in: i64 limbs, out: 16 B/coef DFT limbs
int ntt120_forward(pgb_module *m, LimbSet in, LimbSet out, int jobs_per_batch, int batch, long long and_mask) {
    NttJobs jb = {in, out, jobs_per_batch, jobs_per_batch * batch, nullptr, 0, and_mask};
    if (jb.total_jobs == 0) return PGB_OK;
    if (m->log_n >= 14) return ntt120_forward_large(m, in, out, jobs_per_batch, batch, and_mask);
    NTT_DISPATCH(launch_fwd)
}
int ntt120_forward_skip(pgb_module *m, LimbSet in, LimbSet out, int jobs_per_batch, int batch, const int *skip, bool skip_list) {
    NttJobs jb = {in, out, jobs_per_batch, jobs_per_batch * batch, skip, skip_list ? 1 : 0, -1};
    if (jb.total_jobs == 0) return PGB_OK;
    PGB_REQUIRE(m->log_n < 14, "ntt120_forward_skip: single-CTA sizes only");
    NTT_DISPATCH(launch_fwd)
}
// in: DFT limbs, out: i128 limbs (may alias `in` limb for limb: in-place consume)
int ntt120_inverse_big(pgb_module *m, LimbSet in, LimbSet out, int jobs_per_batch, int batch) {
    NttJobs jb = {in, out, jobs_per_batch, jobs_per_batch * batch, nullptr, 0, -1};
    if (jb.total_jobs == 0) return PGB_OK;
    if (m->log_n >= 14) return ntt120_inverse_large(m, in, out, jobs_per_batch, batch);
    NTT_DISPATCH(launch_inv)
}

template <int L> static int launch_fused(pgb_module *m, const FusedArgs &p, int batch, const int *skip, int skip_list) {
    typedef Geo<L> G;
    size_t smem = (size_t)4 * G::PLANE * sizeof(uint32_t);
    static int ctas_per_sm_dev[32] = {}, sms_dev[32] = {};
    int &ctas_per_sm = ctas_per_sm_dev[m->device & 31], &sms = sms_dev[m->device & 31];
    if (!ctas_per_sm) {
        PGB_CHECK_CUDA(cudaFuncSetAttribute(ntt120_fused_back_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        PGB_CHECK_CUDA(cudaFuncSetAttribute(ntt120_fused_back_kernel<L>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        PGB_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, ntt120_fused_back_kernel<L>, G::T, smem));
        PGB_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, m->device));
        if (ctas_per_sm < 1) ctas_per_sm = 1;
    }
    const int total = p.cols_out * batch;
    const int grid = total < sms * ctas_per_sm ? total : sms * ctas_per_sm;
    PGB_TRY(ensure_carry_ws(m, (size_t)grid * G::NB * sizeof(i128)));
    { ProfScope _ps(m, PROF_DFT_INV);
    ntt120_fused_back_kernel<L><<<grid, G::T, smem, m->stream>>>(p, m->ntt_inv, m->nc, total, (i128 *)m->carry_ws, skip, skip_list);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}
template <int L> static int launch_collapsed(pgb_module *m, const FusedArgs &p, int batch, const int *ok) {
    typedef Geo<L> G;
    size_t smem = (size_t)4 * G::PLANE * sizeof(uint32_t);
    static int ctas_per_sm_dev[32] = {}, sms_dev[32] = {};
    int &ctas_per_sm = ctas_per_sm_dev[m->device & 31], &sms = sms_dev[m->device & 31];
    if (!ctas_per_sm) {
        PGB_CHECK_CUDA(cudaFuncSetAttribute(ntt120_collapsed_back_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        PGB_CHECK_CUDA(cudaFuncSetAttribute(ntt120_collapsed_back_kernel<L>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        PGB_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas_per_sm, ntt120_collapsed_back_kernel<L>, G::T, smem));
        PGB_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, m->device));
        if (ctas_per_sm < 1) ctas_per_sm = 1;
    }
    const int total = p.cols_out * batch;
    const int grid = total < sms * ctas_per_sm ? total : sms * ctas_per_sm;
    { ProfScope _ps(m, PROF_DFT_INV);
    ntt120_collapsed_back_kernel<L><<<grid, G::T, smem, m->stream>>>(p, m->ntt_inv, m->nc, total, ok);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

bool ntt120_fused_supported(const pgb_module *m) { return m->flavour == PGB_NTT120 && m->log_n >= 9 && m->log_n <= 13; }

// exact integer coefficients of every key polynomial (|.| < Q/2, inverse NTT + CRT), then their largest bit length
int ntt120_key_max_bits(pgb_module *m, const char *pmat, int polys, char *coef_ws, int *bits_dev) {
    const uint64_t poly_bytes = 16 * m->n;
    LimbSet kin = {(char *)pmat, poly_bytes, 0}, kout = {coef_ws, poly_bytes, 0};
    PGB_TRY(ntt120_inverse_big(m, kin, kout, polys, 1));
    PGB_CHECK_CUDA(cudaMemsetAsync(bits_dev, 0, sizeof(int), m->stream));
    { ProfScope _ps(m, PROF_OTHER);
    max_bits_i128_kernel<<<296, 256, 0, m->stream>>>((const i128 *)coef_ws, (size_t)polys * m->n, bits_dev);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

static uint32_t pow2_mod_q(uint64_t e, uint32_t q) {
    uint64_t r = 1, b = 2;
    while (e) {
        if (e & 1) r = r * b % q;
        b = b * b % q;
        e >>= 1;
    }
    return (uint32_t)r;
}

// res(cols_out, res_size) <- normalize( idft( a_dft(R polys) x pmat[R][C] ) + small on column 0 ), same base2k, offset res_offset.
// `glwe` / `glwe_bs` / `glwe_words`: the i64 input ciphertexts (all columns), used only to bound the integers for the collapsed path.
int ntt120_fused_back(pgb_module *m, const char *a_dft, uint64_t a_bs, const char *pmat, int R, int C, int cols_out, const char *small,
                      uint64_t small_bs, uint64_t small_limb_stride, int small_size, char *res, uint64_t res_bs, uint64_t res_limb_stride,
                      int res_size, int base2k, int64_t res_offset, int batch, const char *glwe, uint64_t glwe_bs, uint64_t glwe_words,
                      const int *skip, bool skip_list, bool direct, bool small_all_cols, uint64_t pmat_bs) {
    FusedArgs p;
    memset(&p, 0, sizeof p);
    p.a_dft = a_dft; p.a_bs = a_bs; p.pmat = pmat; p.pmat_bs = pmat_bs; p.small = small; p.small_bs = small_bs; p.small_limb_stride = small_limb_stride;
    p.small_size = small_size; p.res = res; p.res_bs = res_bs; p.res_limb_stride = res_limb_stride;
    p.R = R; p.C = C; p.cols_out = cols_out;
    p.direct = direct ? 1 : 0; p.small_all_cols = small_all_cols ? 1 : 0;
    p.K = base2k; p.res_size = res_size; p.a_size = C / cols_out;
    int64_t lsh = res_offset % base2k, lo = res_offset / base2k;
    if (res_offset < 0 && lsh != 0) {
        lsh = (lsh + base2k) % base2k;
        lo -= 1;
    }
    auto clampi = [](int64_t v, int64_t a, int64_t b) { return v < a ? a : (v > b ? b : v); };
    p.lsh = (int)lsh;
    p.res_end = (int)clampi(-lo, 0, res_size);
    p.res_start = (int)clampi((int64_t)p.a_size - lo, 0, res_size);
    p.a_end = (int)clampi(lo, 0, p.a_size);
    p.a_start = (int)clampi((int64_t)res_size + lo, 0, p.a_size);

    // ---- collapsed-key fast path (see the comment above ntt120_collapse_key_kernel) -------------------------------------------
    const uint64_t n = m->n, poly_bytes = 16 * n;
    const int S = p.a_size;
    const uint64_t key_bytes = (uint64_t)R * C * poly_bytes;
    const int *ok = skip;
    const bool try_collapse = glwe && !skip && !direct && pmat_bs == 0 && res_offset == 0 && S >= 2 && S <= 32 && (int64_t)batch * cols_out >= 64 && key_bytes <= ((uint64_t)64 << 20) &&
                              (S - 1) * base2k + 3 < 118 && !opt_on(m, PGB_OPT_NO_COLLAPSE);
    if (try_collapse) {
        // workspace: [collapsed key | key coefficients (i128) | key_bits | ok flags]
        const uint64_t ck_bytes = (uint64_t)R * cols_out * poly_bytes;
        const uint64_t need = ck_bytes + key_bytes + 256 + (uint64_t)batch * sizeof(int);
        if (m->aux_len < need) {
            if (m->aux_ws) {
                PGB_CHECK_CUDA(cudaStreamSynchronize(m->stream));
                cudaFree(m->aux_ws);
            }
            m->aux_ws = nullptr;
            m->aux_len = 0;
            PGB_CHECK_CUDA(cudaMalloc(&m->aux_ws, need));
            m->aux_len = need;
        }
        char *ck = (char *)m->aux_ws, *kcoef = ck + ck_bytes;
        int *key_bits = (int *)(kcoef + key_bytes), *okf = key_bits + 64;
        CollapseArgs ca;
        memset(&ca, 0, sizeof ca);
        ca.pmat = pmat; ca.out = ck; ca.n4 = (int)(n / 4); ca.R = R; ca.C = C; ca.cols_out = cols_out; ca.S = S;
        for (int j = 0; j < S; j++)
            for (int k = 0; k < 4; k++) ca.c[j][k] = pow2_mod_q((uint64_t)(S - 1 - j) * base2k, qk(k));
        { ProfScope _ps(m, PROF_OTHER);
        ntt120_collapse_key_kernel<<<dim3(((unsigned)n + 255) / 256, R * cols_out), 256, 0, m->stream>>>(ca);
        }
        PGB_CHECK_CUDA(cudaGetLastError());
        PGB_TRY(ntt120_key_max_bits(m, pmat, R * C, kcoef, key_bits));
        int rn_bits = 0;
        while (((uint64_t)1 << rn_bits) < (uint64_t)R * n) rn_bits++;
        GuardArgs ga = {glwe, glwe_bs, glwe_words, key_bits, rn_bits + (S - 1) * base2k + 3, okf};
        { ProfScope _ps(m, PROF_OTHER);
        ntt120_collapse_guard_kernel<<<batch, 256, 0, m->stream>>>(ga);
        }
        PGB_CHECK_CUDA(cudaGetLastError());
        FusedArgs pc = p;
        pc.pmat = ck;
        switch (m->log_n) {
        case 9: PGB_TRY(launch_collapsed<9>(m, pc, batch, okf)); break;
        case 10: PGB_TRY(launch_collapsed<10>(m, pc, batch, okf)); break;
        case 11: PGB_TRY(launch_collapsed<11>(m, pc, batch, okf)); break;
        case 12: PGB_TRY(launch_collapsed<12>(m, pc, batch, okf)); break;
        case 13: PGB_TRY(launch_collapsed<13>(m, pc, batch, okf)); break;
        default: pgb_set_error("fused back end: unsupported n"); return PGB_ERR_UNSUPPORTED;
        }
        ok = okf; // the per-limb kernel below only processes the ciphertexts that failed the bound
    }
    switch (m->log_n) {
    case 9: return launch_fused<9>(m, p, batch, ok, (skip && skip_list) ? 1 : 0);
    case 10: return launch_fused<10>(m, p, batch, ok, (skip && skip_list) ? 1 : 0);
    case 11: return launch_fused<11>(m, p, batch, ok, (skip && skip_list) ? 1 : 0);
    case 12: return launch_fused<12>(m, p, batch, ok, (skip && skip_list) ? 1 : 0);
    case 13: return launch_fused<13>(m, p, batch, ok, (skip && skip_list) ? 1 : 0);
    default: pgb_set_error("fused back end: unsupported n"); return PGB_ERR_UNSUPPORTED;
    }
}
