// fft64.cu -- FFT64 flavour: batched forward / inverse negacyclic FFT (K3 / K4) and the f64 element-wise kernels
// (vmp K6, svp K5, add/sub K8).
//
// Conventions (poulpy-cpu-ref/src/reference/fft64/reim/*, SURVEY.md appendix A.5): a real polynomial of n
// coefficients is folded to m = n/2 complex points z_j = a_j + i*a_{j+m}; a DFT limb is [re(m) | im(m)] f64 and
//   out[p] = sum_j z_j * zeta^(j * (4*bitrev_{log m}(p) + 1)),  zeta = exp(2*pi*i / (2n))
// which is exactly the order the reference's fft16/bitwiddle traversal produces (tests/test_oracle_kat.py pins it).
// The inverse is unnormalised; the 1/m and the round-half-away-from-zero of reim_to_znx_i64 (conversion.rs:43-60)
// are fused into its last pass.  Butterflies use FMA (the reference does not): DFT-domain values agree with the
// oracle to a stated tolerance, the rounded i64 results exactly (same contract as poulpy-cpu-avx vs poulpy-cpu-ref,
// poulpy-cpu-avx/src/fft64/reim/fft_avx2_fma.rs:318-353).
#include <math.h>

#include "internal.h"
#include "fft64.cuh"

struct FftJobs {
    LimbSet in, out;
    int jobs_per_batch;
    int total_jobs;
    long long and_mask; // i64 inputs are ANDed with this before conversion (cnv_prepare's masked last limb); -1 = none
};

template <int L, int L0> struct FFwdMid {
    static __device__ __forceinline__ void run(double2 *sm, double *gout, const double2 *tw, int t, bool active, uint32_t root = 1u,
                                               int m_plane = FGeo<L>::M, const double2 *twl = nullptr) {
        typedef FGeo<L> G;
        constexpr int SL = L - L0 - 3;
        const int a = t >> SL, b = t & ((1 << SL) - 1);
        const int base = (a << (SL + 3)) | b;
        const uint32_t hi = (root << L0) | (uint32_t)a;
        double2 x[8];
#pragma unroll
        for (int j = 0; j < 8; j++) x[j] = sm[FPAD(base + (j << SL))];
        if (SL == 0 && twl) { // whole-transform last pass (root == 1): coalesced per-thread twiddles
            double2 w[7];
            load_tw7(w, twl, G::T, t);
            fct_radix8_w(x, w);
        } else {
            fct_radix8<3>(x, tw, hi);
        }
        if (SL == 0) {
            if (active) {
                double2 *ore = reinterpret_cast<double2 *>(gout + base), *oim = reinterpret_cast<double2 *>(gout + m_plane + base);
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    ore[j] = make_double2(x[2 * j].x, x[2 * j + 1].x);
                    oim[j] = make_double2(x[2 * j].y, x[2 * j + 1].y);
                }
            }
        } else {
#pragma unroll
            for (int j = 0; j < 8; j++) sm[FPAD(base + (j << SL))] = x[j];
            __syncthreads();
        }
        FFwdMid<L, (L0 + 3 < L) ? L0 + 3 : L>::run(sm, gout, tw, t, active, root, m_plane, twl);
    }
};
template <int L> struct FFwdMid<L, L> {
    static __device__ __forceinline__ void run(double2 *, double *, const double2 *, int, bool, uint32_t = 1u, int = 0, const double2 * = nullptr) {}
};

template <int L, int LPC> __global__ void __launch_bounds__(FGeo<L>::T *LPC) fft64_fwd_kernel(FftJobs jb, const double2 *__restrict__ tw,
                                                                                         const double2 *__restrict__ twl) {
    typedef FGeo<L> G;
    extern __shared__ __align__(16) double2 fsm[];
    const int slot = threadIdx.x / G::T, t = threadIdx.x % G::T;
    const int job = blockIdx.x * LPC + slot;
    const bool active = job < jb.total_jobs;
    const int b = active ? job / jb.jobs_per_batch : 0, j = active ? job % jb.jobs_per_batch : 0;
    const long long *gin = reinterpret_cast<const long long *>(jb.in.base + (size_t)b * jb.in.batch_stride + (size_t)j * jb.in.limb_stride);
    double *gout = reinterpret_cast<double *>(jb.out.base + (size_t)b * jb.out.batch_stride + (size_t)j * jb.out.limb_stride);
    double2 *sm = fsm + slot * G::PLANE;
    double2 x[8];
#pragma unroll
    for (int jj = 0; jj < 8; jj++) {
        const int idx = t + jj * G::T;
        x[jj] = active ? make_double2((double)(__ldg(gin + idx) & jb.and_mask), (double)(__ldg(gin + G::M + idx) & jb.and_mask)) : make_double2(0.0, 0.0);
    }
    fct_radix8<G::R0>(x, tw, 1u);
    if (L == G::R0) {
        if (active) {
#pragma unroll
            for (int jj = 0; jj < 8; jj++) {
                gout[jj] = x[jj].x;
                gout[G::M + jj] = x[jj].y;
            }
        }
        return;
    }
#pragma unroll
    for (int jj = 0; jj < 8; jj++) sm[FPAD(t + jj * G::T)] = x[jj];
    __syncthreads();
    FFwdMid<L, (L > G::R0) ? G::R0 : L>::run(sm, gout, tw, t, active, 1u, G::M, twl);
}

template <int L, int L0> struct FInvMid {
    static __device__ __forceinline__ void run(double2 *sm, const double2 *tw, int t, uint32_t root = 1u) {
        typedef FGeo<L> G;
        constexpr int SL = L - L0 - 3;
        const int a = t >> SL, b = t & ((1 << SL) - 1);
        const int base = (a << (SL + 3)) | b;
        const uint32_t hi = (root << L0) | (uint32_t)a;
        double2 x[8];
#pragma unroll
        for (int j = 0; j < 8; j++) x[j] = sm[FPAD(base + (j << SL))];
        fgs_radix8<3>(x, tw, hi);
#pragma unroll
        for (int j = 0; j < 8; j++) sm[FPAD(base + (j << SL))] = x[j];
        __syncthreads();
        FInvMid<L, (L0 - 3 >= G::R0) ? L0 - 3 : -1>::run(sm, tw, t, root);
    }
};
template <int L> struct FInvMid<L, -1> {
    static __device__ __forceinline__ void run(double2 *, const double2 *, int, uint32_t = 1u) {}
};

template <int L, int LPC> __global__ void __launch_bounds__(FGeo<L>::T *LPC) fft64_inv_kernel(FftJobs jb, const double2 *__restrict__ tw, double inv_m,
                                                                                         const double2 *__restrict__ twl) {
    typedef FGeo<L> G;
    extern __shared__ __align__(16) double2 fsm[];
    const int slot = threadIdx.x / G::T, t = threadIdx.x % G::T;
    const int job = blockIdx.x * LPC + slot;
    const bool active = job < jb.total_jobs;
    const int b = active ? job / jb.jobs_per_batch : 0, j = active ? job % jb.jobs_per_batch : 0;
    const double *gin = reinterpret_cast<const double *>(jb.in.base + (size_t)b * jb.in.batch_stride + (size_t)j * jb.in.limb_stride);
    long long *gout = reinterpret_cast<long long *>(jb.out.base + (size_t)b * jb.out.batch_stride + (size_t)j * jb.out.limb_stride);
    double2 *sm = fsm + slot * G::PLANE;
    double2 x[8];
    if (L > G::R0) {
        constexpr int L0 = L - 3;
        if (active) {
            const double2 *pre = reinterpret_cast<const double2 *>(gin + 8 * t), *pim = reinterpret_cast<const double2 *>(gin + G::M + 8 * t);
#pragma unroll
            for (int jj = 0; jj < 4; jj++) {
                double2 r = pre[jj], i = pim[jj];
                x[2 * jj] = make_double2(r.x, i.x);
                x[2 * jj + 1] = make_double2(r.y, i.y);
            }
        } else {
#pragma unroll
            for (int jj = 0; jj < 8; jj++) x[jj] = make_double2(0.0, 0.0);
        }
        {
            double2 w[7];
            load_tw7(w, twl, G::T, t);
            fgs_radix8_w(x, w);
        }
#pragma unroll
        for (int jj = 0; jj < 8; jj++) sm[FPAD(8 * t + jj)] = x[jj];
        __syncthreads();
        FInvMid<L, (L - 6 >= G::R0) ? L - 6 : -1>::run(sm, tw, t);
#pragma unroll
        for (int jj = 0; jj < 8; jj++) x[jj] = sm[FPAD(t + jj * G::T)];
    } else {
#pragma unroll
        for (int jj = 0; jj < 8; jj++) x[jj] = active ? make_double2(gin[jj], gin[G::M + jj]) : make_double2(0.0, 0.0);
        __syncthreads();
    }
    fgs_radix8<G::R0>(x, tw, 1u);
    if (active) {
#pragma unroll
        for (int jj = 0; jj < 8; jj++) {
            const int idx = t + jj * G::T;
            gout[idx] = (long long)round(x[jj].x * inv_m);
            gout[G::M + idx] = (long long)round(x[jj].y * inv_m);
        }
    }
}

// ---- fused back end of one accumulator column (CGGI outside the fully fused kernel): inverse transform of the S limbs of (ciphertext,
// column) in one CTA (slot = limb), round (conversion.rs:43-52), + the column's own limbs (vec_znx_big_add_small_assign), same-base2k carry
// chain from the least significant limb (vec_znx_big_normalize) straight into the column -- what idft / add_small / normalize did in three
// launches per column with the i64 big crossing HBM three times.  In place on `res` (a thread reads limb j of a coefficient before it
// writes it; nobody else touches that word).
struct FBackArgs {
    const char *in;  unsigned long long in_bs;   // DFT limbs: poly (j * cols + c) at + ((j * cols + c) * n * 8)
    char *res;       unsigned long long res_bs;  // VecZnx: limb (j, c) at + ((j * cols + c) * n * 8)
    int cols, S, res_size, small_size, K;
    double inv_m;
};
template <int L> __global__ void __launch_bounds__(1024) fft64_back_kernel(FBackArgs p, const double2 *__restrict__ tw, const double2 *__restrict__ twl) {
    typedef FGeo<L> G;
    constexpr int M = G::M, N = 2 * M;
    extern __shared__ __align__(16) double2 fsm[];
    const int slot = threadIdx.x / G::T, t = threadIdx.x % G::T; // slot = limb
    const int b = blockIdx.x / p.cols, c = blockIdx.x % p.cols;
    const double *gin = reinterpret_cast<const double *>(p.in + (size_t)b * p.in_bs) + ((size_t)slot * p.cols + c) * N;
    double2 *sm = fsm + slot * G::PLANE;
    double2 x[8];
    if (L > G::R0) {
        const double2 *pre = reinterpret_cast<const double2 *>(gin + 8 * t), *pim = reinterpret_cast<const double2 *>(gin + M + 8 * t);
#pragma unroll
        for (int jj = 0; jj < 4; jj++) {
            double2 r = pre[jj], i = pim[jj];
            x[2 * jj] = make_double2(r.x, i.x);
            x[2 * jj + 1] = make_double2(r.y, i.y);
        }
        {
            double2 w[7];
            load_tw7(w, twl, G::T, t);
            fgs_radix8_w(x, w);
        }
#pragma unroll
        for (int jj = 0; jj < 8; jj++) sm[FPAD(8 * t + jj)] = x[jj];
        __syncthreads();
        FInvMid<L, (L - 6 >= G::R0) ? L - 6 : -1>::run(sm, tw, t);
#pragma unroll
        for (int jj = 0; jj < 8; jj++) x[jj] = sm[FPAD(t + jj * G::T)];
    } else {
#pragma unroll
        for (int jj = 0; jj < 8; jj++) x[jj] = make_double2(gin[jj], gin[M + jj]);
    }
    fgs_radix8<G::R0>(x, tw, 1u);
    __syncthreads(); // every thread has taken its last-pass inputs: the planes now hold the rounded i64 coefficients
    long long *big = reinterpret_cast<long long *>(sm);
#pragma unroll
    for (int jj = 0; jj < 8; jj++) {
        const int idx = t + jj * G::T;
        big[idx] = (long long)round(x[jj].x * p.inv_m);
        big[M + idx] = (long long)round(x[jj].y * p.inv_m);
    }
    __syncthreads();
    const int a_start = p.res_size < p.S ? p.res_size : p.S; // limbs >= a_start only feed the carry
    long long *res = reinterpret_cast<long long *>(p.res + (size_t)b * p.res_bs) + (size_t)c * N;
    const size_t ls = (size_t)p.cols * N;
    for (int idx = threadIdx.x; idx < N; idx += blockDim.x) {
        long long carry = 0;
        for (int j = p.S - 1; j >= 0; j--) {
            long long v = reinterpret_cast<const long long *>(fsm + j * G::PLANE)[idx];
            if (j < p.small_size) v = (long long)((unsigned long long)v + (unsigned long long)res[(size_t)j * ls + idx]);
            const long long o = norm_step(v, carry, p.K);
            if (j < a_start) res[(size_t)j * ls + idx] = o;
        }
        for (int j = a_start; j < p.res_size; j++) res[(size_t)j * ls + idx] = 0; // normalize.rs:60-66
    }
}
template <int L> static int flaunch_back(pgb_module *m, const FBackArgs &p, int batch) {
    typedef FGeo<L> G;
    const size_t smem = (size_t)p.S * G::PLANE * sizeof(double2);
    static bool attr_set_dev[32] = {};
    bool &attr_set = attr_set_dev[m->device & 31];
    if (!attr_set) {
        PGB_CHECK_CUDA(cudaFuncSetAttribute(fft64_back_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(227 << 10)));
        attr_set = true;
    }
    { ProfScope _ps(m, PROF_DFT_INV);
    fft64_back_kernel<L><<<batch * p.cols, G::T * p.S, smem, m->stream>>>(p, m->fft_inv, m->fft_last_i);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}
bool fft64_fused_back_supported(const pgb_module *m, int S) {
    if (m->flavour != PGB_FFT64 || m->log_n < 7 || m->log_n > 13 || S < 1) return false;
    const size_t M = m->n / 2, T = M / 8, PL = M + (M >> 3) + 2;
    return (size_t)S * T <= 1024 && (size_t)S * PL * sizeof(double2) <= (size_t)(227 << 10);
}
int fft64_fused_back(pgb_module *m, const char *in, uint64_t in_bs, int cols, int S, char *res, uint64_t res_bs, int res_size, int base2k, int batch) {
    FBackArgs p = {in, in_bs, res, res_bs, cols, S, res_size, S < res_size ? S : res_size, base2k, 1.0 / (double)(m->n / 2)};
    switch (m->log_n - 1) {
    case 6: return flaunch_back<6>(m, p, batch);
    case 7: return flaunch_back<7>(m, p, batch);
    case 8: return flaunch_back<8>(m, p, batch);
    case 9: return flaunch_back<9>(m, p, batch);
    case 10: return flaunch_back<10>(m, p, batch);
    case 11: return flaunch_back<11>(m, p, batch);
    case 12: return flaunch_back<12>(m, p, batch);
    default: pgb_set_error("fft64 fused back end: unsupported n"); return PGB_ERR_UNSUPPORTED;
    }
}

int fft64_module_init(pgb_module *m) {
    const uint64_t mm = m->n / 2;
    uint64_t *E = (uint64_t *)malloc(sizeof(uint64_t) * (mm > 2 ? mm : 2));
    E[1] = mm / 2; // numerators over 4m: root block angle 1/4 -> twiddle angle 1/8
    for (uint64_t i = 1; 2 * i + 1 < mm; i++) {
        E[2 * i] = E[i] / 2;
        E[2 * i + 1] = E[i] / 2 + mm;
    }
    double2 *hf = (double2 *)calloc(mm, sizeof(double2)), *hi = (double2 *)calloc(mm, sizeof(double2));
    const long double two_pi = 6.283185307179586476925286766559005768L;
    for (uint64_t i = 1; i < mm; i++) {
        long double ang = two_pi * (long double)E[i] / (long double)(4 * mm);
        double c = (double)cosl(ang), s = (double)sinl(ang);
        hf[i] = make_double2(c, s);
        hi[i] = make_double2(c, -s);
    }
    free(E);
    PGB_CHECK_CUDA(cudaMalloc(&m->fft_fwd, mm * sizeof(double2)));
    PGB_CHECK_CUDA(cudaMalloc(&m->fft_inv, mm * sizeof(double2)));
    PGB_CHECK_CUDA(cudaMemcpy(m->fft_fwd, hf, mm * sizeof(double2), cudaMemcpyHostToDevice));
    PGB_CHECK_CUDA(cudaMemcpy(m->fft_inv, hi, mm * sizeof(double2), cudaMemcpyHostToDevice));
    m->fft_last_f = m->fft_last_i = nullptr;
    if (mm >= 8) { // last-pass tables (fft64.cuh: load_tw7): thread t of T = m/8 owns node hi = T + t
        const uint64_t T = mm / 8;
        double2 *lf = (double2 *)malloc(7 * T * sizeof(double2)), *li = (double2 *)malloc(7 * T * sizeof(double2));
        for (uint64_t t = 0; t < T; t++) {
            const uint64_t node = T + t, idx[7] = {node, 2 * node, 2 * node + 1, 4 * node, 4 * node + 1, 4 * node + 2, 4 * node + 3};
            for (int j = 0; j < 7; j++) {
                lf[j * T + t] = hf[idx[j]];
                li[j * T + t] = hi[idx[j]];
            }
        }
        PGB_CHECK_CUDA(cudaMalloc(&m->fft_last_f, 7 * T * sizeof(double2)));
        PGB_CHECK_CUDA(cudaMalloc(&m->fft_last_i, 7 * T * sizeof(double2)));
        PGB_CHECK_CUDA(cudaMemcpy(m->fft_last_f, lf, 7 * T * sizeof(double2), cudaMemcpyHostToDevice));
        PGB_CHECK_CUDA(cudaMemcpy(m->fft_last_i, li, 7 * T * sizeof(double2), cudaMemcpyHostToDevice));
        free(lf);
        free(li);
    }
    free(hf);
    free(hi);
    return PGB_OK;
}

template <int L> static constexpr int flpc_for() { return FGeo<L>::T >= 128 ? 1 : (128 / FGeo<L>::T > 16 ? 16 : 128 / FGeo<L>::T); }

template <int L> static int flaunch_fwd(pgb_module *m, const FftJobs &jb) {
    constexpr int LPC = flpc_for<L>();
    typedef FGeo<L> G;
    size_t smem = (size_t)LPC * G::PLANE * sizeof(double2);
    static bool attr_set_dev[32] = {}; // per device: function attributes are per device
    bool &attr_set = attr_set_dev[m->device & 31];
    if (!attr_set) {
        PGB_CHECK_CUDA(cudaFuncSetAttribute(fft64_fwd_kernel<L, LPC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    int grid = (jb.total_jobs + LPC - 1) / LPC;
    { ProfScope _ps(m, PROF_DFT_FWD);
    fft64_fwd_kernel<L, LPC><<<grid, G::T * LPC, smem, m->stream>>>(jb, m->fft_fwd, m->fft_last_f);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}
template <int L> static int flaunch_inv(pgb_module *m, const FftJobs &jb) {
    constexpr int LPC = flpc_for<L>();
    typedef FGeo<L> G;
    size_t smem = (size_t)LPC * G::PLANE * sizeof(double2);
    static bool attr_set_dev[32] = {}; // per device: function attributes are per device
    bool &attr_set = attr_set_dev[m->device & 31];
    if (!attr_set) {
        PGB_CHECK_CUDA(cudaFuncSetAttribute(fft64_inv_kernel<L, LPC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    int grid = (jb.total_jobs + LPC - 1) / LPC;
    { ProfScope _ps(m, PROF_DFT_INV);
    fft64_inv_kernel<L, LPC><<<grid, G::T * LPC, smem, m->stream>>>(jb, m->fft_inv, 1.0 / (double)(m->n / 2), m->fft_last_i);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

// ---- m > 8192: global radix-8 top pass + eight size-m/8 sub-transforms (block twiddles rooted at 8 + sub-block) -----------
struct FTopJobs {
    LimbSet in, out;
    int jobs_per_batch, total_jobs, m;
    long long and_mask;
};
__global__ void __launch_bounds__(256) fft64_fwd_top8_kernel(FTopJobs jb, const double2 *__restrict__ tw) {
    const int m = jb.m, s = m >> 3;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= s) return;
    const int job = blockIdx.y, b = job / jb.jobs_per_batch, j = job % jb.jobs_per_batch;
    const long long *gin = reinterpret_cast<const long long *>(jb.in.base + (size_t)b * jb.in.batch_stride + (size_t)j * jb.in.limb_stride);
    double *gout = reinterpret_cast<double *>(jb.out.base + (size_t)b * jb.out.batch_stride + (size_t)j * jb.out.limb_stride);
    double2 x[8];
#pragma unroll
    for (int jj = 0; jj < 8; jj++) x[jj] = make_double2((double)(__ldg(gin + i + jj * s) & jb.and_mask), (double)(__ldg(gin + m + i + jj * s) & jb.and_mask));
    fct_radix8<3>(x, tw, 1u);
#pragma unroll
    for (int jj = 0; jj < 8; jj++) {
        gout[i + jj * s] = x[jj].x;
        gout[m + i + jj * s] = x[jj].y;
    }
}
template <int L> __global__ void __launch_bounds__(FGeo<L>::T) fft64_fwd_sub_kernel(LimbSet out, int jobs_per_batch, int m_total,
                                                                                  const double2 *__restrict__ tw) {
    typedef FGeo<L> G;
    extern __shared__ __align__(16) double2 fsm[];
    const int t = threadIdx.x;
    const int sb = blockIdx.x & 7, limb = blockIdx.x >> 3;
    const int b = limb / jobs_per_batch, j = limb % jobs_per_batch;
    double *g = reinterpret_cast<double *>(out.base + (size_t)b * out.batch_stride + (size_t)j * out.limb_stride) + (size_t)sb * G::M;
    const uint32_t root = 8u | (uint32_t)sb;
    double2 x[8];
#pragma unroll
    for (int jj = 0; jj < 8; jj++) x[jj] = make_double2(g[t + jj * G::T], g[m_total + t + jj * G::T]);
    fct_radix8<G::R0>(x, tw, root);
#pragma unroll
    for (int jj = 0; jj < 8; jj++) fsm[FPAD(t + jj * G::T)] = x[jj];
    __syncthreads();
    FFwdMid<L, G::R0>::run(fsm, g, tw, t, true, root, m_total);
}
template <int L> __global__ void __launch_bounds__(FGeo<L>::T) fft64_inv_sub_kernel(LimbSet in, LimbSet out, int jobs_per_batch, int m_total,
                                                                                  const double2 *__restrict__ tw) {
    typedef FGeo<L> G;
    extern __shared__ __align__(16) double2 fsm[];
    const int t = threadIdx.x;
    const int sb = blockIdx.x & 7, limb = blockIdx.x >> 3;
    const int b = limb / jobs_per_batch, j = limb % jobs_per_batch;
    const double *gi = reinterpret_cast<const double *>(in.base + (size_t)b * in.batch_stride + (size_t)j * in.limb_stride) + (size_t)sb * G::M;
    double *go = reinterpret_cast<double *>(out.base + (size_t)b * out.batch_stride + (size_t)j * out.limb_stride) + (size_t)sb * G::M;
    const uint32_t root = 8u | (uint32_t)sb;
    double2 x[8];
    {
        const double2 *pre = reinterpret_cast<const double2 *>(gi + 8 * t), *pim = reinterpret_cast<const double2 *>(gi + m_total + 8 * t);
#pragma unroll
        for (int jj = 0; jj < 4; jj++) {
            double2 r = pre[jj], i = pim[jj];
            x[2 * jj] = make_double2(r.x, i.x);
            x[2 * jj + 1] = make_double2(r.y, i.y);
        }
    }
    fgs_radix8<3>(x, tw, (root << (L - 3)) | (uint32_t)t);
#pragma unroll
    for (int jj = 0; jj < 8; jj++) fsm[FPAD(8 * t + jj)] = x[jj];
    __syncthreads();
    FInvMid<L, (L - 6 >= G::R0) ? L - 6 : -1>::run(fsm, tw, t, root);
#pragma unroll
    for (int jj = 0; jj < 8; jj++) x[jj] = fsm[FPAD(t + jj * G::T)];
    fgs_radix8<G::R0>(x, tw, root);
#pragma unroll
    for (int jj = 0; jj < 8; jj++) {
        go[t + jj * G::T] = x[jj].x;
        go[m_total + t + jj * G::T] = x[jj].y;
    }
}
// in place on the f64 limb left by the sub-transforms: top three levels, scale by 1/m, round, reinterpret as i64
__global__ void __launch_bounds__(256) fft64_inv_top8_kernel(LimbSet io, int jobs_per_batch, int m, const double2 *__restrict__ tw, double inv_m) {
    const int s = m >> 3;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= s) return;
    const int job = blockIdx.y, b = job / jobs_per_batch, j = job % jobs_per_batch;
    double *g = reinterpret_cast<double *>(io.base + (size_t)b * io.batch_stride + (size_t)j * io.limb_stride);
    double2 x[8];
#pragma unroll
    for (int jj = 0; jj < 8; jj++) x[jj] = make_double2(g[i + jj * s], g[m + i + jj * s]);
    fgs_radix8<3>(x, tw, 1u);
    long long *o = reinterpret_cast<long long *>(g);
#pragma unroll
    for (int jj = 0; jj < 8; jj++) {
        o[i + jj * s] = (long long)round(x[jj].x * inv_m);
        o[m + i + jj * s] = (long long)round(x[jj].y * inv_m);
    }
}

template <int L> static int flaunch_fwd_sub(pgb_module *m, LimbSet out, int jobs_per_batch, int total) {
    typedef FGeo<L> G;
    size_t smem = (size_t)G::PLANE * sizeof(double2);
    static bool attr_set_dev[32] = {}; // per device: function attributes are per device
    bool &attr_set = attr_set_dev[m->device & 31];
    if (!attr_set) {
        PGB_CHECK_CUDA(cudaFuncSetAttribute(fft64_fwd_sub_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    { ProfScope _ps(m, PROF_DFT_FWD);
    fft64_fwd_sub_kernel<L><<<total * 8, G::T, smem, m->stream>>>(out, jobs_per_batch, (int)(m->n / 2), m->fft_fwd);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}
template <int L> static int flaunch_inv_sub(pgb_module *m, LimbSet in, LimbSet out, int jobs_per_batch, int total) {
    typedef FGeo<L> G;
    size_t smem = (size_t)G::PLANE * sizeof(double2);
    static bool attr_set_dev[32] = {}; // per device: function attributes are per device
    bool &attr_set = attr_set_dev[m->device & 31];
    if (!attr_set) {
        PGB_CHECK_CUDA(cudaFuncSetAttribute(fft64_inv_sub_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set = true;
    }
    { ProfScope _ps(m, PROF_DFT_INV);
    fft64_inv_sub_kernel<L><<<total * 8, G::T, smem, m->stream>>>(in, out, jobs_per_batch, (int)(m->n / 2), m->fft_inv);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}
static int fft64_forward_large(pgb_module *m, LimbSet in, LimbSet out, int jobs_per_batch, int batch, long long and_mask) {
    const int total = jobs_per_batch * batch, mm = (int)(m->n / 2);
    PGB_REQUIRE(total <= 65535, "FFT64 large-n path: more than 65535 limbs per call (split the batch)");
    FTopJobs tj = {in, out, jobs_per_batch, total, mm, and_mask};
    dim3 grid(((unsigned)(mm >> 3) + 255) / 256, total);
    { ProfScope _ps(m, PROF_DFT_FWD);
    fft64_fwd_top8_kernel<<<grid, 256, 0, m->stream>>>(tj, m->fft_fwd);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return m->log_n == 15 ? flaunch_fwd_sub<11>(m, out, jobs_per_batch, total) : flaunch_fwd_sub<12>(m, out, jobs_per_batch, total);
}
static int fft64_inverse_large(pgb_module *m, LimbSet in, LimbSet out, int jobs_per_batch, int batch) {
    const int total = jobs_per_batch * batch, mm = (int)(m->n / 2);
    PGB_REQUIRE(total <= 65535, "FFT64 large-n path: more than 65535 limbs per call (split the batch)");
    PGB_TRY(m->log_n == 15 ? flaunch_inv_sub<11>(m, in, out, jobs_per_batch, total) : flaunch_inv_sub<12>(m, in, out, jobs_per_batch, total));
    dim3 grid(((unsigned)(mm >> 3) + 255) / 256, total);
    { ProfScope _ps(m, PROF_DFT_INV);
    fft64_inv_top8_kernel<<<grid, 256, 0, m->stream>>>(out, jobs_per_batch, mm, m->fft_inv, 1.0 / (double)mm);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

#define FFT_DISPATCH(fn)                           \
    switch (m->log_n - 1) {                        \
    case 3: return fn<3>(m, jb);                   \
    case 4: return fn<4>(m, jb);                   \
    case 5: return fn<5>(m, jb);                   \
    case 6: return fn<6>(m, jb);                   \
    case 7: return fn<7>(m, jb);                   \
    case 8: return fn<8>(m, jb);                   \
    case 9: return fn<9>(m, jb);                   \
    case 10: return fn<10>(m, jb);                 \
    case 11: return fn<11>(m, jb);                 \
    case 12: return fn<12>(m, jb);                 \
    case 13: return fn<13>(m, jb);                 \
    default:                                       \
        pgb_set_error("FFT64: n = 2^%d not supported by the single-CTA path (16 <= n <= 16384)", m->log_n); \
        return PGB_ERR_UNSUPPORTED;                \
    }

int fft64_forward(pgb_module *m, LimbSet in, LimbSet out, int jobs_per_batch, int batch, long long and_mask) {
    FftJobs jb = {in, out, jobs_per_batch, jobs_per_batch * batch, and_mask};
    if (jb.total_jobs == 0) return PGB_OK;
    if (m->log_n >= 15) return fft64_forward_large(m, in, out, jobs_per_batch, batch, and_mask);
    FFT_DISPATCH(flaunch_fwd)
}
int fft64_inverse_big(pgb_module *m, LimbSet in, LimbSet out, int jobs_per_batch, int batch) {
    FftJobs jb = {in, out, jobs_per_batch, jobs_per_batch * batch, -1};
    if (jb.total_jobs == 0) return PGB_OK;
    if (m->log_n >= 15) return fft64_inverse_large(m, in, out, jobs_per_batch, batch);
    FFT_DISPATCH(flaunch_inv)
}

// ---- vmp / svp / add / sub on [re | im] limbs ------------------------------------------------------------
struct FVmpArgs {
    const char *a;  uint64_t a_bs;
    char *res;      uint64_t res_bs;
    const char *pm; uint64_t pm_bs;  // item z's matrix at pm + (z / pm_div) * pm_bs
    uint32_t m2;     // double2 words per half limb (= m / 2)
    uint32_t row_max, C, col0, ncols_out, pm_div;
};
// each thread: two consecutive complex frequencies (double2 of re, double2 of im), CT output columns
template <int CT> __global__ void __launch_bounds__(128) fft64_vmp_kernel(FVmpArgs p) {
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= p.m2) return;
    const uint32_t c0 = blockIdx.y * CT;
    const size_t poly_words = (size_t)2 * p.m2; // double2 words per poly
    const double2 *a = reinterpret_cast<const double2 *>(p.a + (size_t)blockIdx.z * p.a_bs) + u;
    const double2 *pm = reinterpret_cast<const double2 *>(p.pm + (size_t)(blockIdx.z / p.pm_div) * p.pm_bs) + u + (size_t)(p.col0 + c0) * poly_words;
    double2 *res = reinterpret_cast<double2 *>(p.res + (size_t)blockIdx.z * p.res_bs) + u + (size_t)c0 * poly_words;
    const int nc = min((uint32_t)CT, p.ncols_out - c0);
    double2 accr[CT], acci[CT];
#pragma unroll
    for (int c = 0; c < CT; c++) accr[c] = acci[c] = make_double2(0.0, 0.0);
#pragma unroll 2
    for (uint32_t r = 0; r < p.row_max; r++) { // two rows of loads in flight per thread: the matrix is streamed once (evict-first)
        const double2 ar = __ldg(a + (size_t)r * poly_words), ai = __ldg(a + (size_t)r * poly_words + p.m2);
        const double2 *mrow = pm + (size_t)r * p.C * poly_words;
#pragma unroll
        for (int c = 0; c < CT; c++) {
            if (c < nc) {
                const double2 br = __ldcs(mrow + (size_t)c * poly_words), bi = __ldcs(mrow + (size_t)c * poly_words + p.m2);
                accr[c].x += ar.x * br.x - ai.x * bi.x;
                accr[c].y += ar.y * br.y - ai.y * bi.y;
                acci[c].x += ar.x * bi.x + ai.x * br.x;
                acci[c].y += ar.y * bi.y + ai.y * br.y;
            }
        }
    }
#pragma unroll
    for (int c = 0; c < CT; c++) {
        if (c < nc) {
            res[(size_t)c * poly_words] = accr[c];
            res[(size_t)c * poly_words + p.m2] = acci[c];
        }
    }
}
int fft64_vmp(pgb_module *m, const char *a, uint64_t a_bs, char *res, uint64_t res_bs, const char *pm, uint64_t pm_bs,
              uint32_t row_max, uint32_t C, uint32_t col0, uint32_t ncols_out, uint32_t batch, uint32_t pm_div) {
    if (ncols_out == 0 || batch == 0) return PGB_OK;
    FVmpArgs p = {a, a_bs, res, res_bs, pm, pm_bs, (uint32_t)(m->n / 4), row_max, C, col0, ncols_out, pm_div};
    // output polys per thread: 2 (default) or 4 (PGB_OPT_VMP_CT).  Measured on B200 in the streaming regime (scripts/vmp_stream.py,
    // profiles/r2_vmp_stream.md): two polys per thread reach 95-103 % of the measured copy bandwidth at every sweep shape, four 74-89 % --
    // the re-reads of `a` that four would save are L2 hits, the extra CTAs and the 70 (vs 128) registers are what the stream needs
    const int ct = m->opt[PGB_OPT_VMP_CT] == 4 ? 4 : 2;
    dim3 block(128);
    { ProfScope _ps(m, PROF_VMP);
    if (ct == 2) fft64_vmp_kernel<2><<<dim3((p.m2 + 127) / 128, (ncols_out + 1) / 2, batch), block, 0, m->stream>>>(p);
    else fft64_vmp_kernel<4><<<dim3((p.m2 + 127) / 128, (ncols_out + 3) / 4, batch), block, 0, m->stream>>>(p);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

enum { FEW_ADD = 0, FEW_SUB = 1, FEW_NEG = 2, FEW_MUL = 5 };
struct FEwArgs {
    LimbSet dst, a, b;
    uint32_t m;
};
template <int OP> __global__ void __launch_bounds__(256) fft64_ew_kernel(FEwArgs p) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; // complex index
    if (i >= p.m) return;
    const uint32_t j = blockIdx.y, b = blockIdx.z;
    double *dst = reinterpret_cast<double *>(p.dst.base + (size_t)b * p.dst.batch_stride + (size_t)j * p.dst.limb_stride);
    const double *a = reinterpret_cast<const double *>(p.a.base + (size_t)b * p.a.batch_stride + (size_t)j * p.a.limb_stride);
    const double ar = a[i], ai = a[i + p.m];
    if (OP == FEW_NEG) {
        dst[i] = -ar;
        dst[i + p.m] = -ai;
        return;
    }
    const double *bb = reinterpret_cast<const double *>(p.b.base + (size_t)b * p.b.batch_stride + (size_t)j * p.b.limb_stride);
    const double br = bb[i], bi = bb[i + p.m];
    if (OP == FEW_ADD) {
        dst[i] = ar + br;
        dst[i + p.m] = ai + bi;
    } else if (OP == FEW_SUB) {
        dst[i] = ar - br;
        dst[i + p.m] = ai - bi;
    } else {
        dst[i] = ar * br - ai * bi;
        dst[i + p.m] = ar * bi + ai * br;
    }
}
int fft64_ew(pgb_module *m, int op, LimbSet dst, LimbSet a, LimbSet b, uint32_t jobs, uint32_t batch) {
    if (jobs == 0 || batch == 0) return PGB_OK;
    ProfScope _ps(m, PROF_ELEMENTWISE);
    FEwArgs p = {dst, a, b, (uint32_t)(m->n / 2)};
    dim3 block(256), grid((p.m + 255) / 256, jobs, batch);
    switch (op) {
    case FEW_ADD: fft64_ew_kernel<FEW_ADD><<<grid, block, 0, m->stream>>>(p); break;
    case FEW_SUB: fft64_ew_kernel<FEW_SUB><<<grid, block, 0, m->stream>>>(p); break;
    case FEW_NEG: fft64_ew_kernel<FEW_NEG><<<grid, block, 0, m->stream>>>(p); break;
    default: fft64_ew_kernel<FEW_MUL><<<grid, block, 0, m->stream>>>(p); break;
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}
