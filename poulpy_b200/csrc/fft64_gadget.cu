// fft64_gadget.cu -- the whole gadget product (GLWE key-switch / GGSW x GLWE external product, dsize = 1, same base2k) of the FFT64
// flavour as ONE persistent kernel: i64 GLWE in -> i64 GLWE out, nothing else touches HBM (the prepared key streams from L2).
//
// Restates, per ciphertext, the HAL sequence of poulpy-core/src/keyswitching/glwe.rs:207-239,106-108 and
// external_product/glwe.rs:197-271,138-140 on the FFT64 backend:
//     vec_znx_dft_apply (R limbs; reference/fft64/vec_znx_dft.rs:160-200)
//  -> vmp_apply_dft_to_dft (fft64/vmp.rs:144-264, rows accumulated in row order)
//  -> vec_znx_idft_apply_consume (vec_znx_dft.rs:264-288: x 1/m, round half away from zero)
//  -> vec_znx_big_add_small_assign (fft64/vec_znx_big.rs, wrapping i64)
//  -> vec_znx_big_normalize, same base2k, offset 0 (reference/vec_znx/normalize.rs:52-148 with the i64 steps of
//     reference/znx/normalization.rs:24-323)
// Unlike the NTT120 kernel there is no collapsed key: f64 cannot hold the 2^((S-1)K) spread, so every output limb gets its own
// inverse transform and the rounded limbs are chained by the carry exactly like the unfused sequence.
//
// Mapping: one CTA owns one ciphertext at a time (persistent loop).  A transform of m = n/2 complex points is run by a "slot" of
// T = m/8 threads (radix-8 passes through padded shared memory, FMA butterflies, as in fft64.cu); the CTA holds NS = cols_out * LPR
// slots.  The R forward transforms stay resident in R shared-memory planes.  In the last forward pass and the first inverse pass a
// thread owns the same eight frequencies, so the key products need no barrier: thread t of a slot multiplies rows x key for
// frequencies 8t..8t+7 in registers and walks straight into the inverse passes.  Slot s serves output column s % cols_out; the LPR
// slots of a column take LPR consecutive limbs per round and hand their rounded i64 coefficients to the column's carry chain
// (registers when LPR == 1, the slot's own plane + a named barrier otherwise).
#include <stdlib.h>

#include "internal.h"
#include "fft64.cuh"

namespace {

struct FGadgetArgs {
    const char *in;  unsigned long long in_bs;   // GLWE inputs (i64), limb (j, col) at ((j * in_cols + col) * n) words
    char *res;       unsigned long long res_bs;  // GLWE outputs (i64), limb (j, col) at ((j * cols_out + col) * n) words
    const double *pmat;                          // key in the kernel's layout (fft64_gadget_key_kernel): [row][C][re | im][q][t] double2
    const double2 *twl_f, *twl_i;                // last forward / first inverse pass twiddles, [7][T]: thread t's seven values, coalesced
    int in_cols, row_cols, row_col0, R, C, cols_out;
    int small_size;                              // limbs of input column 0 added to output column 0 (key-switch), 0 = none
    int K, S, res_size, batch;
    // input poly r (limb r / row_cols) multiplies key row src_row[r] with its limbs shifted by di[r], into output limbs j < jmax[r] only
    // (dsize == 1: src_row = r, di = 0, jmax = S; dsize == 2: the digit groups of keyswitching/glwe.rs:332-379, see fft64_gadget_fused)
    signed char src_row[16], di[16], jmax[16];
    double inv_m;
    // automorphism epilogue (AUT instances only): the coefficient at source position j goes to j * aut_p mod 2n (negated when that lands
    // in [n, 2n)).  x = rounded product + body.  mode 1: res = normalize(aut(x) + a), 2: normalize(aut(x) - a), 3: normalize(a - aut(x)),
    // a = the first post_size limbs of the INPUT ciphertext, every column (automorphism/glwe_ct.rs:95-275: big_automorphism,
    // big_(add|sub)_small, big_normalize); mode 4: res = aut(normalize(x)) (glwe_automorphism, glwe_ct.rs:51-72)
    int aut_mode, post_size;
    uint32_t aut_p;
};

// one coefficient of the automorphism epilogue: v = rounded product (+ body already added) at source position js of limb j, column c
__device__ __forceinline__ void aut_emit(const FGadgetArgs &p, long long v, long long &carry, int K, int N, int js, const long long *post_limb,
                                         long long *out_limb, bool store) {
    const uint32_t e = ((uint32_t)js * p.aut_p) & (uint32_t)(2 * N - 1);
    const int jo = (int)(e & (uint32_t)(N - 1));
    const bool flip = e >= (uint32_t)N;
    const int mode = p.aut_mode;
    unsigned long long x = (unsigned long long)v;
    if (mode != 4) {
        if ((mode == 3) != flip) x = 0ull - x;
        if (post_limb) {
            const unsigned long long a = (unsigned long long)__ldg(post_limb + jo);
            x = mode == 2 ? x - a : x + a;
        }
    }
    long long o = norm_step((long long)x, carry, K);
    if (mode == 4 && flip) o = (long long)(0ull - (unsigned long long)o);
    if (store) out_limb[jo] = o;
}

template <int T> __device__ __forceinline__ void slot_sync(int slot) {
    if (T <= 32) __syncwarp();
    else asm volatile("bar.sync %0, %1;" ::"r"(slot + 1), "r"(T) : "memory");
}
__device__ __forceinline__ void prefetch_l2_bulk(const void *gptr, uint32_t bytes) { // bytes: multiple of 16
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gptr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void group_sync(int id, int threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }

template <int L, int L0, bool TWS> struct GFwd {
    static __device__ __forceinline__ void run(double2 *buf, const double2 *tw, const double2 *twl, int t, int slot) {
        constexpr int SL = L - L0 - 3;
        const int a = t >> SL, b = t & ((1 << SL) - 1), base = (a << (SL + 3)) | b;
        double2 x[8];
#pragma unroll
        for (int j = 0; j < 8; j++) x[j] = buf[FPAD(base + (j << SL))];
        if (SL == 0) {
            double2 w[7];
            load_tw7(w, twl, FGeo<L>::T, t);
            fct_radix8_w(x, w);
        } else {
            fct_radix8<3, TWS>(x, tw, (1u << L0) | (uint32_t)a);
        }
#pragma unroll
        for (int j = 0; j < 8; j++) buf[FPAD(base + (j << SL))] = x[j];
        if (SL > 0) slot_sync<FGeo<L>::T>(slot); // after the last pass every thread only re-reads its own eight values
        GFwd<L, (L0 + 3 < L) ? L0 + 3 : L, TWS>::run(buf, tw, twl, t, slot);
    }
};
template <int L, bool TWS> struct GFwd<L, L, TWS> {
    static __device__ __forceinline__ void run(double2 *, const double2 *, const double2 *, int, int) {}
};
template <int L, int L0, bool TWS> struct GInv {
    static __device__ __forceinline__ void run(double2 *buf, const double2 *tw, int t, int slot) {
        typedef FGeo<L> G;
        constexpr int SL = L - L0 - 3;
        const int a = t >> SL, b = t & ((1 << SL) - 1), base = (a << (SL + 3)) | b;
        double2 x[8];
#pragma unroll
        for (int j = 0; j < 8; j++) x[j] = buf[FPAD(base + (j << SL))];
        fgs_radix8<3, TWS>(x, tw, (1u << L0) | (uint32_t)a);
#pragma unroll
        for (int j = 0; j < 8; j++) buf[FPAD(base + (j << SL))] = x[j];
        slot_sync<G::T>(slot);
        GInv<L, (L0 - 3 >= G::R0) ? L0 - 3 : -1, TWS>::run(buf, tw, t, slot);
    }
};
template <int L, bool TWS> struct GInv<L, -1, TWS> {
    static __device__ __forceinline__ void run(double2 *, const double2 *, int, int) {}
};


template <int LM, int LPR, bool TWS, bool AUT> __global__ void __launch_bounds__(512, 1)
fft64_gadget_kernel(const __grid_constant__ FGadgetArgs p, const double2 *__restrict__ twf_g, const double2 *__restrict__ twi_g) {
    typedef FGeo<LM> G;
    constexpr int M = 1 << LM, N = 2 * M, T = G::T, PL = G::PLANE;
    constexpr int CPT = 16 / LPR; // coefficients of a column per thread of its slot group
    static_assert(LM > G::R0 && T >= 32 && (16 % LPR) == 0, "geometry");
    extern __shared__ __align__(16) double2 gsm[];
    const int cols_out = p.cols_out, NS = cols_out * LPR, R = p.R, S = p.S, K = p.K;
    const int slot = threadIdx.x / T, t = threadIdx.x % T;
    const int c = slot % cols_out, g = slot / cols_out; // output column and position inside the column's slot group
    double2 *planes = gsm;                               // R resident forward transforms
    double2 *work = gsm + (size_t)(R + slot) * PL;       // this slot's inverse-transform plane
    const double2 *twf = twf_g, *twi = twi_g;
    if (TWS) {
        double2 *tws = gsm + (size_t)(R + NS) * PL;
        for (int i = threadIdx.x; i < M; i += blockDim.x) {
            tws[i] = twf_g[i];
            tws[M + i] = twi_g[i];
        }
        twf = tws;
        twi = tws + M;
        __syncthreads();
    }
    const int a_start = p.res_size < S ? p.res_size : S; // limbs j >= a_start are carry-only
    const size_t res_ls = (size_t)cols_out * N, in_ls = (size_t)p.in_cols * N;
    const int nrounds = (S + LPR - 1) / LPR;
    const int gt = g * T + t, GT = LPR * T;

    for (int ct = blockIdx.x; ct < p.batch; ct += gridDim.x) {
        const long long *in = reinterpret_cast<const long long *>(p.in + (size_t)ct * p.in_bs);
        long long *res = reinterpret_cast<long long *>(p.res + (size_t)ct * p.res_bs);
        // L2 prefetch (TMA bulk prefetch, one thread per 8n-byte limb): the mask limbs of this CTA's next ciphertext and the body limbs
        // this one needs in its carry chain
        if ((int)threadIdx.x < R + p.small_size) {
            const int u = threadIdx.x;
            if (u < p.small_size) {
                prefetch_l2_bulk(in + (size_t)u * in_ls, N * 8);
            } else if (ct + (int)gridDim.x < p.batch) {
                const int r = u - p.small_size, limb = r / p.row_cols, col = r % p.row_cols + p.row_col0;
                prefetch_l2_bulk(in + (size_t)gridDim.x * (p.in_bs / 8) + ((size_t)limb * p.in_cols + col) * N, N * 8);
            }
        }
        // ---- forward transforms of the R input limbs ------------------------------------------------------------------------------
        for (int r = slot; r < R; r += NS) {
            const int limb = r / p.row_cols, col = r % p.row_cols + p.row_col0;
            const long long *src = in + ((size_t)limb * p.in_cols + col) * N;
            double2 *buf = planes + (size_t)r * PL;
            double2 x[8];
#pragma unroll
            for (int jj = 0; jj < 8; jj++) {
                const int idx = t + jj * T;
                x[jj] = make_double2((double)__ldg(src + idx), (double)__ldg(src + idx + M)); // reim_from_znx_i64 (conversion.rs:19-28)
            }
            fct_radix8<G::R0, TWS>(x, twf, 1u);
#pragma unroll
            for (int jj = 0; jj < 8; jj++) buf[FPAD(t + jj * T)] = x[jj];
            slot_sync<T>(slot);
            GFwd<LM, G::R0, TWS>::run(buf, twf, p.twl_f, t, slot);
        }
        __syncthreads(); // the products read every plane
        // ---- output limbs, least significant first: products -> inverse transform -> round -> carry chain ------------------------------
        long long carry[CPT];
#pragma unroll
        for (int i = 0; i < CPT; i++) carry[i] = 0;
        for (int k = 0; k < nrounds; k++) {
            const int jl = k * LPR + g, j = S - 1 - jl;
            const bool valid = jl < S;
            double2 x[8];
            if (valid) {
#pragma unroll
                for (int jj = 0; jj < 8; jj++) x[jj] = make_double2(0.0, 0.0);
                const double2 *kp = reinterpret_cast<const double2 *>(p.pmat) + t; // + key poly index * M
                // rows accumulate in row order (reim4_add_mul, reim4/arithmetic_ref.rs:223-232), FMA-contracted; the key values come from L2
                // in the kernel's own layout: load q of a warp covers 512 contiguous bytes
                for (int r = 0; r < R; r++) {
                    if (j >= p.jmax[r]) continue; // CTA-uniform per slot: this input limb does not reach output limb j
                    const double2 *kr = kp + ((size_t)p.src_row[r] * p.C + (size_t)(j + p.di[r]) * cols_out + c) * M, *ki = kr + M / 2;
                    double br[8], bi[8];
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        const double2 u = __ldg(kr + q * T), v = __ldg(ki + q * T);
                        br[2 * q] = u.x; br[2 * q + 1] = u.y; bi[2 * q] = v.x; bi[2 * q + 1] = v.y;
                    }
                    const double2 *ap = planes + (size_t)r * PL;
#pragma unroll
                    for (int jj = 0; jj < 8; jj++) {
                        const double2 a = ap[FPAD(8 * t + jj)];
                        x[jj].x = fma(a.x, br[jj], x[jj].x); x[jj].x = fma(-a.y, bi[jj], x[jj].x);
                        x[jj].y = fma(a.x, bi[jj], x[jj].y); x[jj].y = fma(a.y, br[jj], x[jj].y);
                    }
                }
                {
                    double2 w[7];
                    load_tw7(w, p.twl_i, T, t);
                    fgs_radix8_w(x, w);
                }
#pragma unroll
                for (int jj = 0; jj < 8; jj++) work[FPAD(8 * t + jj)] = x[jj];
                slot_sync<T>(slot);
                GInv<LM, (LM - 6 >= G::R0) ? LM - 6 : -1, TWS>::run(work, twi, t, slot);
#pragma unroll
                for (int jj = 0; jj < 8; jj++) x[jj] = work[FPAD(t + jj * T)];
                if (LPR == 1) slot_sync<T>(slot); // the next round's products overwrite the plane (write-after-read found by racecheck)
                fgs_radix8<G::R0, TWS>(x, twi, 1u);
            }
            if (LPR == 1) {
                // the thread that produced a coefficient also owns its carry: no shared-memory round trip
                if (valid) {
                    const bool with_small = c == 0 && j < p.small_size;
                    const long long *sp = in + (size_t)j * in_ls + t; // input column 0 (the body)
                    long long *op = res + (size_t)j * res_ls + (size_t)c * N + t;
#pragma unroll
                    for (int jj = 0; jj < 8; jj++) {
                        long long v0 = (long long)round(x[jj].x * p.inv_m), v1 = (long long)round(x[jj].y * p.inv_m); // conversion.rs:43-52
                        if (with_small) {
                            v0 = (long long)((unsigned long long)v0 + (unsigned long long)__ldg(sp + jj * T));
                            v1 = (long long)((unsigned long long)v1 + (unsigned long long)__ldg(sp + jj * T + M));
                        }
                        if constexpr (AUT) {
                            const long long *post = j < p.post_size ? in + (size_t)j * in_ls + (size_t)c * N : nullptr;
                            long long *ol = res + (size_t)j * res_ls + (size_t)c * N;
                            aut_emit(p, v0, carry[2 * jj], K, N, t + jj * T, post, ol, j < a_start);
                            aut_emit(p, v1, carry[2 * jj + 1], K, N, t + jj * T + M, post, ol, j < a_start);
                        } else {
                        const long long o0 = norm_step(v0, carry[2 * jj], K), o1 = norm_step(v1, carry[2 * jj + 1], K);
                        if (j < a_start) {
                            op[jj * T] = o0;
                            op[jj * T + M] = o1;
                        }
                        }
                    }
                }
            } else {
                if (valid) {
                    slot_sync<T>(slot); // the last pass has read its inputs: the plane now takes the rounded i64 coefficients
                    long long *big = reinterpret_cast<long long *>(work);
#pragma unroll
                    for (int jj = 0; jj < 8; jj++) {
                        big[t + jj * T] = (long long)round(x[jj].x * p.inv_m);
                        big[t + jj * T + M] = (long long)round(x[jj].y * p.inv_m);
                    }
                }
                group_sync(8 + c, GT);
                // the LPR * T threads of the column's group split its n coefficients and walk this round's limbs in order
                for (int l = 0; l < LPR; l++) {
                    const int j2 = S - 1 - (k * LPR + l);
                    if (j2 < 0) break;
                    const long long *big = reinterpret_cast<const long long *>(gsm + (size_t)(R + c + l * cols_out) * PL);
                    const bool with_small = c == 0 && j2 < p.small_size;
                    const long long *sp = in + (size_t)j2 * in_ls + gt;
                    long long *op = res + (size_t)j2 * res_ls + (size_t)c * N + gt;
#pragma unroll
                    for (int i = 0; i < CPT; i++) {
                        long long v = big[gt + i * GT];
                        if (with_small) v = (long long)((unsigned long long)v + (unsigned long long)__ldg(sp + i * GT));
                        if constexpr (AUT) {
                            const long long *post = j2 < p.post_size ? in + (size_t)j2 * in_ls + (size_t)c * N : nullptr;
                            aut_emit(p, v, carry[i], K, N, gt + i * GT, post, res + (size_t)j2 * res_ls + (size_t)c * N, j2 < a_start);
                        } else {
                        const long long o = norm_step(v, carry[i], K);
                        if (j2 < a_start) op[i * GT] = o;
                        }
                    }
                }
                group_sync(8 + c, GT); // the planes are rewritten by the next round
            }
        }
        // limbs beyond the key size are zero (normalize.rs:60-66)
        if (p.res_size > a_start) {
            if (LPR == 1) {
                for (int j = a_start; j < p.res_size; j++) {
                    long long *op = res + (size_t)j * res_ls + (size_t)c * N + t;
#pragma unroll
                    for (int jj = 0; jj < 8; jj++) {
                        op[jj * T] = 0;
                        op[jj * T + M] = 0;
                    }
                }
            } else {
                for (int j = a_start; j < p.res_size; j++) {
                    long long *op = res + (size_t)j * res_ls + (size_t)c * N + gt;
#pragma unroll
                    for (int i = 0; i < CPT; i++) op[i * GT] = 0;
                }
            }
        }
        __syncthreads(); // the next ciphertext's forward transforms overwrite the planes
    }
}

// key re-layout: out[(r * C + p)][part][q][t] (double2) = in[(r * C + p)][part][8t + 2q, 8t + 2q + 1], part = re / im
__global__ void __launch_bounds__(256) fft64_gadget_key_kernel(const double *__restrict__ in, double2 *__restrict__ out, int M, int polys) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x; // output double2 index inside one half poly: q * T + t
    const int T = M / 8;
    if (i >= M / 2) return;
    const int q = i / T, t = i % T;
    const size_t poly = blockIdx.y;
    const double *src = in + poly * 2 * (size_t)M + (size_t)blockIdx.z * M + 8 * t + 2 * q;
    out[poly * (size_t)M + (size_t)blockIdx.z * (M / 2) + i] = make_double2(src[0], src[1]);
    (void)polys;
}
template <int LM, int LPR, bool TWS, bool AUT> int launch_a(pgb_module *m, const FGadgetArgs &p, size_t smem) {
    static int sms_dev[32] = {};
    int &sms = sms_dev[m->device & 31];
    if (!sms) {
        PGB_CHECK_CUDA(cudaFuncSetAttribute(fft64_gadget_kernel<LM, LPR, TWS, AUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(227 << 10)));
        PGB_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, m->device));
    }
    const int threads = p.cols_out * LPR * FGeo<LM>::T;
    const int grid = p.batch < sms ? p.batch : sms;
    { ProfScope _ps(m, PROF_GADGET);
    fft64_gadget_kernel<LM, LPR, TWS, AUT><<<grid, threads, smem, m->stream>>>(p, m->fft_fwd, m->fft_inv);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}
template <int LM, int LPR, bool TWS> int launch(pgb_module *m, const FGadgetArgs &p, size_t smem) {
    return p.aut_mode ? launch_a<LM, LPR, TWS, true>(m, p, smem) : launch_a<LM, LPR, TWS, false>(m, p, smem);
}
template <int LM> int launch_lm(pgb_module *m, const FGadgetArgs &p, int lpr, bool tws, size_t smem) {
    if (tws) {
        switch (lpr) {
        case 1: return launch<LM, 1, true>(m, p, smem);
        case 2: return launch<LM, 2, true>(m, p, smem);
        default: return launch<LM, 4, true>(m, p, smem);
        }
    }
    switch (lpr) {
    case 1: return launch<LM, 1, false>(m, p, smem);
    case 2: return launch<LM, 2, false>(m, p, smem);
    default: return launch<LM, 4, false>(m, p, smem);
    }
}

// slots per column (limbs in flight per round), whether the twiddles fit in shared memory next to the planes, bytes of shared memory
bool plan(const pgb_module *m, int R, int cols_out, int S, int *lpr_out, bool *tws_out, size_t *smem_out) {
    const size_t M = m->n / 2, T = M / 8, PL = M + (M >> 3) + 2;
    const size_t cap = (size_t)227 << 10, tw_bytes = 2 * M * sizeof(double2);
    for (int lpr = 4; lpr >= 1; lpr >>= 1) {
        if ((size_t)cols_out * lpr * T > 512 || (lpr > 1 && lpr > 2 * S)) continue;
        if (cols_out * lpr > 7) continue; // named barriers 1..7 are the slots', 8..11 the column groups'
        const size_t planes = (size_t)(R + cols_out * lpr) * PL * sizeof(double2);
        if (planes > cap) continue;
        *lpr_out = lpr;
        *tws_out = planes + tw_bytes <= cap;
        *smem_out = planes + (*tws_out ? tw_bytes : 0);
        return true;
    }
    return false;
}

} // namespace

bool fft64_gadget_supported(const pgb_module *m, int R, int cols_out, int S, int base2k, int batch) {
    if (m->flavour != PGB_FFT64 || m->log_n < 9 || m->log_n > 12) return false;
    if (opt_on(m, PGB_OPT_NO_GADGET)) return false;
    // FGadgetArgs holds the row tables of at most 16 input polys
    if (cols_out < 1 || cols_out > 4 || R < 1 || R > 16 || S < 1 || base2k < 1 || base2k > 63 || batch < 1) return false;
    int lpr;
    bool tws;
    size_t smem;
    return plan(m, R, cols_out, S, &lpr, &tws, &smem);
}

// dsize == 2: R = a_size * row_cols input polys in their natural order, `key_rows` = rows * cols_in of the key, `group_limit` = bound on
// the limbs of a digit group (dnum for the key-switch, 0 = none for the external product); the row mapping is the one of
// ntt120_gadget_fused.  (dsize >= 3 is not offered: there the reference's FFT64 vmp leaves stale limbs in its temporary, fft64/vmp.rs:263.)
int fft64_gadget_fused(pgb_module *m, const char *in, uint64_t in_bs, int in_cols, int row_cols, int row_col0, int R, const char *pmat, int C,
                       int cols_out, int small_size, char *res, uint64_t res_bs, int res_size, int base2k, int batch, int dsize, int a_size,
                       int key_rows, int group_limit, int aut_mode, int64_t aut_p, int post_size) {
    FGadgetArgs p;
    memset(&p, 0, sizeof p);
    p.aut_mode = aut_mode;
    p.post_size = post_size;
    if (aut_mode) {
        const int64_t two_n = 2 * (int64_t)m->n;
        p.aut_p = (uint32_t)(((aut_p % two_n) + two_n) % two_n);
        if (!(p.aut_p & 1)) {
            pgb_set_error("fft64 gadget kernel: automorphism index must be odd");
            return PGB_ERR_SHAPE;
        }
    }
    if (dsize < 1) dsize = 1;
    if (dsize == 1) key_rows = R;
    if (R > 16) {
        pgb_set_error("fft64 gadget kernel: more than 16 input polys");
        return PGB_ERR_UNSUPPORTED;
    }
    for (int r = 0; r < R; r++) {
        const int S = C / cols_out;
        if (dsize == 1) {
            p.src_row[r] = (signed char)r; p.di[r] = 0; p.jmax[r] = (signed char)S;
            continue;
        }
        const int l = r / row_cols, ci = r % row_cols, di = dsize - 1 - l % dsize, jl = l / dsize;
        int group = (a_size + di) / dsize;
        if (group_limit > 0 && group > group_limit) group = group_limit;
        const int src = jl * row_cols + ci;
        const int cut = dsize - di - 2, size_di = S - (cut > 0 ? cut : 0);
        int jm = S - di < size_di ? S - di : size_di;
        if (jl >= group || src >= key_rows || jm < 0) jm = 0;
        p.src_row[r] = (signed char)(jm ? src : 0); p.di[r] = (signed char)(jm ? di : 0); p.jmax[r] = (signed char)jm;
    }
    p.in = in; p.in_bs = in_bs; p.res = res; p.res_bs = res_bs; p.pmat = (const double *)pmat;
    p.in_cols = in_cols; p.row_cols = row_cols; p.row_col0 = row_col0; p.R = R; p.C = C; p.cols_out = cols_out; p.small_size = small_size;
    p.K = base2k; p.S = C / cols_out; p.res_size = res_size; p.batch = batch;
    p.inv_m = 1.0 / (double)(m->n / 2);
    // workspace: the key in the kernel's layout; kept in the module's key cache for a PINNED key (pgb_gadget_key_pin)
    const uint64_t M = m->n / 2;
    const uint64_t key_bytes = (uint64_t)key_rows * C * m->n * 8;
    const uint64_t sig[KEY_SIG_WORDS] = {2, (uint64_t)key_rows, (uint64_t)C, 0, 0, 0, 0, 0, 0, 0};
    const bool pinned = key_is_pinned(m, pmat);
    double2 *kperm = pinned ? (double2 *)key_cache_find(m, pmat, sig) : nullptr;
    const bool have = kperm != nullptr;
    if (pinned && !have) PGB_TRY(key_cache_insert(m, pmat, key_bytes, sig, key_bytes + 256, (void **)&kperm));
    if (!pinned) {
        const uint64_t need = key_bytes + 256;
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
        kperm = (double2 *)m->aux_ws;
    }
    if (!have) {
        { ProfScope _ps(m, PROF_OTHER);
        fft64_gadget_key_kernel<<<dim3(((unsigned)(M / 2) + 255) / 256, key_rows * C, 2), 256, 0, m->stream>>>((const double *)pmat, kperm, (int)M, key_rows * C);
        }
        PGB_CHECK_CUDA(cudaGetLastError());
    }
    p.pmat = (const double *)kperm;
    p.twl_f = m->fft_last_f;
    p.twl_i = m->fft_last_i;
    int lpr;
    bool tws;
    size_t smem;
    if (!plan(m, R, cols_out, p.S, &lpr, &tws, &smem)) {
        pgb_set_error("fft64 gadget kernel: shape does not fit");
        return PGB_ERR_UNSUPPORTED;
    }
    switch (m->log_n) {
    case 9: return launch_lm<8>(m, p, lpr, tws, smem);
    case 10: return launch_lm<9>(m, p, lpr, tws, smem);
    case 11: return launch_lm<10>(m, p, lpr, tws, smem);
    case 12: return launch_lm<11>(m, p, lpr, tws, smem);
    default: pgb_set_error("fft64 gadget kernel: unsupported n"); return PGB_ERR_UNSUPPORTED;
    }
}
