// cggi.cu -- CGGI blind rotation (block-binary), batched and device resident (C3).
// Restates poulpy-bin-fhe/src/blind_rotation/algorithms/cggi/algorithm.rs:275-368 over the batched HAL kernels.
#include <stdlib.h>

#include "internal.h"

static inline bool R_ok(uint64_t cols, uint64_t dnum) {
    const uint64_t R = cols * dnum;
    return R == 1 || R == 2 || R == 3 || R == 4 || R == 6 || R == 8;
}

// x_pow_a[i] = svp_prepare(X^i), i in [0, 2n)  (cggi/key_prepared.rs:66-75, utils.rs:6-41 with y = 0)
__global__ void xpow_fill_kernel(long long *buf, uint32_t n) {
    const uint32_t ai = blockIdx.x; // [0, 2n)
    long long *p = buf + (size_t)ai * n;
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
        long long v = 0;
        if (ai < n) v = (i == ai) ? 1 : 0;
        else v = (i == ((ai - n) & (n - 1))) ? -1 : 0;
        p[i] = v;
    }
}
extern "C" int pgb_cggi_x_pow_a(pgb_module *m, pgb_svp_ppol *res) {
    PGB_REQUIRE(res->n == m->n && res->cols == 2 * m->n, "cggi_x_pow_a: res must be an SvpPPol with 2n columns");
    const uint64_t n = m->n, pb = prep_bytes(m);
    long long *buf = nullptr;
    PGB_CHECK_CUDA(cudaMalloc(&buf, 2 * n * n * 8));
    { ProfScope _ps(m, PROF_OTHER);
    xpow_fill_kernel<<<(unsigned)(2 * n), 256, 0, m->stream>>>(buf, (uint32_t)n);
    }
    LimbSet in = {(char *)buf, n * 8, 0}, out = {(char *)res->data, n * pb, 0};
    int s = m->flavour == PGB_NTT120 ? ntt120_forward(m, in, out, (int)(2 * n), 1) : fft64_forward(m, in, out, (int)(2 * n), 1);
    cudaStreamSynchronize(m->stream);
    cudaFree(buf);
    return s;
}

extern "C" size_t pgb_cggi_blind_rotate_tmp_bytes(const pgb_module *m, uint64_t rank, uint64_t res_size, uint64_t dnum, uint64_t brk_size,
                                                  uint64_t batch) {
    (void)res_size;
    const uint64_t n = m->n, pb = prep_bytes(m), bb = big_bytes(m), cols = rank + 1;
    uint64_t t = 0;
    t += align_up(batch * n * cols * dnum * pb);     // acc_dft
    t += align_up(batch * n * cols * brk_size * pb); // vmp_res
    t += align_up(batch * n * cols * brk_size * pb); // acc_add_dft
    t += align_up(batch * n * brk_size * pb);        // vmp_xai
    t += align_up(batch * n * brk_size * bb);        // acc_add_big
    return t + ALIGN;
}

// acc[b][col][j] = (acc + x_pow_a[a_b] * v) - v   for every column and limb: the three HAL calls of algorithm.rs:351-355
// (svp_apply_dft_to_dft into vmp_xai, vec_znx_dft_add_assign, vec_znx_dft_sub_assign) in one pass.
struct XaiArgs {
    char *acc;       uint64_t acc_bs;  // acc_add_dft polys (cols * size), batch stride
    const char *v;   uint64_t v_bs;    // vmp_res polys
    const char *xpa;                   // x_pow_a table: 2n polys of ScalarPrep
    const long long *lwe; uint64_t lwe_stride; // a_i of item b at lwe[b * lwe_stride]
    uint32_t n, polys;
};
#include "ntt120.cuh"
__global__ void __launch_bounds__(256) cggi_xai_ntt120_kernel(XaiArgs p) {
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x; // uint4 index inside a poly
    if (u >= p.n) return;
    const n120::PrimeRt pr(u / (p.n / 4));
    const uint32_t q = pr.q;
    const uint32_t b = blockIdx.z, poly = blockIdx.y;
    const long long ai = p.lwe[(size_t)b * p.lwe_stride];
    const uint32_t pos = (uint32_t)((ai + (long long)(2 * p.n)) & (long long)(2 * p.n - 1));
    const uint4 w = __ldg(reinterpret_cast<const uint4 *>(p.xpa + (size_t)pos * p.n * 16) + u);
    const uint4 v = *(reinterpret_cast<const uint4 *>(p.v + (size_t)b * p.v_bs + (size_t)poly * p.n * 16) + u);
    uint4 *ap = reinterpret_cast<uint4 *>(p.acc + (size_t)b * p.acc_bs + (size_t)poly * p.n * 16) + u;
    const uint4 a = *ap;
    auto f = [&](uint32_t acc, uint32_t ww, uint32_t vv) {
        uint32_t pv = pr.reduce((unsigned long long)ww * vv);
        uint32_t t = n120::csub(acc + pv, q);
        return t >= vv ? t - vv : t - vv + q;
    };
    *ap = make_uint4(f(a.x, w.x, v.x), f(a.y, w.y, v.y), f(a.z, w.z, v.z), f(a.w, w.w, v.w));
}
// One launch per block of `bs` LWE coefficients (NTT120): acc_add[c] = sum_t ( x_pow_a[a_t] * v_t[c] - v_t[c] ),  v_t[c] = sum_r acc_dft[r] * BRK_t[r][c],
// i.e. the bs x (vmp_apply_dft_to_dft + svp_apply_dft_to_dft + dft_add_assign + dft_sub_assign) of algorithm.rs:338-357 with the C partial sums
// in registers: the limb-wise sequence moves 864 KB per ciphertext and block through HBM at the bench shape, this kernel 96 KB.  Every
// intermediate is canonical, so the result is bit-identical to the per-key kernels (ntt120_vmp_kernel + cggi_xai_ntt120_kernel).
struct BlockArgs {
    const char *acc_dft; uint64_t acc_bs;   // R polys per ciphertext
    char *acc_add;       uint64_t add_bs;   // C polys per ciphertext (written, not accumulated)
    const char *brk;     uint64_t brk_bytes; // key of LWE coefficient i at brk + i * brk_bytes, layout [r][c] polys
    const char *xpa;
    const long long *lwe; uint64_t lwe_stride; // a_{blk + t} of item b at lwe[b * lwe_stride + t]
    uint32_t n, R, C, bs;
};
// BT ciphertexts per thread: a key word loaded from L2 serves all of them (with one ciphertext per thread every CTA re-read the block's
// 786 KB of key: 6.6 TB/s of L2 traffic at the bench shape, the limiter of the first version)
// SM = 1: the block's inputs a[i][r] and the table values w[i][t] sit in thread-private shared-memory slots instead of registers
// (162 registers allowed one CTA of eight warps per SM: latency bound); SM = 0: registers / L2 (shapes whose staging does not fit)
template <int RMAX, int BT, int SM> __global__ void __launch_bounds__(256, SM ? 2 : 1) cggi_block_ntt120_kernel(BlockArgs p, uint32_t batch) {
    extern __shared__ __align__(16) uint4 bsm[];
    uint4 *asm_ = bsm + threadIdx.x;                                 // a slot (i * RMAX + r) at asm_[(i * RMAX + r) * 256]
    uint4 *wsm = bsm + (size_t)BT * RMAX * 256;                      // w slot [(i * bs + t) * 256 + tid]
    constexpr int w_in_smem = SM;
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x; // uint4 index inside a poly
    if (u >= p.n) return;
    const n120::PrimeRt pr(u / (p.n / 4));
    const uint32_t q = pr.q, b0 = blockIdx.z * BT;
    const size_t poly = (size_t)p.n; // uint4 per poly
    uint4 a[SM ? 1 : BT][SM ? 1 : RMAX]; // SM = 0: the block's inputs stay in registers for all bs x C products
    uint32_t pos[BT];
#pragma unroll
    for (int i = 0; i < BT; i++) {
        const uint32_t b = b0 + i < batch ? b0 + i : batch - 1; // the tail repeats the last ciphertext (its stores are skipped)
        const uint4 *ap = reinterpret_cast<const uint4 *>(p.acc_dft + (size_t)b * p.acc_bs) + u;
#pragma unroll
        for (int r = 0; r < RMAX; r++) {
            const uint4 v = r < (int)p.R ? __ldg(ap + (size_t)r * poly) : make_uint4(0, 0, 0, 0);
            if (SM) asm_[(i * RMAX + r) * 256] = v;
            else a[SM ? 0 : i][SM ? 0 : r] = v;
        }
    }
    if (w_in_smem) { // the table values do not depend on the output poly: without this every one of the C passes re-read them from L2
        for (uint32_t t = 0; t < p.bs; t++)
#pragma unroll
            for (int i = 0; i < BT; i++) {
                const uint32_t b = b0 + i < batch ? b0 + i : batch - 1;
                const long long ai = p.lwe[(size_t)b * p.lwe_stride + t];
                const uint32_t ps = (uint32_t)((ai + (long long)(2 * p.n)) & (long long)(2 * p.n - 1));
                const uint4 w = __ldg(reinterpret_cast<const uint4 *>(p.xpa + (size_t)ps * p.n * 16) + u);
                wsm[(i * p.bs + t) * 256 + threadIdx.x] =
                    make_uint4(w.x ? w.x - 1 : q - 1, w.y ? w.y - 1 : q - 1, w.z ? w.z - 1 : q - 1, w.w ? w.w - 1 : q - 1); // w - 1 mod q
            }
    }
    // (s + w v) - v = s + (w - 1) v (mod q): the bs updates of one output poly accumulate as u64 products of (w - 1) in [0, q) and a lazy
    // v in [0, 2q) (each < 2^61, bs <= 8), reduced once -- same canonical result as the per-key kernels, half the instructions
    auto lazy = [&](unsigned long long x) { // any u64 -> [0, 2q)
        const uint32_t hi = (uint32_t)(x >> 32), lo = (uint32_t)x;
        return n120::csub(n120::mul_shoup(hi, pr.c32, pr.c32s, q) + (lo - (lo >> 30) * q), 2 * q);
    };
    for (uint32_t c = 0; c < p.C; c++) {
        unsigned long long acc[BT][4];
#pragma unroll
        for (int i = 0; i < BT; i++) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0;
        for (uint32_t t = 0; t < p.bs; t++) {
            const uint4 *key = reinterpret_cast<const uint4 *>(p.brk + (size_t)t * p.brk_bytes) + u + (size_t)c * poly;
            uint4 mv[RMAX];
#pragma unroll
            for (int r = 0; r < RMAX; r++) mv[r] = r < (int)p.R ? __ldg(key + (size_t)r * p.C * poly) : make_uint4(0, 0, 0, 0);
            if (!w_in_smem) {
#pragma unroll
                for (int i = 0; i < BT; i++) {
                    const uint32_t b = b0 + i < batch ? b0 + i : batch - 1;
                    const long long ai = p.lwe[(size_t)b * p.lwe_stride + t];
                    pos[i] = (uint32_t)((ai + (long long)(2 * p.n)) & (long long)(2 * p.n - 1));
                }
            }
#pragma unroll
            for (int i = 0; i < BT; i++) {
                uint4 w;
                if (w_in_smem) {
                    w = wsm[(i * p.bs + t) * 256 + threadIdx.x];
                } else {
                    w = __ldg(reinterpret_cast<const uint4 *>(p.xpa + (size_t)pos[i] * p.n * 16) + u);
                    w = make_uint4(w.x ? w.x - 1 : q - 1, w.y ? w.y - 1 : q - 1, w.z ? w.z - 1 : q - 1, w.w ? w.w - 1 : q - 1); // w - 1 mod q
                }
                unsigned long long s0 = 0, s1 = 0, s2 = 0, s3 = 0;
#pragma unroll
                for (int r = 0; r < RMAX; r++) { // R <= 16: the u64 sums cannot overflow (ntt120_vmp_kernel reduces every 16 rows)
                    const uint4 av = SM ? asm_[(i * RMAX + r) * 256] : a[SM ? 0 : i][SM ? 0 : r];
                    s0 += (unsigned long long)av.x * mv[r].x; s1 += (unsigned long long)av.y * mv[r].y;
                    s2 += (unsigned long long)av.z * mv[r].z; s3 += (unsigned long long)av.w * mv[r].w;
                }
                acc[i][0] += (unsigned long long)w.x * lazy(s0); acc[i][1] += (unsigned long long)w.y * lazy(s1);
                acc[i][2] += (unsigned long long)w.z * lazy(s2); acc[i][3] += (unsigned long long)w.w * lazy(s3);
            }
        }
#pragma unroll
        for (int i = 0; i < BT; i++)
            if (b0 + i < batch)
                (reinterpret_cast<uint4 *>(p.acc_add + (size_t)(b0 + i) * p.add_bs) + u)[(size_t)c * poly] =
                    make_uint4(pr.reduce(acc[i][0]), pr.reduce(acc[i][1]), pr.reduce(acc[i][2]), pr.reduce(acc[i][3]));
    }
}
__global__ void __launch_bounds__(256) cggi_xai_fft64_kernel(XaiArgs p) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; // complex index
    const uint32_t m = p.n / 2;
    if (i >= m) return;
    const uint32_t b = blockIdx.z, poly = blockIdx.y;
    const long long ai = p.lwe[(size_t)b * p.lwe_stride];
    const uint32_t pos = (uint32_t)((ai + (long long)(2 * p.n)) & (long long)(2 * p.n - 1));
    const double *w = reinterpret_cast<const double *>(p.xpa + (size_t)pos * p.n * 8);
    const double *v = reinterpret_cast<const double *>(p.v + (size_t)b * p.v_bs + (size_t)poly * p.n * 8);
    double *a = reinterpret_cast<double *>(p.acc + (size_t)b * p.acc_bs + (size_t)poly * p.n * 8);
    const double wr = __ldg(w + i), wi = __ldg(w + i + m), vr = v[i], vi = v[i + m];
    const double pr = wr * vr - wi * vi, pi = wr * vi + wi * vr; // reim_mul(ppol, v)
    a[i] = (a[i] + pr) - vr;
    a[i + m] = (a[i + m] + pi) - vi;
}

// FFT64 counterpart of cggi_block_ntt120_kernel for the shapes the fully fused kernel (cggi_fused.cu) does not take: the key products of
// one block and their X^{a_t} - 1 updates in one launch, acc_add written once.  Per frequency the operations and their order are those
// of fft64_vmp_kernel followed by cggi_xai_fft64_kernel (v = sum_r a_r k_r in row order; acc = (acc + w v) - v, acc starting at 0), so
// the result is the limb-wise sequence's bit for bit; what disappears is vmp_res / acc_add crossing HBM 2 x block_size times.
// Thread: two consecutive complex frequencies (double2 of re, double2 of im) x CT output polys; grid (m2 / 128, C / CT, batch).
template <int CT> __global__ void __launch_bounds__(128) cggi_block_fft64_kernel(BlockArgs p) {
    const uint32_t m2 = p.n / 4; // double2 words per half poly
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= m2) return;
    const uint32_t b = blockIdx.z, c0 = blockIdx.y * CT;
    const size_t poly_words = (size_t)2 * m2;
    const int nc = min((uint32_t)CT, p.C - c0);
    const double2 *a = reinterpret_cast<const double2 *>(p.acc_dft + (size_t)b * p.acc_bs) + u;
    double2 sr[CT], si[CT];
#pragma unroll
    for (int c = 0; c < CT; c++) sr[c] = si[c] = make_double2(0.0, 0.0);
    for (uint32_t t = 0; t < p.bs; t++) {
        const long long ai = p.lwe[(size_t)b * p.lwe_stride + t];
        const uint32_t pos = (uint32_t)((ai + (long long)(2 * p.n)) & (long long)(2 * p.n - 1));
        const double2 *w = reinterpret_cast<const double2 *>(p.xpa + (size_t)pos * p.n * 8) + u;
        const double2 wr = __ldg(w), wi = __ldg(w + m2);
        const double2 *pm = reinterpret_cast<const double2 *>(p.brk + (size_t)t * p.brk_bytes) + u + (size_t)c0 * poly_words;
        double2 vr[CT], vi[CT];
#pragma unroll
        for (int c = 0; c < CT; c++) vr[c] = vi[c] = make_double2(0.0, 0.0);
        for (uint32_t r = 0; r < p.R; r++) {
            const double2 ar = __ldg(a + (size_t)r * poly_words), ai2 = __ldg(a + (size_t)r * poly_words + m2);
            const double2 *mrow = pm + (size_t)r * p.C * poly_words;
#pragma unroll
            for (int c = 0; c < CT; c++) {
                if (c < nc) {
                    const double2 br = __ldg(mrow + (size_t)c * poly_words), bi = __ldg(mrow + (size_t)c * poly_words + m2);
                    vr[c].x += ar.x * br.x - ai2.x * bi.x;
                    vr[c].y += ar.y * br.y - ai2.y * bi.y;
                    vi[c].x += ar.x * bi.x + ai2.x * br.x;
                    vi[c].y += ar.y * bi.y + ai2.y * br.y;
                }
            }
        }
#pragma unroll
        for (int c = 0; c < CT; c++) {
            const double prx = wr.x * vr[c].x - wi.x * vi[c].x, pix = wr.x * vi[c].x + wi.x * vr[c].x; // reim_mul(ppol, v)
            const double pry = wr.y * vr[c].y - wi.y * vi[c].y, piy = wr.y * vi[c].y + wi.y * vr[c].y;
            sr[c].x = (sr[c].x + prx) - vr[c].x;
            sr[c].y = (sr[c].y + pry) - vr[c].y;
            si[c].x = (si[c].x + pix) - vi[c].x;
            si[c].y = (si[c].y + piy) - vi[c].y;
        }
    }
    double2 *res = reinterpret_cast<double2 *>(p.acc_add + (size_t)b * p.add_bs) + u + (size_t)c0 * poly_words;
#pragma unroll
    for (int c = 0; c < CT; c++) {
        if (c < nc) {
            res[(size_t)c * poly_words] = sr[c];
            res[(size_t)c * poly_words + m2] = si[c];
        }
    }
}

// BT ciphertexts per thread: a key word loaded from L2 serves all of them, and the block's inputs a[bi][r] are staged once in
// thread-private shared-memory slots instead of being re-read for every LWE coefficient of the block (the one-ciphertext version moves
// 6.2 MB of key words + 1.5 MB of inputs per ciphertext and block through L2 at the circuit-bootstrapping shape: its limiter).
// Same sums in the same row order per (ciphertext, frequency, output poly) as cggi_block_fft64_kernel, with the row products FMA-contracted
// as in fft64_gadget_kernel (the f64 pipeline is exact after rounding as long as the error stays below 1/2: DESIGN section 4).
template <int CT, int BT> __global__ void __launch_bounds__(128) cggi_block_fft64_bt_kernel(BlockArgs p, uint32_t B) {
    extern __shared__ __align__(16) double2 a_s[]; // [BT][R][re | im][128]
    const uint32_t m2 = p.n / 4;
    const uint32_t tid = threadIdx.x, u = blockIdx.x * blockDim.x + tid;
    if (u >= m2) return; // no block-wide synchronisation below: every shared-memory slot belongs to one thread
    const uint32_t b0 = blockIdx.z * BT, c0 = blockIdx.y * CT;
    const int nb = min((uint32_t)BT, B - b0), nc = min((uint32_t)CT, p.C - c0);
    const size_t poly_words = (size_t)2 * m2;
#pragma unroll
    for (int bi = 0; bi < BT; bi++) {
        const double2 *a = reinterpret_cast<const double2 *>(p.acc_dft + (size_t)(b0 + (bi < nb ? bi : 0)) * p.acc_bs) + u;
        for (uint32_t r = 0; r < p.R; r++) {
            a_s[((bi * p.R + r) * 2 + 0) * 128 + tid] = __ldg(a + (size_t)r * poly_words);
            a_s[((bi * p.R + r) * 2 + 1) * 128 + tid] = __ldg(a + (size_t)r * poly_words + m2);
        }
    }
    double2 sr[BT][CT], si[BT][CT];
#pragma unroll
    for (int bi = 0; bi < BT; bi++)
#pragma unroll
        for (int c = 0; c < CT; c++) sr[bi][c] = si[bi][c] = make_double2(0.0, 0.0);
    for (uint32_t t = 0; t < p.bs; t++) {
        double2 wr[BT], wi[BT];
#pragma unroll
        for (int bi = 0; bi < BT; bi++) {
            const long long ai = p.lwe[(size_t)(b0 + (bi < nb ? bi : 0)) * p.lwe_stride + t];
            const uint32_t pos = (uint32_t)((ai + (long long)(2 * p.n)) & (long long)(2 * p.n - 1));
            const double2 *w = reinterpret_cast<const double2 *>(p.xpa + (size_t)pos * p.n * 8) + u;
            wr[bi] = __ldg(w);
            wi[bi] = __ldg(w + m2);
        }
        const double2 *pm = reinterpret_cast<const double2 *>(p.brk + (size_t)t * p.brk_bytes) + u + (size_t)c0 * poly_words;
        double2 vr[BT][CT], vi[BT][CT];
#pragma unroll
        for (int bi = 0; bi < BT; bi++)
#pragma unroll
            for (int c = 0; c < CT; c++) vr[bi][c] = vi[bi][c] = make_double2(0.0, 0.0);
        for (uint32_t r = 0; r < p.R; r++) {
            const double2 *mrow = pm + (size_t)r * p.C * poly_words;
            double2 br[CT], bim[CT];
#pragma unroll
            for (int c = 0; c < CT; c++) {
                const int cc = c < nc ? c : 0;
                br[c] = __ldg(mrow + (size_t)cc * poly_words);
                bim[c] = __ldg(mrow + (size_t)cc * poly_words + m2);
            }
#pragma unroll
            for (int bi = 0; bi < BT; bi++) {
                const double2 ar = a_s[((bi * p.R + r) * 2 + 0) * 128 + tid], ai2 = a_s[((bi * p.R + r) * 2 + 1) * 128 + tid];
#pragma unroll
                for (int c = 0; c < CT; c++) {
                    // rows accumulate in row order, FMA-contracted like fft64_gadget_kernel (reim4_add_mul): 4 instead of 6 FP64 instructions
                    vr[bi][c].x = fma(ar.x, br[c].x, vr[bi][c].x); vr[bi][c].x = fma(-ai2.x, bim[c].x, vr[bi][c].x);
                    vr[bi][c].y = fma(ar.y, br[c].y, vr[bi][c].y); vr[bi][c].y = fma(-ai2.y, bim[c].y, vr[bi][c].y);
                    vi[bi][c].x = fma(ar.x, bim[c].x, vi[bi][c].x); vi[bi][c].x = fma(ai2.x, br[c].x, vi[bi][c].x);
                    vi[bi][c].y = fma(ar.y, bim[c].y, vi[bi][c].y); vi[bi][c].y = fma(ai2.y, br[c].y, vi[bi][c].y);
                }
            }
        }
#pragma unroll
        for (int bi = 0; bi < BT; bi++)
#pragma unroll
            for (int c = 0; c < CT; c++) {
                const double2 v_r = vr[bi][c], v_i = vi[bi][c];
                const double prx = wr[bi].x * v_r.x - wi[bi].x * v_i.x, pix = wr[bi].x * v_i.x + wi[bi].x * v_r.x; // reim_mul(ppol, v)
                const double pry = wr[bi].y * v_r.y - wi[bi].y * v_i.y, piy = wr[bi].y * v_i.y + wi[bi].y * v_r.y;
                sr[bi][c].x = (sr[bi][c].x + prx) - v_r.x;
                sr[bi][c].y = (sr[bi][c].y + pry) - v_r.y;
                si[bi][c].x = (si[bi][c].x + pix) - v_i.x;
                si[bi][c].y = (si[bi][c].y + piy) - v_i.y;
            }
    }
#pragma unroll
    for (int bi = 0; bi < BT; bi++) {
        if (bi >= nb) break;
        double2 *res = reinterpret_cast<double2 *>(p.acc_add + (size_t)(b0 + bi) * p.add_bs) + u + (size_t)c0 * poly_words;
#pragma unroll
        for (int c = 0; c < CT; c++) {
            if (c < nc) {
                res[(size_t)c * poly_words] = sr[bi][c];
                res[(size_t)c * poly_words + m2] = si[bi][c];
            }
        }
    }
}

// ---- extended blind rotation (algorithm.rs:121-273): the accumulator is `ext` interleaved rings; items are (ciphertext b, ring i) at
// index b * ext + i.  Which source ring and which X^a table entry a ring takes depends on the ciphertext's own a_t (and is decided per
// item on the device); the reference's skip conditions are kept verbatim (see the oracle's note on a_hi = 0 / 2n - 1).
struct ExtInitArgs {
    char *acc; uint64_t acc_item;        // acc item stride (bytes); column 0, limb j at + j * cols * n * 8
    const char *lut; uint64_t lut_item;  // lut[j]: VecZnx(1 col), limb l at + l * n * 8
    const long long *lwe; uint64_t lwe_stride;
    uint32_t n, ext, cols;
};
__global__ void __launch_bounds__(256) cggi_ext_init_kernel(ExtInitArgs p) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; // destination coefficient
    if (k >= p.n) return;
    const uint32_t item = blockIdx.z, b = item / p.ext, i = item % p.ext, n = p.n;
    const long long two_n_ext = 2ll * n * p.ext;
    const unsigned long long b_pos = (unsigned long long)((p.lwe[(size_t)b * p.lwe_stride] + two_n_ext) & (two_n_ext - 1));
    const uint32_t b_hi = (uint32_t)(b_pos / p.ext), b_lo = (uint32_t)(b_pos & (p.ext - 1));
    const uint32_t j = i < b_lo ? p.ext - b_lo + i : i - b_lo;   // (:185-190)
    const uint32_t rot = i < b_lo ? b_hi + 1 : b_hi;
    const uint32_t mp_2n = rot & (2 * n - 1), mp_1n = mp_2n & (n - 1);
    const bool neg_first = mp_2n < n;
    const long long *src = reinterpret_cast<const long long *>(p.lut + (size_t)j * p.lut_item + (size_t)blockIdx.y * n * 8);
    long long *dst = reinterpret_cast<long long *>(p.acc + (size_t)item * p.acc_item + (size_t)blockIdx.y * p.cols * n * 8);
    long long v;
    bool neg;
    if (k < mp_1n) { v = src[n - mp_1n + k]; neg = neg_first; }
    else { v = src[k - mp_1n]; neg = !neg_first; }
    dst[k] = neg ? (long long)(0ull - (unsigned long long)v) : v;
}
// acc_add[b][i][poly] = (acc_add + x_pow_a[idx] * v[b][j][poly]) - v[b][i][poly] with (j, idx, skip) from a_t of ciphertext b (:216-258)
struct XaiExtArgs {
    char *acc;       uint64_t acc_item;
    const char *v;   uint64_t v_item;
    const char *xpa;
    const long long *lwe; uint64_t lwe_stride;
    uint32_t n, ext;
};
__device__ __forceinline__ bool ext_route(long long ai, uint32_t n, uint32_t ext, uint32_t i, uint32_t &j, uint32_t &idx) {
    const long long two_n_ext = 2ll * n * ext;
    const unsigned long long pos = (unsigned long long)((ai + two_n_ext) & (two_n_ext - 1));
    const uint32_t hi = (uint32_t)(pos / ext), lo = (uint32_t)(pos & (ext - 1));
    if (lo == 0) { j = i; idx = hi; return hi != 0; }
    if (i < lo) { j = ext - lo + i; idx = hi + 1; return ((hi + 1) & (2 * n - 1)) != 0; }
    j = i - lo; idx = hi;
    return hi != 0;
}
__global__ void __launch_bounds__(256) cggi_xai_ext_ntt120_kernel(XaiExtArgs p) {
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= p.n) return;
    const uint32_t item = blockIdx.z, b = item / p.ext, i = item % p.ext, poly = blockIdx.y;
    uint32_t j, idx;
    if (!ext_route(p.lwe[(size_t)b * p.lwe_stride], p.n, p.ext, i, j, idx)) return;
    const n120::PrimeRt pr(u / (p.n / 4));
    const uint32_t q = pr.q;
    const uint4 w = __ldg(reinterpret_cast<const uint4 *>(p.xpa + (size_t)idx * p.n * 16) + u);
    const uint4 vj = *(reinterpret_cast<const uint4 *>(p.v + (size_t)(b * p.ext + j) * p.v_item + (size_t)poly * p.n * 16) + u);
    const uint4 vi = *(reinterpret_cast<const uint4 *>(p.v + (size_t)item * p.v_item + (size_t)poly * p.n * 16) + u);
    uint4 *ap = reinterpret_cast<uint4 *>(p.acc + (size_t)item * p.acc_item + (size_t)poly * p.n * 16) + u;
    const uint4 a = *ap;
    auto f = [&](uint32_t acc, uint32_t ww, uint32_t x, uint32_t y) {
        const uint32_t t = n120::csub(acc + pr.reduce((unsigned long long)ww * x), q);
        return t >= y ? t - y : t - y + q;
    };
    *ap = make_uint4(f(a.x, w.x, vj.x, vi.x), f(a.y, w.y, vj.y, vi.y), f(a.z, w.z, vj.z, vi.z), f(a.w, w.w, vj.w, vi.w));
}
__global__ void __launch_bounds__(256) cggi_xai_ext_fft64_kernel(XaiExtArgs p) {
    const uint32_t c = blockIdx.x * blockDim.x + threadIdx.x; // complex index
    const uint32_t m = p.n / 2;
    if (c >= m) return;
    const uint32_t item = blockIdx.z, b = item / p.ext, i = item % p.ext, poly = blockIdx.y;
    uint32_t j, idx;
    if (!ext_route(p.lwe[(size_t)b * p.lwe_stride], p.n, p.ext, i, j, idx)) return;
    const double *w = reinterpret_cast<const double *>(p.xpa + (size_t)idx * p.n * 8);
    const double *vj = reinterpret_cast<const double *>(p.v + (size_t)(b * p.ext + j) * p.v_item + (size_t)poly * p.n * 8);
    const double *vi = reinterpret_cast<const double *>(p.v + (size_t)item * p.v_item + (size_t)poly * p.n * 8);
    double *a = reinterpret_cast<double *>(p.acc + (size_t)item * p.acc_item + (size_t)poly * p.n * 8);
    const double wr = __ldg(w + c), wi = __ldg(w + c + m), xr = vj[c], xi = vj[c + m];
    const double pr = wr * xr - wi * xi, pi = wr * xi + wi * xr; // reim_mul(ppol, v[j])
    a[c] = (a[c] + pr) - vi[c];
    a[c + m] = (a[c + m] + pi) - vi[c + m];
}

int cggi_blind_rotate_impl(pgb_module *m, pgb_vec_znx *res, const int64_t *lwe_2n, uint64_t n_lwe, const pgb_vec_znx *lut,
                           const pgb_vmp_pmat *brk, const pgb_svp_ppol *x_pow_a, uint64_t block_size, uint64_t base2k, const pgb_batch *bt,
                           void *scratch, size_t scratch_len) {
    PGB_REQUIRE(bt && bt->count >= 1 && bt->count <= 65535, "cggi_blind_rotate: batch count must be in [1, 65535]");
    PGB_REQUIRE(res->n == m->n && lut->n == m->n && brk->n == m->n && x_pow_a->n == m->n, "cggi_blind_rotate: ring degree mismatch");
    PGB_REQUIRE(x_pow_a->cols == 2 * m->n, "cggi_blind_rotate: x_pow_a must have 2n columns");
    PGB_REQUIRE(brk->cols_in == res->cols && brk->cols_out == res->cols, "cggi_blind_rotate: brk rank does not match res");
    PGB_REQUIRE(block_size >= 1, "cggi_blind_rotate: block_size must be >= 1");
    const uint64_t n = m->n, pb = prep_bytes(m), bb = big_bytes(m), B = bt->count, cols = res->cols;
    const uint64_t dnum = brk->rows, bsize = brk->size;
    const size_t need = pgb_cggi_blind_rotate_tmp_bytes(m, cols - 1, res->size, dnum, bsize, B);
    if (scratch_len < need) {
        pgb_set_error("cggi_blind_rotate: scratch of %zu bytes < required %zu", scratch_len, need);
        return PGB_ERR_SCRATCH;
    }
    Arena ar = {(char *)scratch, scratch_len, 0};
    const uint64_t acc_bs = n * cols * dnum * pb, vres_bs = n * cols * bsize * pb, xai_bs = n * bsize * pb, big_bs = n * bsize * bb;
    pgb_vec_znx_dft acc_dft = mk(ar.take(B * acc_bs), n, cols, dnum);
    pgb_vec_znx_dft vmp_res = mk(ar.take(B * vres_bs), n, cols, bsize);
    pgb_vec_znx_dft acc_add = mk(ar.take(B * vres_bs), n, cols, bsize);
    ar.take(B * xai_bs); // vmp_xai of the reference: not materialised (fused)
    pgb_vec_znx_big acc_big = mk(ar.take(B * big_bs), n, 1, bsize);
    const uint64_t brk_bytes = pgb_bytes_of_vmp_pmat(m, brk->rows, brk->cols_in, brk->cols_out, brk->size);
    const uint64_t lwe_stride = n_lwe + 1;

    // out.zero(); out[0] = X^b * LUT (algorithm.rs:317-320)
    auto init_acc = [&]() -> int {
        PGB_CHECK_CUDA(cudaMemset2DAsync(res->data, bt->stride_res, 0, n * cols * res->size * 8, B, m->stream));
        const uint64_t mn = umin64(res->size, lut->size);
        LimbSet R = {(char *)res->data, res->cols * n * 8, bt->stride_res};
        LimbSet L = {(char *)lut->data, lut->cols * n * 8, 0};
        return znx_rotate(m, R, L, 0, (const long long *)lwe_2n, (uint32_t)lwe_stride, (uint32_t)mn, (uint32_t)B);
    };
    PGB_TRY(init_acc());
    if (m->flavour == PGB_NTT120 && !opt_on(m, PGB_OPT_NO_FUSION) && bt->stride_res % 8 == 0 &&
        cggi_ntt_fused_supported(m, cols, dnum, bsize, block_size) && lut->cols == 1) {
        // whole rotation in one launch on two of the four primes when the device-measured bound allows (cggi_ntt_fused.cu); otherwise,
        // or when the kernel found an accumulator coefficient outside the bound, the four-prime sequence below redoes the batch
        bool handled = false;
        PGB_TRY(cggi_fused_ntt120(m, (long long *)res->data, bt->stride_res / 8, (const long long *)lwe_2n, lwe_stride, (const char *)brk->data,
                                  brk_bytes, (const char *)x_pow_a->data, (int)n_lwe, (int)block_size, (int)base2k, (int)cols, (int)dnum,
                                  (int)bsize, (int)res->size, (int)B, (const long long *)lut->data, n * umin64(res->size, lut->size), &handled));
        if (handled) return PGB_OK;
        PGB_TRY(init_acc());
    }
    if (cggi_fused_supported(m, cols, dnum, bsize) && (R_ok(cols, dnum)) && !opt_on(m, PGB_OPT_NO_FUSION)) {
        PGB_REQUIRE(bt->stride_res % 8 == 0, "cggi_blind_rotate: res stride must be a multiple of 8 bytes");
        return cggi_fused_fft64(m, (long long *)res->data, bt->stride_res / 8, (const long long *)lwe_2n, lwe_stride, (const double *)brk->data,
                                brk_bytes / 8, (const double *)x_pow_a->data, (int)n_lwe, (int)block_size, (int)base2k, (int)cols, (int)dnum,
                                (int)bsize, (int)res->size, (int)B);
    }
    for (uint64_t blk = 0; blk + block_size <= n_lwe; blk += block_size) { // chunks_exact
        pgb_batch btd = {B, acc_bs, bt->stride_res, 0};
        if (res->size >= dnum && !opt_on(m, PGB_OPT_NO_FUSION)) {
            // the first dnum limbs of every column are the polys 0 .. cols * dnum - 1 of both layouts: one transform launch per block
            LimbSet fin = {(char *)res->data, n * 8, bt->stride_res}, fout = {(char *)acc_dft.data, n * pb, acc_bs};
            if (m->flavour == PGB_NTT120) PGB_TRY(ntt120_forward(m, fin, fout, (int)(cols * dnum), (int)B));
            else PGB_TRY(fft64_forward(m, fin, fout, (int)(cols * dnum), (int)B, -1));
        } else {
            for (uint64_t j = 0; j < cols; j++) PGB_TRY(pgb_vec_znx_dft_apply_batched(m, 1, 0, &acc_dft, j, res, j, &btd));
        }
        if (m->flavour == PGB_NTT120 && cols * dnum <= 16 && block_size <= 8 && !opt_on(m, PGB_OPT_NO_FUSION)) {
            // the block's key products and X^{a_t} - 1 updates in one launch (cggi_block_ntt120_kernel)
            BlockArgs ba = {(const char *)acc_dft.data, acc_bs, (char *)acc_add.data, vres_bs, (const char *)brk->data + blk * brk_bytes, brk_bytes,
                            (const char *)x_pow_a->data, (const long long *)lwe_2n + 1 + blk, lwe_stride, (uint32_t)n, (uint32_t)(cols * dnum),
                            (uint32_t)(cols * bsize), (uint32_t)block_size};
            ProfScope _ps(m, PROF_VMP);
            // staging per CTA: (BT * RMAX + BT * block_size) slots of 256 x 16 bytes; two CTAs per SM need <= 113 KB each
            #define BLOCK_LAUNCH(RM, BTV, LIMKB)                                                                                  \
                {                                                                                                                 \
                    const dim3 grid(((uint32_t)n + 255) / 256, 1, (uint32_t)((B + (BTV) - 1) / (BTV)));                           \
                    const size_t sb = (size_t)((BTV) * (RM) + (BTV) * block_size) * 256 * 16;                                     \
                    if (sb <= (size_t)((LIMKB) << 10)) {                                                                          \
                        static bool attr_dev[32] = {};                                                                            \
                        if (!attr_dev[m->device & 31]) {                                                                          \
                            PGB_CHECK_CUDA(cudaFuncSetAttribute(cggi_block_ntt120_kernel<RM, BTV, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (LIMKB) << 10)); \
                            attr_dev[m->device & 31] = true;                                                                      \
                        }                                                                                                         \
                        cggi_block_ntt120_kernel<RM, BTV, 1><<<grid, 256, sb, m->stream>>>(ba, (uint32_t)B);                      \
                    } else {                                                                                                      \
                        cggi_block_ntt120_kernel<RM, BTV, 0><<<grid, 256, 0, m->stream>>>(ba, (uint32_t)B);                       \
                    }                                                                                                             \
                }
            // the row loops are unrolled over RMAX: rows beyond R cost their multiply-adds anyway, so the tile follows R closely (R = 9,
            // the circuit-bootstrapping shape: 57 ms per blind rotation of 512 with RMAX = 16, 44 ms with 12).  Two ciphertexts per
            // thread at RMAX = 12 need 152 KB of staging = one CTA per SM: measured slower (59 ms).
            if (cols * dnum <= 4) BLOCK_LAUNCH(4, 4, 113)
            else if (cols * dnum <= 6) BLOCK_LAUNCH(6, 2, 113)
            else if (cols * dnum <= 8) BLOCK_LAUNCH(8, 2, 113)
            else if (cols * dnum <= 9) BLOCK_LAUNCH(9, 1, 113)
            else if (cols * dnum <= 10) BLOCK_LAUNCH(10, 1, 113)
            else if (cols * dnum <= 12) BLOCK_LAUNCH(12, 1, 113)
            else BLOCK_LAUNCH(16, 1, 113)
            #undef BLOCK_LAUNCH
            PGB_CHECK_CUDA(cudaGetLastError());
        } else if (m->flavour == PGB_FFT64 && n >= 8 && !opt_on(m, PGB_OPT_NO_FUSION)) {
            BlockArgs ba = {(const char *)acc_dft.data, acc_bs, (char *)acc_add.data, vres_bs, (const char *)brk->data + blk * brk_bytes, brk_bytes,
                            (const char *)x_pow_a->data, (const long long *)lwe_2n + 1 + blk, lwe_stride, (uint32_t)n, (uint32_t)(cols * dnum),
                            (uint32_t)(cols * bsize), (uint32_t)block_size};
            ProfScope _ps(m, PROF_VMP);
            constexpr int CT = 4, CT2 = 2, BT = 2;
            const size_t sb = (size_t)BT * cols * dnum * 2 * 128 * sizeof(double2);
            if (B >= 2 && sb <= (size_t)(100 << 10) && !opt_on(m, PGB_OPT_CGGI_BLOCK_BT1)) { // two ciphertexts per thread share every key word
                static bool attr_dev[32] = {};
                if (!attr_dev[m->device & 31]) {
                    PGB_CHECK_CUDA(cudaFuncSetAttribute(cggi_block_fft64_bt_kernel<CT2, BT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 << 10));
                    attr_dev[m->device & 31] = true;
                }
                const dim3 grid(((uint32_t)(n / 4) + 127) / 128, (uint32_t)((cols * bsize + CT2 - 1) / CT2), (uint32_t)((B + BT - 1) / BT));
                cggi_block_fft64_bt_kernel<CT2, BT><<<grid, 128, sb, m->stream>>>(ba, (uint32_t)B);
            } else {
                const dim3 grid(((uint32_t)(n / 4) + 127) / 128, (uint32_t)((cols * bsize + CT - 1) / CT), (uint32_t)B);
                cggi_block_fft64_kernel<CT><<<grid, 128, 0, m->stream>>>(ba);
            }
            PGB_CHECK_CUDA(cudaGetLastError());
        } else {
        PGB_CHECK_CUDA(cudaMemsetAsync(acc_add.data, 0, B * vres_bs, m->stream)); // vec_znx_dft_zero on every column
        for (uint64_t t = 0; t < block_size; t++) {
            pgb_vmp_pmat ski = *brk;
            ski.data = (char *)brk->data + (blk + t) * brk_bytes;
            pgb_batch btv = {B, vres_bs, acc_bs, 0};
            PGB_TRY(vmp_apply_impl(m, &vmp_res, &acc_dft, &ski, 0, &btv));
            XaiArgs xa = {(char *)acc_add.data, vres_bs, (const char *)vmp_res.data, vres_bs, (const char *)x_pow_a->data,
                          (const long long *)lwe_2n + 1 + blk + t, lwe_stride, (uint32_t)n, (uint32_t)(cols * bsize)};
            ProfScope _ps(m, PROF_ELEMENTWISE);
            if (m->flavour == PGB_NTT120) {
                dim3 grid(((uint32_t)n + 255) / 256, xa.polys, (uint32_t)B);
                cggi_xai_ntt120_kernel<<<grid, 256, 0, m->stream>>>(xa);
            } else {
                dim3 grid(((uint32_t)(n / 2) + 255) / 256, xa.polys, (uint32_t)B);
                cggi_xai_fft64_kernel<<<grid, 256, 0, m->stream>>>(xa);
            }
            PGB_CHECK_CUDA(cudaGetLastError());
        }
        }
        if (m->flavour == PGB_NTT120 && ntt120_fused_supported(m) && !opt_on(m, PGB_OPT_NO_FUSION)) {
            // algorithm.rs:361-365 for all columns in one launch: inverse transform + CRT + add_small (the accumulator column itself) +
            // normalize, nothing but acc_add and the accumulator touches HBM
            PGB_TRY(ntt120_fused_back(m, (const char *)acc_add.data, vres_bs, nullptr, 0, (int)(cols * bsize), (int)cols, (const char *)res->data,
                                      bt->stride_res, res->cols * n * 8, (int)umin64(bsize, res->size), (char *)res->data, bt->stride_res,
                                      res->cols * n * 8, (int)res->size, (int)base2k, 0, (int)B, nullptr, 0, 0, nullptr, false, true, true));
            continue;
        }
        if (m->flavour == PGB_FFT64 && base2k >= 1 && base2k <= 63 && fft64_fused_back_supported(m, (int)bsize) && !opt_on(m, PGB_OPT_NO_FUSION)) {
            // algorithm.rs:361-365 for all columns in one launch (fft64_back_kernel): acc_add is read once, the accumulator updated in place
            PGB_TRY(fft64_fused_back(m, (const char *)acc_add.data, vres_bs, (int)cols, (int)bsize, (char *)res->data, bt->stride_res,
                                     (int)res->size, (int)base2k, (int)B));
            continue;
        }
        for (uint64_t i = 0; i < cols; i++) { // algorithm.rs:361-365
            pgb_batch bti = {B, big_bs, vres_bs, 0};
            PGB_TRY(pgb_vec_znx_idft_apply_batched(m, &acc_big, 0, &acc_add, i, &bti));
            pgb_batch bts = {B, big_bs, bt->stride_res, 0};
            PGB_TRY(big_add_small_impl(m, &acc_big, 0, res, i, &bts));
            pgb_batch btn = {B, bt->stride_res, big_bs, 0};
            PGB_TRY(big_normalize_impl(m, res, base2k, 0, i, &acc_big, base2k, 0, 0, true, &btn));
        }
    }
    return PGB_OK;
}
// execute_block_binary_extended over a batch (algorithm.rs:121-273): the limb-wise HAL sequence with B * ext accumulator items
extern "C" size_t pgb_cggi_blind_rotate_extended_tmp_bytes(const pgb_module *m, uint64_t rank, uint64_t res_size, uint64_t dnum, uint64_t brk_size,
                                                           uint64_t ext, uint64_t batch) {
    const uint64_t n = m->n, pb = prep_bytes(m), bb = big_bytes(m), cols = rank + 1, items = batch * ext;
    return align_up(items * n * cols * res_size * 8) + align_up(items * n * cols * dnum * pb) + 2 * align_up(items * n * cols * brk_size * pb) +
           align_up(items * n * brk_size * bb) + ALIGN;
}
extern "C" int pgb_cggi_blind_rotate_extended_batched(pgb_module *m, pgb_vec_znx *res, const int64_t *lwe_2n, uint64_t n_lwe, const pgb_vec_znx *lut,
                                                      uint64_t ext, const pgb_vmp_pmat *brk, const pgb_svp_ppol *x_pow_a, uint64_t block_size,
                                                      uint64_t base2k, const pgb_batch *bt, void *scratch, size_t scratch_len) {
    PGB_REQUIRE(bt && bt->count >= 1 && bt->count * ext <= 65535, "cggi_blind_rotate_extended: batch * extension_factor must be in [1, 65535]");
    PGB_REQUIRE(ext >= 1 && (ext & (ext - 1)) == 0, "cggi_blind_rotate_extended: extension_factor must be a power of two");
    PGB_REQUIRE(res->n == m->n && lut->n == m->n && brk->n == m->n && x_pow_a->n == m->n, "cggi_blind_rotate_extended: ring degree mismatch");
    PGB_REQUIRE(x_pow_a->cols == 2 * m->n && lut->cols == 1, "cggi_blind_rotate_extended: x_pow_a needs 2n columns, the LUT one");
    PGB_REQUIRE(brk->cols_in == res->cols && brk->cols_out == res->cols, "cggi_blind_rotate_extended: brk rank does not match res");
    PGB_REQUIRE(block_size >= 1, "cggi_blind_rotate_extended: block_size must be >= 1");
    const uint64_t n = m->n, pb = prep_bytes(m), bb = big_bytes(m), B = bt->count, cols = res->cols, items = B * ext;
    const uint64_t dnum = brk->rows, bsize = brk->size;
    const size_t need = pgb_cggi_blind_rotate_extended_tmp_bytes(m, cols - 1, res->size, dnum, bsize, ext, B);
    if (scratch_len < need) {
        pgb_set_error("cggi_blind_rotate_extended: scratch of %zu bytes < required %zu", scratch_len, need);
        return PGB_ERR_SCRATCH;
    }
    Arena ar = {(char *)scratch, scratch_len, 0};
    const uint64_t acc_item = n * cols * res->size * 8, accd_bs = n * cols * dnum * pb, vres_bs = n * cols * bsize * pb, big_bs = n * bsize * bb;
    pgb_vec_znx acc = mk(ar.take(items * acc_item), n, cols, res->size);
    pgb_vec_znx_dft acc_dft = mk(ar.take(items * accd_bs), n, cols, dnum);
    pgb_vec_znx_dft vmp_res = mk(ar.take(items * vres_bs), n, cols, bsize);
    pgb_vec_znx_dft acc_add = mk(ar.take(items * vres_bs), n, cols, bsize);
    pgb_vec_znx_big acc_big = mk(ar.take(items * big_bs), n, 1, bsize);
    const uint64_t brk_bytes = pgb_bytes_of_vmp_pmat(m, brk->rows, brk->cols_in, brk->cols_out, brk->size);
    const uint64_t lwe_stride = n_lwe + 1;
    // acc[i].zero(); acc[i][0] = X^{b_hi (+1)} * lut[j] (:159-190)
    PGB_CHECK_CUDA(cudaMemsetAsync(acc.data, 0, items * acc_item, m->stream));
    {
        const uint64_t mn = umin64(res->size, lut->size);
        ExtInitArgs ia = {(char *)acc.data, acc_item, (const char *)lut->data, n * lut->size * 8, (const long long *)lwe_2n, lwe_stride, (uint32_t)n,
                          (uint32_t)ext, (uint32_t)cols};
        ProfScope _ps(m, PROF_OTHER);
        cggi_ext_init_kernel<<<dim3(((uint32_t)n + 255) / 256, (uint32_t)mn, (uint32_t)items), 256, 0, m->stream>>>(ia);
        PGB_CHECK_CUDA(cudaGetLastError());
    }
    for (uint64_t blk = 0; blk + block_size <= n_lwe; blk += block_size) {
        pgb_batch btd = {items, accd_bs, acc_item, 0};
        const bool fuse = !opt_on(m, PGB_OPT_NO_FUSION);
        if (acc.size >= dnum && fuse) { // one transform launch for all columns (see cggi_blind_rotate_impl)
            LimbSet fin = {(char *)acc.data, n * 8, acc_item}, fout = {(char *)acc_dft.data, n * pb, accd_bs};
            if (m->flavour == PGB_NTT120) PGB_TRY(ntt120_forward(m, fin, fout, (int)(cols * dnum), (int)items));
            else PGB_TRY(fft64_forward(m, fin, fout, (int)(cols * dnum), (int)items, -1));
        } else {
            for (uint64_t j = 0; j < cols; j++) PGB_TRY(pgb_vec_znx_dft_apply_batched(m, 1, 0, &acc_dft, j, &acc, j, &btd));
        }
        PGB_CHECK_CUDA(cudaMemsetAsync(acc_add.data, 0, items * vres_bs, m->stream));
        for (uint64_t t = 0; t < block_size; t++) {
            pgb_vmp_pmat ski = *brk;
            ski.data = (char *)brk->data + (blk + t) * brk_bytes;
            pgb_batch btv = {items, vres_bs, accd_bs, 0};
            PGB_TRY(vmp_apply_impl(m, &vmp_res, &acc_dft, &ski, 0, &btv));
            XaiExtArgs xa = {(char *)acc_add.data, vres_bs, (const char *)vmp_res.data, vres_bs, (const char *)x_pow_a->data,
                             (const long long *)lwe_2n + 1 + blk + t, lwe_stride, (uint32_t)n, (uint32_t)ext};
            ProfScope _ps(m, PROF_ELEMENTWISE);
            if (m->flavour == PGB_NTT120)
                cggi_xai_ext_ntt120_kernel<<<dim3(((uint32_t)n + 255) / 256, (uint32_t)(cols * bsize), (uint32_t)items), 256, 0, m->stream>>>(xa);
            else
                cggi_xai_ext_fft64_kernel<<<dim3(((uint32_t)(n / 2) + 255) / 256, (uint32_t)(cols * bsize), (uint32_t)items), 256, 0, m->stream>>>(xa);
            PGB_CHECK_CUDA(cudaGetLastError());
        }
        // (:262-268) inverse transform + add_small + normalize of every column of every item: one launch where the fused back ends apply
        if (fuse && m->flavour == PGB_NTT120 && ntt120_fused_supported(m)) {
            PGB_TRY(ntt120_fused_back(m, (const char *)acc_add.data, vres_bs, nullptr, 0, (int)(cols * bsize), (int)cols, (const char *)acc.data,
                                      acc_item, cols * n * 8, (int)umin64(bsize, acc.size), (char *)acc.data, acc_item, cols * n * 8, (int)acc.size,
                                      (int)base2k, 0, (int)items, nullptr, 0, 0, nullptr, false, true, true));
            continue;
        }
        if (fuse && m->flavour == PGB_FFT64 && base2k >= 1 && base2k <= 63 && fft64_fused_back_supported(m, (int)bsize)) {
            PGB_TRY(fft64_fused_back(m, (const char *)acc_add.data, vres_bs, (int)cols, (int)bsize, (char *)acc.data, acc_item, (int)acc.size,
                                     (int)base2k, (int)items));
            continue;
        }
        for (uint64_t i = 0; i < cols; i++) {
            pgb_batch bti = {items, big_bs, vres_bs, 0};
            PGB_TRY(pgb_vec_znx_idft_apply_batched(m, &acc_big, 0, &acc_add, i, &bti));
            pgb_batch bts = {items, big_bs, acc_item, 0};
            PGB_TRY(big_add_small_impl(m, &acc_big, 0, &acc, i, &bts));
            pgb_batch btn = {items, acc_item, big_bs, 0};
            PGB_TRY(big_normalize_impl(m, &acc, base2k, 0, i, &acc_big, base2k, 0, 0, true, &btn));
        }
    }
    // res <- acc[0] of every ciphertext (:270-272)
    PGB_CHECK_CUDA(cudaMemcpy2DAsync(res->data, bt->stride_res, acc.data, ext * acc_item, acc_item, B, cudaMemcpyDeviceToDevice, m->stream));
    return PGB_OK;
}

extern "C" int pgb_cggi_blind_rotate_batched(pgb_module *m, pgb_vec_znx *res, const int64_t *lwe_2n, uint64_t n_lwe, const pgb_vec_znx *lut,
                                             const pgb_vmp_pmat *brk, const pgb_svp_ppol *x_pow_a, uint64_t block_size, uint64_t base2k,
                                             const pgb_batch *bt, void *scratch, size_t scratch_len) {
    return cggi_blind_rotate_impl(m, res, lwe_2n, n_lwe, lut, brk, x_pow_a, block_size, base2k, bt, scratch, scratch_len);
}


// ---- mod_switch_2n on the device (algorithms/mod.rs:136-181) ---------------------------------------------------------
struct ModSwitchArgs {
    const char *lwe; uint64_t lwe_bs, limb_stride; // VecZnx(n = n_lwe + 1, cols = 1, size): limb j at + j * limb_stride bytes
    long long *res;                                 // [batch][len]
    uint32_t len, base2k, log2n, size;
    int rot_left;
};
__global__ void __launch_bounds__(256) cggi_mod_switch_kernel(ModSwitchArgs p) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.len) return;
    const char *src = p.lwe + (size_t)blockIdx.y * p.lwe_bs;
    long long x = reinterpret_cast<const long long *>(src)[i];
    if (p.rot_left) x = (long long)(0ull - (unsigned long long)x);
    if (p.base2k > p.log2n) {
        const uint32_t diff = p.base2k - (p.log2n - 1);
        x = (long long)((unsigned long long)x + (1ull << (diff - 1))) >> diff; // div_round_by_pow2 (:179-181)
    } else {
        const uint32_t rem = p.base2k - (p.log2n % p.base2k);
        const uint32_t size = (p.log2n + p.base2k - 1) / p.base2k;
        for (uint32_t j = 1; j < size; j++) {
            const long long y = reinterpret_cast<const long long *>(src + (size_t)j * p.limb_stride)[i];
            if (j == size - 1 && rem != p.base2k) x = (long long)(((unsigned long long)x << (p.base2k - rem)) + (unsigned long long)(y >> rem));
            else x = (long long)(((unsigned long long)x << p.base2k) + (unsigned long long)y);
        }
    }
    p.res[(size_t)blockIdx.y * p.len + i] = x;
}
extern "C" int pgb_cggi_mod_switch_2n_batched(pgb_module *m, int64_t *res, const pgb_vec_znx *lwe, uint64_t lwe_base2k, uint64_t two_n_domain,
                                              int rot_left, const pgb_batch *bt) {
    PGB_REQUIRE(bt && bt->count >= 1 && bt->count <= 65535, "cggi_mod_switch_2n: batch count must be in [1, 65535]");
    PGB_REQUIRE(lwe->cols == 1 && lwe->size >= 1 && lwe->n >= 2, "cggi_mod_switch_2n: lwe must be a one-column VecZnx of n_lwe + 1 coefficients");
    PGB_REQUIRE(lwe_base2k >= 1 && lwe_base2k <= 62 && two_n_domain >= 2, "cggi_mod_switch_2n: bad base2k / domain");
    uint32_t log2n = 0;
    while (((uint64_t)1 << log2n) < two_n_domain) log2n++; // usize::BITS - (n - 1).leading_zeros()
    log2n += 1;
    const uint32_t size_needed = lwe_base2k > log2n ? 1 : (uint32_t)((log2n + lwe_base2k - 1) / lwe_base2k);
    PGB_REQUIRE(lwe->size >= size_needed, "cggi_mod_switch_2n: lwe has %llu limbs, %u needed", (unsigned long long)lwe->size, size_needed);
    ModSwitchArgs p = {(const char *)lwe->data, bt->stride_a, lwe->n * 8, (long long *)res, (uint32_t)lwe->n, (uint32_t)lwe_base2k, log2n,
                       (uint32_t)lwe->size, rot_left};
    { ProfScope _ps(m, PROF_OTHER);
    cggi_mod_switch_kernel<<<dim3(((uint32_t)lwe->n + 255) / 256, (uint32_t)bt->count), 256, 0, m->stream>>>(p);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

// ---- execute_standard (algorithm.rs:370-443): block_size == 1 keys ------------------------------------------------------
// out += (X^{a} - 1) * tmp for every limb of every column: glwe_mul_xp_minus_one_assign (operations/glwe.rs:1051-1062:
// tmp' = rotate(a, tmp) - tmp, reference/vec_znx/mul_xp_minus_one.rs:24-38) followed by glwe_add_assign (api/operations.rs:273-289)
struct XpAddArgs {
    char *out; uint64_t out_bs;
    const char *tmp; uint64_t tmp_bs;
    const long long *lwe; uint64_t lwe_stride;
    uint32_t n, limbs;
};
__global__ void __launch_bounds__(256) cggi_xpm1_add_kernel(XpAddArgs p) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    const uint32_t b = blockIdx.z, limb = blockIdx.y;
    const long long a = p.lwe[(size_t)b * p.lwe_stride];
    const uint32_t mp = (uint32_t)(a & (long long)(2 * p.n - 1));
    const long long *t = reinterpret_cast<const long long *>(p.tmp + (size_t)b * p.tmp_bs) + (size_t)limb * p.n;
    long long *o = reinterpret_cast<long long *>(p.out + (size_t)b * p.out_bs) + (size_t)limb * p.n;
    const uint32_t s = (i - mp) & (2 * p.n - 1); // coefficient s of tmp lands on i (negated when it wrapped once)
    const unsigned long long r = s < p.n ? (unsigned long long)t[s] : 0ull - (unsigned long long)t[s - p.n];
    o[i] = (long long)((unsigned long long)o[i] + (r - (unsigned long long)t[i]));
}

extern "C" size_t pgb_cggi_blind_rotate_standard_tmp_bytes(const pgb_module *m, uint64_t rank, uint64_t res_size, uint64_t res_base2k,
                                                           const pgb_vmp_pmat *brk, uint64_t brk_base2k, uint64_t batch) {
    const uint64_t acc = align_up(batch * m->n * (rank + 1) * res_size * 8);
    return acc + pgb_glwe_external_product_tmp_bytes(m, res_size, res_size, res_base2k, brk, brk_base2k, 1, batch) + ALIGN;
}
extern "C" int pgb_cggi_blind_rotate_standard_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, const int64_t *lwe_2n,
                                                      uint64_t n_lwe, const pgb_vec_znx *lut, const pgb_vmp_pmat *brk, uint64_t brk_base2k,
                                                      const pgb_batch *bt, void *scratch, size_t scratch_len) {
    PGB_REQUIRE(bt && bt->count >= 1 && bt->count <= 65535, "cggi_blind_rotate_standard: batch count must be in [1, 65535]");
    PGB_REQUIRE(res->n == m->n && lut->n == m->n && brk->n == m->n, "cggi_blind_rotate_standard: ring degree mismatch");
    PGB_REQUIRE(brk->cols_in == res->cols && brk->cols_out == res->cols, "cggi_blind_rotate_standard: brk rank does not match res");
    const uint64_t n = m->n, B = bt->count, cols = res->cols;
    const size_t need = pgb_cggi_blind_rotate_standard_tmp_bytes(m, cols - 1, res->size, res_base2k, brk, brk_base2k, B);
    if (scratch_len < need) {
        pgb_set_error("cggi_blind_rotate_standard: scratch of %zu bytes < required %zu", scratch_len, need);
        return PGB_ERR_SCRATCH;
    }
    const uint64_t tmp_bs = n * cols * res->size * 8;
    Arena ar = {(char *)scratch, scratch_len, 0};
    pgb_vec_znx tmp = mk(ar.take(B * tmp_bs), n, cols, res->size);
    char *ep_scratch = ar.rest();
    const size_t ep_len = ar.rest_len();
    const uint64_t brk_bytes = pgb_bytes_of_vmp_pmat(m, brk->rows, brk->cols_in, brk->cols_out, brk->size);
    const uint64_t lwe_stride = n_lwe + 1;
    // out.zero(); out[0] = X^b * LUT (:412-415)
    PGB_CHECK_CUDA(cudaMemset2DAsync(res->data, bt->stride_res, 0, n * cols * res->size * 8, B, m->stream));
    {
        const uint64_t mn = umin64(res->size, lut->size);
        LimbSet R = {(char *)res->data, res->cols * n * 8, bt->stride_res};
        LimbSet L = {(char *)lut->data, lut->cols * n * 8, 0};
        PGB_TRY(znx_rotate(m, R, L, 0, (const long long *)lwe_2n, (uint32_t)lwe_stride, (uint32_t)mn, (uint32_t)B));
    }
    for (uint64_t i = 0; i < n_lwe; i++) {
        pgb_vmp_pmat ski = *brk;
        ski.data = (char *)brk->data + i * brk_bytes;
        pgb_batch bte = {B, tmp_bs, bt->stride_res, 0};
        PGB_TRY(pgb_glwe_external_product_batched(m, &tmp, res_base2k, res, res_base2k, &ski, brk_base2k, 1, &bte, ep_scratch, ep_len)); // :429
        XpAddArgs xa = {(char *)res->data, bt->stride_res, (const char *)tmp.data, tmp_bs, (const long long *)lwe_2n + 1 + i, lwe_stride,
                        (uint32_t)n, (uint32_t)(cols * res->size)};
        { ProfScope _ps(m, PROF_ELEMENTWISE);
        cggi_xpm1_add_kernel<<<dim3(((uint32_t)n + 255) / 256, xa.limbs, (uint32_t)B), 256, 0, m->stream>>>(xa); // :432-435
        }
        PGB_CHECK_CUDA(cudaGetLastError());
    }
    pgb_batch btn = {B, bt->stride_res, bt->stride_res, 0};
    for (uint64_t c = 0; c < cols; c++) // glwe_normalize_assign (:440): in place, one thread owns a coefficient across limbs
        PGB_TRY(big_normalize_impl(m, res, res_base2k, 0, c, res, res_base2k, c, 0, false, &btn));
    return PGB_OK;
}

// ---- host-buffer front end (BlindRotationExecute::execute over host-resident LWE in / GLWE out, cggi/algorithm.rs:88-117) --------------
// Per bootstrap lwe_size * (n_lwe + 1) * 8 bytes go up and (rank + 1) * res_size * n * 8 bytes come back (5.5 KB / 16 KB at the bench
// shape against ~10 us of compute), so unlike the key-switch this path is not PCIe bound: all LWEs go up in one copy, the mod switch and
// the rotations run in whole-wave chunks on the module's stream and every finished chunk is copied back on a second stream while the
// next one computes.
static uint64_t cggi_host_chunk(const pgb_module *m, uint64_t count) {
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, m->device);
    const uint64_t wave = (uint64_t)sms * 4; // ciphertexts one wave of the persistent kernels holds (4 per SM at n = 512)
    if (count <= 2 * wave) return count;
    const uint64_t waves = div_ceil64(count, wave), per = div_ceil64(waves, 4);
    return umin64(per * wave, 65535 / wave * wave);
}
extern "C" int pgb_cggi_blind_rotate_host(pgb_module *m, int64_t *res_host, uint64_t rank, uint64_t res_size, const int64_t *lwe_host,
                                          uint64_t n_lwe, uint64_t lwe_size, uint64_t lwe_base2k, int rot_left, const pgb_vec_znx *lut,
                                          const pgb_vmp_pmat *brk, const pgb_svp_ppol *x_pow_a, uint64_t block_size, uint64_t base2k,
                                          uint64_t count) {
    PGB_REQUIRE(res_host && lwe_host && lut && brk && x_pow_a, "cggi_blind_rotate_host: null argument");
    PGB_REQUIRE(lwe_size >= 1 && res_size >= 1 && n_lwe >= 1, "cggi_blind_rotate_host: empty shapes");
    if (count == 0) return PGB_OK;
    const uint64_t n = m->n, cols = rank + 1, len = n_lwe + 1;
    const uint64_t lwe_item = lwe_size * len * 8, res_item = n * cols * res_size * 8;
    const uint64_t chunk = cggi_host_chunk(m, count);
    const size_t tmp = pgb_cggi_blind_rotate_tmp_bytes(m, rank, res_size, brk->rows, brk->size, chunk);
    const uint64_t o_lwe = 0, o_2n = o_lwe + align_up(count * lwe_item), o_res = o_2n + align_up(count * len * 8),
                   o_tmp = o_res + align_up(count * res_item);
    PGB_TRY(ensure_ws(m, o_tmp + align_up(tmp) + ALIGN));
    char *ws = (char *)m->ws;
    cudaStream_t s_in = m->aux_stream[0], s_out = m->aux_stream[1], s_c = m->stream;
    PGB_CHECK_CUDA(cudaMemcpyAsync(ws + o_lwe, lwe_host, count * lwe_item, cudaMemcpyHostToDevice, s_in));
    PGB_CHECK_CUDA(cudaEventRecord(m->ev[0], s_in));
    PGB_CHECK_CUDA(cudaStreamWaitEvent(s_c, m->ev[0], 0));
    // mod_switch_2n of every LWE (algorithms/mod.rs:136-176), at most 65535 per launch
    for (uint64_t first = 0; first < count; first += 65535) {
        const uint64_t cnt = umin64(65535, count - first);
        pgb_vec_znx lv = {ws + o_lwe + first * lwe_item, len, 1, lwe_size, lwe_size};
        pgb_batch btm = {cnt, 0, lwe_item, 0};
        PGB_TRY(pgb_cggi_mod_switch_2n_batched(m, (int64_t *)(ws + o_2n) + first * len, &lv, lwe_base2k, 2 * n, rot_left, &btm));
    }
    int slot = 0;
    for (uint64_t first = 0; first < count; first += chunk, slot ^= 1) {
        const uint64_t cnt = umin64(chunk, count - first);
        pgb_vec_znx rv = {ws + o_res + first * res_item, n, cols, res_size, res_size};
        pgb_batch bt = {cnt, res_item, 0, 0};
        PGB_TRY(cggi_blind_rotate_impl(m, &rv, (const int64_t *)(ws + o_2n) + first * len, n_lwe, lut, brk, x_pow_a, block_size, base2k, &bt,
                                       ws + o_tmp, m->ws_len - o_tmp));
        PGB_CHECK_CUDA(cudaEventRecord(m->ev[2 + slot], s_c));
        PGB_CHECK_CUDA(cudaStreamWaitEvent(s_out, m->ev[2 + slot], 0));
        PGB_CHECK_CUDA(cudaMemcpyAsync((char *)res_host + first * res_item, rv.data, cnt * res_item, cudaMemcpyDeviceToHost, s_out));
    }
    PGB_CHECK_CUDA(cudaStreamSynchronize(s_out));
    PGB_CHECK_CUDA(cudaStreamSynchronize(s_c));
    return PGB_OK;
}
