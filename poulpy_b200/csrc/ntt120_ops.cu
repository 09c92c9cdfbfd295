// ntt120_ops.cu -- DFT-domain element-wise kernels of the NTT120 flavour: vmp (K6), svp (K5), add/sub/copy/zero (K8).
//
// A DFT "poly" is 16*n bytes: four planes [k][n] of canonical u32 residues.  Every kernel here is a pure
// stream over polys (HBM-bound): each thread owns one 128-bit word (four consecutive frequencies of one prime).
//   vmp : res[c][k][f] = sum_r a[r][k][f] * M[r][c][k][f] mod Q[k]
//         (poulpy-cpu-ref/src/reference/ntt120/vmp.rs:169-288, mat_vec.rs:343-447; products accumulate in u64,
//          exact for 16 rows at a time, one Barrett-style reduction per 16 rows)
//   svp : res[j][k][f] = ppol[k][f] * b[j][k][f] mod Q[k]      (svp.rs:87-180)
//   add/sub/neg/copy/zero on canonical residues                   (vec_znx_dft.rs:418-652, ntt120/prim.rs:64-165)
#include <stdlib.h>

#include "internal.h"
#include "ntt120.cuh"

using namespace n120;

struct VmpArgs {
    const char *a;  uint64_t a_bs;     // a polys: a + b*a_bs + r*poly_bytes
    char *res;      uint64_t res_bs;   // res polys: res + b*res_bs + c*poly_bytes
    const char *pm; uint64_t pm_bs;    // pmat polys: pm + (b / pm_div)*pm_bs + (r*C + c)*poly_bytes
    uint32_t n4;                        // uint4 words per plane (= n / 4)
    uint32_t row_max, C, col0, ncols_out, pm_div;
};

template <int CT> __global__ void __launch_bounds__(256) ntt120_vmp_kernel(VmpArgs p) {
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x; // uint4 index inside a poly, [0, 4*n4)
    if (u >= 4 * p.n4) return;
    const PrimeRt pr(u / p.n4);
    const uint32_t c0 = blockIdx.y * CT;
    const size_t poly_words = (size_t)4 * p.n4;
    const uint4 *a = reinterpret_cast<const uint4 *>(p.a + (size_t)blockIdx.z * p.a_bs) + u;
    const uint4 *pm = reinterpret_cast<const uint4 *>(p.pm + (size_t)(blockIdx.z / p.pm_div) * p.pm_bs) + u + (size_t)(p.col0 + c0) * poly_words;
    uint4 *res = reinterpret_cast<uint4 *>(p.res + (size_t)blockIdx.z * p.res_bs) + u + (size_t)c0 * poly_words;
    const int nc = min((uint32_t)CT, p.ncols_out - c0);

    unsigned long long acc[CT][4];
#pragma unroll
    for (int c = 0; c < CT; c++) acc[c][0] = acc[c][1] = acc[c][2] = acc[c][3] = 0;

    for (uint32_t r0 = 0; r0 < p.row_max; r0 += 16) {
        const uint32_t r1 = min(r0 + 16, p.row_max);
#pragma unroll 2
        for (uint32_t r = r0; r < r1; r++) {
            const uint4 av = __ldg(a + (size_t)r * poly_words);
            const uint4 *mrow = pm + (size_t)r * p.C * poly_words;
            uint4 mv[CT];
#pragma unroll
            for (int c = 0; c < CT; c++) mv[c] = c < nc ? __ldcs(mrow + (size_t)c * poly_words) : make_uint4(0, 0, 0, 0); // streamed once
#pragma unroll
            for (int c = 0; c < CT; c++) {
                acc[c][0] += (unsigned long long)av.x * mv[c].x;
                acc[c][1] += (unsigned long long)av.y * mv[c].y;
                acc[c][2] += (unsigned long long)av.z * mv[c].z;
                acc[c][3] += (unsigned long long)av.w * mv[c].w;
            }
        }
#pragma unroll
        for (int c = 0; c < CT; c++) {
#pragma unroll
            for (int i = 0; i < 4; i++) acc[c][i] = pr.reduce(acc[c][i]);
        }
    }
#pragma unroll
    for (int c = 0; c < CT; c++) {
        if (c < nc) res[(size_t)c * poly_words] = make_uint4((uint32_t)acc[c][0], (uint32_t)acc[c][1], (uint32_t)acc[c][2], (uint32_t)acc[c][3]);
    }
}

// Batch-tiled variant for matrices that do not fit in L2 (CKKS relinearisation key: 220-440 MB): one thread applies a loaded matrix
// word to BT batch items, so the matrix crosses HBM once per BT ciphertexts instead of once per ciphertext.
template <int CT, int BT> __global__ void __launch_bounds__(256) ntt120_vmp_bt_kernel(VmpArgs p, uint32_t batch) {
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= 4 * p.n4) return;
    const PrimeRt pr(u / p.n4);
    const uint32_t c0 = blockIdx.y * CT, b0 = blockIdx.z * BT;
    const size_t poly_words = (size_t)4 * p.n4;
    const uint4 *pm = reinterpret_cast<const uint4 *>(p.pm) + u + (size_t)(p.col0 + c0) * poly_words;
    const int nc = min((uint32_t)CT, p.ncols_out - c0), nb = min((uint32_t)BT, batch - b0);
    unsigned long long acc[BT][CT][4];
#pragma unroll
    for (int b = 0; b < BT; b++)
#pragma unroll
        for (int c = 0; c < CT; c++) acc[b][c][0] = acc[b][c][1] = acc[b][c][2] = acc[b][c][3] = 0;
    for (uint32_t r0 = 0; r0 < p.row_max; r0 += 16) {
        const uint32_t r1 = min(r0 + 16, p.row_max);
        for (uint32_t r = r0; r < r1; r++) {
            const uint4 *mrow = pm + (size_t)r * p.C * poly_words;
            uint4 mv[CT], av[BT];
#pragma unroll
            for (int c = 0; c < CT; c++) mv[c] = c < nc ? __ldcs(mrow + (size_t)c * poly_words) : make_uint4(0, 0, 0, 0);
#pragma unroll
            for (int b = 0; b < BT; b++)
                av[b] = b < nb ? __ldg(reinterpret_cast<const uint4 *>(p.a + (size_t)(b0 + b) * p.a_bs) + u + (size_t)r * poly_words) : make_uint4(0, 0, 0, 0);
#pragma unroll
            for (int b = 0; b < BT; b++)
#pragma unroll
                for (int c = 0; c < CT; c++) {
                    acc[b][c][0] += (unsigned long long)av[b].x * mv[c].x;
                    acc[b][c][1] += (unsigned long long)av[b].y * mv[c].y;
                    acc[b][c][2] += (unsigned long long)av[b].z * mv[c].z;
                    acc[b][c][3] += (unsigned long long)av[b].w * mv[c].w;
                }
        }
#pragma unroll
        for (int b = 0; b < BT; b++)
#pragma unroll
            for (int c = 0; c < CT; c++)
#pragma unroll
                for (int i = 0; i < 4; i++) acc[b][c][i] = pr.reduce(acc[b][c][i]);
    }
#pragma unroll
    for (int b = 0; b < BT; b++)
#pragma unroll
        for (int c = 0; c < CT; c++)
            if (b < nb && c < nc)
                (reinterpret_cast<uint4 *>(p.res + (size_t)(b0 + b) * p.res_bs) + u + (size_t)(c0 + c) * poly_words)[0] =
                    make_uint4((uint32_t)acc[b][c][0], (uint32_t)acc[b][c][1], (uint32_t)acc[b][c][2], (uint32_t)acc[b][c][3]);
}

int ntt120_vmp(pgb_module *m, const char *a, uint64_t a_bs, char *res, uint64_t res_bs, const char *pm, uint64_t pm_bs,
               uint32_t row_max, uint32_t C, uint32_t col0, uint32_t ncols_out, uint32_t batch, uint32_t pm_div) {
    if (ncols_out == 0 || batch == 0) return PGB_OK;
    VmpArgs p = {a, a_bs, res, res_bs, pm, pm_bs, (uint32_t)(m->n / 4), row_max, C, col0, ncols_out, pm_div};
    const uint32_t words = (uint32_t)m->n; // uint4 words per poly
    dim3 block(256);
    const int ct_sel = (int)m->opt[PGB_OPT_VMP_CT];
    const uint64_t key_bytes = (uint64_t)row_max * C * 16 * m->n;
    if (pm_bs == 0 && batch >= 4 && key_bytes >= ((uint64_t)48 << 20) && !opt_on(m, PGB_OPT_VMP_NO_BT)) {
        ProfScope _ps(m, PROF_VMP);
        dim3 grid((words + 255) / 256, (ncols_out + 1) / 2, (batch + 3) / 4);
        ntt120_vmp_bt_kernel<2, 4><<<grid, block, 0, m->stream>>>(p, batch);
        PGB_CHECK_CUDA(cudaGetLastError());
        return PGB_OK;
    }
    // Output polys per thread: 2 (default), 4 or 8 (PGB_OPT_VMP_CT).  Measured on B200 (scripts/vmp_stream.py, profiles/r2_vmp_stream.md):
    // two polys per thread are never slower than four (streaming regime 0.88-0.94 of the measured copy bandwidth against 0.77-0.81, one
    // product of the largest sweep shape 0.88 against 0.71): the re-reads of `a` that a wider tile saves are L2 hits, while 52 registers
    // (5 CTAs / SM) instead of 78 (3 CTAs / SM) give the stream the loads in flight it needs and a finer wave granularity
    const int ct = ct_sel ? ct_sel : 2;
    { ProfScope _ps(m, PROF_VMP);
    if (ct == 2 || ncols_out <= 2) {
        dim3 grid((words + 255) / 256, (ncols_out + 1) / 2, batch);
        ntt120_vmp_kernel<2><<<grid, block, 0, m->stream>>>(p);
    } else if (ct == 8 && ncols_out >= 8) {
        dim3 grid((words + 255) / 256, (ncols_out + 7) / 8, batch);
        ntt120_vmp_kernel<8><<<grid, block, 0, m->stream>>>(p);
    } else {
        dim3 grid((words + 255) / 256, (ncols_out + 3) / 4, batch);
        ntt120_vmp_kernel<4><<<grid, block, 0, m->stream>>>(p);
    }
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

// The reference's NTT120 vmp computes the LAST output poly of an odd col_max < ncols from the paired-column block of the prepared layout read
// with the single-column stride (reference/ntt120/vmp.rs:262-273: vec_mat1col_product_x2 at `last * nrows * 16`): row i of the product
// takes matrix row i >> 1, column last + (i & 1).  "Identical to the reference on the same inputs" includes this, so the shape gets its
// own (cold) kernel instead of the mathematically defined product.
__global__ void __launch_bounds__(256) ntt120_vmp_odd_last_kernel(VmpArgs p, uint32_t last) {
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= 4 * p.n4) return;
    const PrimeRt pr(u / p.n4);
    const size_t poly_words = (size_t)4 * p.n4;
    const uint4 *a = reinterpret_cast<const uint4 *>(p.a + (size_t)blockIdx.z * p.a_bs) + u;
    const uint4 *pm = reinterpret_cast<const uint4 *>(p.pm + (size_t)(blockIdx.z / p.pm_div) * p.pm_bs) + u;
    unsigned long long acc[4] = {0, 0, 0, 0};
    for (uint32_t i = 0; i < p.row_max; i++) {
        const uint4 av = __ldg(a + (size_t)i * poly_words);
        const uint4 mv = __ldg(pm + ((size_t)(i >> 1) * p.C + last + (i & 1)) * poly_words);
        acc[0] += (unsigned long long)av.x * mv.x; acc[1] += (unsigned long long)av.y * mv.y;
        acc[2] += (unsigned long long)av.z * mv.z; acc[3] += (unsigned long long)av.w * mv.w;
        if ((i & 15) == 15)
#pragma unroll
            for (int j = 0; j < 4; j++) acc[j] = pr.reduce(acc[j]);
    }
    (reinterpret_cast<uint4 *>(p.res + (size_t)blockIdx.z * p.res_bs) + u)[0] =
        make_uint4(pr.reduce(acc[0]), pr.reduce(acc[1]), pr.reduce(acc[2]), pr.reduce(acc[3]));
}
int ntt120_vmp_odd_last(pgb_module *m, const char *a, uint64_t a_bs, char *res_poly, uint64_t res_bs, const char *pm, uint64_t pm_bs,
                        uint32_t row_max, uint32_t C, uint32_t last, uint32_t batch, uint32_t pm_div) {
    VmpArgs p = {a, a_bs, res_poly, res_bs, pm, pm_bs, (uint32_t)(m->n / 4), row_max, C, 0, 1, pm_div};
    ProfScope _ps(m, PROF_VMP);
    ntt120_vmp_odd_last_kernel<<<dim3(((uint32_t)m->n + 255) / 256, 1, batch), 256, 0, m->stream>>>(p, last);
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

// ---- element-wise over limb sets ---------------------------------------------------------------------

struct EwArgs {
    LimbSet dst, a, b;
    uint32_t n4;            // uint4 words per plane
    uint32_t jobs_per_batch;
};

__device__ __forceinline__ uint32_t addq(uint32_t x, uint32_t y, uint32_t q) { return csub(x + y, q); }
__device__ __forceinline__ uint32_t subq(uint32_t x, uint32_t y, uint32_t q) { return x >= y ? x - y : x - y + q; }
__device__ __forceinline__ uint32_t negq(uint32_t x, uint32_t q) { return x == 0 ? 0 : q - x; }

template <int OP> __global__ void __launch_bounds__(256) ntt120_ew_kernel(EwArgs p) {
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= 4 * p.n4) return;
    const PrimeRt pr(u / p.n4);
    const uint32_t q = pr.q;
    const uint32_t j = blockIdx.y, b = blockIdx.z;
    uint4 *dst = reinterpret_cast<uint4 *>(p.dst.base + (size_t)b * p.dst.batch_stride + (size_t)j * p.dst.limb_stride) + u;
    uint4 r = make_uint4(0, 0, 0, 0);
    if (OP != EW_ZERO) {
        const uint4 x = *(reinterpret_cast<const uint4 *>(p.a.base + (size_t)b * p.a.batch_stride + (size_t)j * p.a.limb_stride) + u);
        if (OP == EW_COPY) r = x;
        else if (OP == EW_NEG) r = make_uint4(negq(x.x % q, q), negq(x.y % q, q), negq(x.z % q, q), negq(x.w % q, q));
        else {
            const uint4 y = *(reinterpret_cast<const uint4 *>(p.b.base + (size_t)b * p.b.batch_stride + (size_t)j * p.b.limb_stride) + u);
            if (OP == EW_ADD) r = make_uint4(addq(x.x, y.x, q), addq(x.y, y.y, q), addq(x.z, y.z, q), addq(x.w, y.w, q));
            else if (OP == EW_SUB) r = make_uint4(subq(x.x, y.x, q), subq(x.y, y.y, q), subq(x.z, y.z, q), subq(x.w, y.w, q));
            else { // EW_MUL
                r = make_uint4(pr.reduce((unsigned long long)x.x * y.x), pr.reduce((unsigned long long)x.y * y.y),
                               pr.reduce((unsigned long long)x.z * y.z), pr.reduce((unsigned long long)x.w * y.w));
            }
        }
    }
    *dst = r;
}

// op over `jobs` limbs per batch item; a/b may alias dst limb for limb (pure element-wise)
int ntt120_ew(pgb_module *m, int op, LimbSet dst, LimbSet a, LimbSet b, uint32_t jobs, uint32_t batch) {
    if (jobs == 0 || batch == 0) return PGB_OK;
    ProfScope _ps(m, PROF_ELEMENTWISE);
    EwArgs p = {dst, a, b, (uint32_t)(m->n / 4), jobs};
    dim3 block(256), grid(((uint32_t)m->n + 255) / 256, jobs, batch);
    switch (op) {
    case EW_ADD: ntt120_ew_kernel<EW_ADD><<<grid, block, 0, m->stream>>>(p); break;
    case EW_SUB: ntt120_ew_kernel<EW_SUB><<<grid, block, 0, m->stream>>>(p); break;
    case EW_NEG: ntt120_ew_kernel<EW_NEG><<<grid, block, 0, m->stream>>>(p); break;
    case EW_COPY: ntt120_ew_kernel<EW_COPY><<<grid, block, 0, m->stream>>>(p); break;
    case EW_ZERO: ntt120_ew_kernel<EW_ZERO><<<grid, block, 0, m->stream>>>(p); break;
    default: ntt120_ew_kernel<EW_MUL><<<grid, block, 0, m->stream>>>(p); break;
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}
