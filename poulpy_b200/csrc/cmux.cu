// cmux.cu -- the CMux of poulpy-bin-fhe (glwe_sub, glwe_normalize_inplace, glwe_external_product_inplace, glwe_add_inplace,
// glwe_normalize_inplace), batched and device resident, with one prepared GGSW selector per ciphertext or one shared by the batch:
//
//     res = normalize( normalize(t - f) (x) s_b + f )
//
// t, f, res are GLWEs of rank k in base 2^base2k; s_b = s.data + b * ggsw_stride is a prepared GGSW (VmpPMat(dnum, k + 1, k + 1, size))
// in base 2^ggsw_base2k.  The difference kernel below writes normalize(t - f) in one pass; the external product and the final add +
// normalise run on the routes described at pgb_glwe_cmux_batched.
#include "internal.h"

// ---- d = normalize_assign(t - f) -------------------------------------------------------------------------------------------------------
// One thread per (coefficient, column, ciphertext).  Limb j < size of d is t[j] - f[j] in wrapping i64 (a limb missing from an operand
// reads as 0), normalised from the last limb up with the carry in a register: the lsh = 0 steps of vec_znx_normalize_assign
// (reference/vec_znx/normalize.rs:403-425), whose first step keeps only the digit and whose last step drops the carry.  `fr`, when set,
// receives f (limbs >= f_size zeroed) in the same pass: the FFT64 fused route adds it inside its carry chain.
struct CmuxDiffArgs {
    const char *t; uint64_t t_bs; // VecZnx(cols, t_size) per item, limb j at + j * words words
    const char *f; uint64_t f_bs; // VecZnx(cols, f_size)
    char *d;       uint64_t d_bs; // VecZnx(cols, size)
    char *fr;      uint64_t fr_bs; // VecZnx(cols, size) or null
    uint32_t words;               // n * cols: words per limb
    int t_size, f_size, size, K;
};
__global__ void __launch_bounds__(256) cmux_diff_kernel(CmuxDiffArgs p) {
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x; // column * n + coefficient
    if (u >= p.words) return;
    const size_t b = blockIdx.y, ls = p.words;
    const long long *t = reinterpret_cast<const long long *>(p.t + b * p.t_bs) + u;
    const long long *f = reinterpret_cast<const long long *>(p.f + b * p.f_bs) + u;
    long long *d = reinterpret_cast<long long *>(p.d + b * p.d_bs) + u;
    long long *fr = p.fr ? reinterpret_cast<long long *>(p.fr + b * p.fr_bs) + u : nullptr;
    const int sh = 64 - p.K;
    long long carry = 0;
    for (int j = p.size - 1; j >= 0; j--) {
        const long long tv = j < p.t_size ? __ldg(t + (size_t)j * ls) : 0;
        const long long fv = j < p.f_size ? __ldg(f + (size_t)j * ls) : 0;
        const long long x = (long long)((unsigned long long)tv - (unsigned long long)fv);
        const long long dg = (long long)((unsigned long long)x << sh) >> sh;                // get_digit
        const long long c = (long long)((unsigned long long)x - (unsigned long long)dg) >> p.K; // get_carry
        long long out;
        if (j == p.size - 1) {
            out = dg;
            carry = c;
        } else {
            const long long dc = (long long)((unsigned long long)dg + (unsigned long long)carry);
            out = (long long)((unsigned long long)dc << sh) >> sh;
            carry = (long long)((unsigned long long)c + (unsigned long long)(((long long)((unsigned long long)dc - (unsigned long long)out)) >> p.K));
        }
        d[(size_t)j * ls] = out;
        if (fr) fr[(size_t)j * ls] = fv;
    }
}

static int launch_diff(pgb_module *m, char *d, uint64_t d_bs, uint64_t size, const pgb_vec_znx *t, uint64_t t_bs, const pgb_vec_znx *f,
                       uint64_t f_bs, char *fr, uint64_t fr_bs, uint64_t base2k, uint64_t B) {
    const uint64_t words = m->n * t->cols;
    CmuxDiffArgs p = {(const char *)t->data, t_bs, (const char *)f->data, f_bs, d, d_bs, fr, fr_bs, (uint32_t)words, (int)t->size, (int)f->size,
                      (int)size, (int)base2k};
    { ProfScope _ps(m, PROF_NORMALIZE);
    cmux_diff_kernel<<<dim3((uint32_t)((words + 255) / 256), (uint32_t)B), 256, 0, m->stream>>>(p);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

// steps 4 and 5 on the routes that leave the external product in res: res[i] += f[i] (i < min(res.size, f.size)), normalize_assign
static int add_f_normalize(pgb_module *m, pgb_vec_znx *res, uint64_t res_bs, const pgb_vec_znx *f, uint64_t f_bs, uint64_t base2k, uint64_t B) {
    pgb_batch bta = {B, res_bs, f_bs, 0}, btn = {B, res_bs, 0, 0};
    for (uint64_t c = 0; c < res->cols; c++) {
        if (f->size) PGB_TRY(pgb_vec_znx_add_assign_batched(m, res, c, f, c, &bta));
        PGB_TRY(pgb_vec_znx_normalize_assign_batched(m, base2k, res, c, &btn));
    }
    return PGB_OK;
}

// ---- shape checks ------------------------------------------------------------------------------------------------------------------------
// data non-null and 16-byte aligned (the external-product kernels read GLWEs with 16-byte loads); the batch stride a multiple of 16 and at
// least one item, or 0 for a read-only operand shared by the batch
static int check_glwe(const char *name, const pgb_module *m, const pgb_vec_znx *v, uint64_t cols, uint64_t stride, uint64_t count, bool shared_ok) {
    PGB_REQUIRE(v->n == m->n, "glwe_cmux: %s has ring degree %llu, the module %llu", name, (unsigned long long)v->n, (unsigned long long)m->n);
    PGB_REQUIRE(v->cols == cols, "glwe_cmux: %s has %llu columns, the selector %llu", name, (unsigned long long)v->cols, (unsigned long long)cols);
    PGB_REQUIRE(v->size <= 65535, "glwe_cmux: %s has %llu limbs", name, (unsigned long long)v->size);
    PGB_REQUIRE(v->data != nullptr && (uintptr_t)v->data % 16 == 0, "glwe_cmux: %s data must be non-null and 16-byte aligned", name);
    const uint64_t item = v->n * v->cols * v->size * 8;
    PGB_REQUIRE(stride % 16 == 0 && (count == 1 || stride >= item || (shared_ok && stride == 0)),
                "glwe_cmux: %s batch stride %llu must be a multiple of 16 and at least one item (%llu bytes)%s", name, (unsigned long long)stride,
                (unsigned long long)item, shared_ok ? ", or 0" : "");
    return PGB_OK;
}

extern "C" size_t pgb_glwe_cmux_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t t_size, uint64_t f_size, uint64_t base2k,
                                          const pgb_vmp_pmat *s, uint64_t ggsw_base2k, uint64_t dsize, uint64_t batch) {
    (void)t_size; (void)f_size;
    // d (the difference, res.size limbs) | the external product's scratch for an input of res.size limbs, which also holds the buffers of the
    // fused routes (a_dft, and res_dft on FFT64)
    return align_up(batch * m->n * s->cols_in * res_size * 8) +
           pgb_glwe_external_product_tmp_bytes(m, res_size, res_size, base2k, s, ggsw_base2k, dsize, batch);
}

// Routes (all bit-exact with the five steps; DESIGN.md §3.5b):
//  * ggsw_stride == 0: d in scratch, then pgb_glwe_external_product_batched (with its single-kernel routes, gadget_fused in core.cu),
//    add f, normalise.
//  * per-item selectors, dsize == 1, ggsw_base2k == base2k, f.size <= min(res.size, s.size), fusion on:
//      NTT120 (n = 2^9 .. 2^13): d -> forward transform -> ntt120_fused_back with the per-item matrix stride and small = f on every column;
//      FFT64 (fft64_fused_back_supported): d and res = f -> forward transform -> vmp with the per-item matrix stride -> fft64_fused_back,
//      which adds res's own limbs inside its carry chain.
//    Both replace normalize(normalize(big) + f) by normalize(big + f): equal because f has no limb where the big integer is truncated.
//  * anything else: d -> (base conversion) -> the limb-wise external product with the per-item matrix stride -> add f, normalise.
extern "C" int pgb_glwe_cmux_batched(pgb_module *m, pgb_vec_znx *res, const pgb_vec_znx *t, const pgb_vec_znx *f, uint64_t base2k,
                                     const pgb_vmp_pmat *s, uint64_t ggsw_stride, uint64_t ggsw_base2k, uint64_t dsize, const pgb_batch *bt,
                                     void *scratch, size_t scratch_len) {
    PGB_REQUIRE(bt && bt->count >= 1 && bt->count <= 65535, "glwe_cmux: batch count must be in [1, 65535]");
    PGB_REQUIRE(res && t && f && s && s->data, "glwe_cmux: null argument");
    const uint64_t B = bt->count, n = m->n, pb = prep_bytes(m);
    PGB_REQUIRE(s->n == n, "glwe_cmux: the selector has ring degree %llu, the module %llu", (unsigned long long)s->n, (unsigned long long)n);
    PGB_REQUIRE(s->cols_in == s->cols_out && s->cols_in >= 1 && s->rows >= 1 && s->size >= 1,
                "glwe_cmux: the selector must be a non-empty VmpPMat(dnum, k + 1, k + 1, size)");
    const uint64_t cols = s->cols_in;
    PGB_TRY(check_glwe("res", m, res, cols, bt->stride_res, B, false));
    PGB_TRY(check_glwe("t", m, t, cols, bt->stride_a, B, true));
    PGB_TRY(check_glwe("f", m, f, cols, bt->stride_b, B, true));
    PGB_REQUIRE(res->size >= 1, "glwe_cmux: res must have at least one limb");
    PGB_REQUIRE(dsize >= 1, "glwe_cmux: dsize must be >= 1");
    PGB_REQUIRE(base2k >= 1 && base2k <= 63 && ggsw_base2k >= 1 && ggsw_base2k <= 63, "glwe_cmux: base2k and ggsw_base2k must be in [1, 63]");
    const uint64_t s_item = pgb_bytes_of_vmp_pmat(m, s->rows, cols, cols, s->size);
    PGB_REQUIRE((uintptr_t)s->data % 16 == 0 && (ggsw_stride == 0 || (ggsw_stride % 16 == 0 && ggsw_stride >= s_item)),
                "glwe_cmux: selector data must be 16-byte aligned and ggsw_stride 0 or a multiple of 16 of at least one prepared GGSW (%llu bytes)",
                (unsigned long long)s_item);
    const uint64_t need = pgb_glwe_cmux_tmp_bytes(m, res->size, t->size, f->size, base2k, s, ggsw_base2k, dsize, B);
    PGB_REQUIRE(scratch != nullptr && (uintptr_t)scratch % 256 == 0, "glwe_cmux: scratch must be non-null and 256-byte aligned");
    if (scratch_len < need) {
        pgb_set_error("glwe_cmux: scratch of %zu bytes < required %llu", scratch_len, (unsigned long long)need);
        return PGB_ERR_SCRATCH;
    }
    // res is written while t, f and the selectors are still read: no overlap at all (t and f are read-only and may overlap each other)
    const uint64_t res_ext = batch_extent(n * cols * res->size * 8, bt->stride_res, B);
    const uint64_t t_ext = batch_extent(n * cols * t->size * 8, bt->stride_a, B), f_ext = batch_extent(n * cols * f->size * 8, bt->stride_b, B);
    const uint64_t s_ext = batch_extent(s_item, ggsw_stride, B);
    if (ranges_overlap(res->data, res_ext, t->data, t_ext) || ranges_overlap(res->data, res_ext, f->data, f_ext) ||
        ranges_overlap(res->data, res_ext, s->data, s_ext)) {
        pgb_set_error("glwe_cmux: res must not overlap t, f or a selector");
        return PGB_ERR_ALIAS;
    }
    if (ranges_overlap(scratch, scratch_len, res->data, res_ext) || ranges_overlap(scratch, scratch_len, t->data, t_ext) ||
        ranges_overlap(scratch, scratch_len, f->data, f_ext) || ranges_overlap(scratch, scratch_len, s->data, s_ext)) {
        pgb_set_error("glwe_cmux: scratch must not overlap res, t, f or a selector");
        return PGB_ERR_ALIAS;
    }

    // ---- step 1 + 2 on every route: d = normalize(t - f), res.size limbs -----------------------------------------------------------------
    const uint64_t S = s->size, rs = res->size;
    const uint64_t d_bs = n * cols * rs * 8;
    Arena ar = {(char *)scratch, scratch_len, 0};
    char *sp = (char *)ar.take(B * d_bs);
    pgb_vec_znx d = mk(sp, n, cols, rs);

    if (ggsw_stride == 0) { // one selector for the batch: the external product with every route it has
        PGB_TRY(launch_diff(m, sp, d_bs, rs, t, bt->stride_a, f, bt->stride_b, nullptr, 0, base2k, B));
        pgb_batch bte = {B, bt->stride_res, d_bs, 0};
        PGB_TRY(pgb_glwe_external_product_batched(m, res, base2k, &d, base2k, s, ggsw_base2k, dsize, &bte, ar.rest(), ar.rest_len()));
        return add_f_normalize(m, res, bt->stride_res, f, bt->stride_b, base2k, B);
    }

    const bool fuse = dsize == 1 && ggsw_base2k == base2k && f->size <= umin64(rs, S) && !opt_on(m, PGB_OPT_NO_FUSION);
    const uint64_t R = umin64(s->rows * cols, cols * rs); // rows of the vector-matrix product (external_product/glwe.rs:231)
    const uint64_t a_dft_bs = n * cols * rs * pb, res_dft_bs = n * cols * S * pb;
    if (fuse && ntt120_fused_supported(m)) {
        char *a_dft = (char *)ar.take(B * a_dft_bs);
        PGB_TRY(launch_diff(m, sp, d_bs, rs, t, bt->stride_a, f, bt->stride_b, nullptr, 0, base2k, B));
        LimbSet in = {sp, n * 8, d_bs}, out = {a_dft, n * pb, a_dft_bs}; // polys (limb, column) are consecutive on both sides
        PGB_TRY(ntt120_forward(m, in, out, (int)(rs * cols), (int)B));
        return ntt120_fused_back(m, a_dft, a_dft_bs, (const char *)s->data, (int)R, (int)(cols * S), (int)cols, (const char *)f->data, bt->stride_b,
                                 cols * n * 8, (int)f->size, (char *)res->data, bt->stride_res, cols * n * 8, (int)rs, (int)base2k, 0, (int)B,
                                 nullptr, 0, 0, nullptr, false, false, true, ggsw_stride);
    }
    if (fuse && fft64_fused_back_supported(m, (int)S)) {
        char *res_dft = (char *)ar.take(B * res_dft_bs), *a_dft = (char *)ar.take(B * a_dft_bs);
        PGB_TRY(launch_diff(m, sp, d_bs, rs, t, bt->stride_a, f, bt->stride_b, (char *)res->data, bt->stride_res, base2k, B));
        LimbSet in = {sp, n * 8, d_bs}, out = {a_dft, n * pb, a_dft_bs};
        PGB_TRY(fft64_forward(m, in, out, (int)(rs * cols), (int)B));
        pgb_vec_znx_dft rd = {res_dft, n, cols, S, S}, ad = {a_dft, n, cols, rs, rs};
        pgb_batch btv = {B, res_dft_bs, a_dft_bs, ggsw_stride};
        PGB_TRY(vmp_apply_impl(m, &rd, &ad, s, 0, &btv));
        return fft64_fused_back(m, res_dft, res_dft_bs, (int)cols, (int)S, (char *)res->data, bt->stride_res, (int)rs, (int)base2k, (int)B);
    }

    // ---- limb-wise: the external product's HAL sequence with the per-item matrix stride -----------------------------------------------
    pgb_vec_znx_dft res_dft = mk(ar.take(B * res_dft_bs), n, cols, S);
    PGB_TRY(launch_diff(m, sp, d_bs, rs, t, bt->stride_a, f, bt->stride_b, nullptr, 0, base2k, B));
    pgb_vec_znx ain; // the input in ggsw_base2k, as the external product does
    uint64_t ain_bs;
    PGB_TRY(glwe_to_base2k(m, ar, &d, d_bs, base2k, ggsw_base2k, B, &ain, &ain_bs));
    const uint64_t a_dft_max = div_ceil64(ain.size, dsize);
    pgb_vec_znx_dft a_dft = mk(ar.take(B * n * cols * a_dft_max * pb), n, cols, a_dft_max);
    void *tmp = dsize > 1 ? ar.take(B * res_dft_bs) : nullptr;
    PGB_REQUIRE(res_dft.data && ain.data && a_dft.data && (dsize == 1 || tmp), "glwe_cmux: scratch exhausted");
    PGB_TRY(external_product_limbwise(m, res, bt->stride_res, base2k, &ain, ain_bs, s, ggsw_stride, ggsw_base2k, dsize, B, &res_dft, &a_dft, tmp));
    return add_f_normalize(m, res, bt->stride_res, f, bt->stride_b, base2k, B);
}
