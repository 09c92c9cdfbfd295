// core.cu -- CoreImpl-tier batched pipelines: GLWE key-switch (C1) and GGSW x GLWE external product (C2), device resident,
// plus the host-buffer front ends that stage through pinned memory.
//
// The call sequences restate poulpy-core/src/keyswitching/glwe.rs:53-109, :207-239, :298-380 and
// poulpy-core/src/external_product/glwe.rs:99-141, :197-271; every step runs over the whole batch on the module's
// stream with no host round trip in between.
#include <stdlib.h>

#include <string>
#include <thread>
#include <vector>

#include "internal.h"

// glwe_normalize (poulpy-core/src/operations/glwe.rs:1286-1310) into a buffer of size ceil(a.size*a_base2k / base2k)
static uint64_t conv_size(uint64_t a_size, uint64_t a_base2k, uint64_t base2k) { return div_ceil64(a_size * a_base2k, base2k); }

int glwe_to_base2k(pgb_module *m, Arena &ar, const pgb_vec_znx *a, uint64_t a_bs, uint64_t from, uint64_t to, uint64_t B, pgb_vec_znx *out,
                   uint64_t *out_bs) {
    *out = *a;
    *out_bs = a_bs;
    if (from == to) return PGB_OK;
    const uint64_t cs = conv_size(a->size, from, to);
    *out_bs = m->n * a->cols * cs * 8;
    *out = mk(ar.take(B * *out_bs), m->n, a->cols, cs);
    pgb_batch btn = {B, *out_bs, a_bs, 0};
    for (uint64_t i = 0; i < a->cols; i++) PGB_TRY(big_normalize_impl(m, out, to, 0, i, a, from, i, 0, false, &btn));
    return PGB_OK;
}

// ---- gglwe_product_dft (keyswitching/glwe.rs:298-380) ---------------------------------------------------------------------------
// res_dft(cols_out, pmat.size) <- a_dft(cols, a_size) x pmat ; ai / tmp are scratch DFT buffers for dsize > 1.
static int gadget_product(pgb_module *m, pgb_vec_znx_dft *res, const pgb_vec_znx_dft *a, const pgb_vmp_pmat *pmat, uint64_t dsize,
                          pgb_vec_znx_dft *ai, pgb_vec_znx_dft *tmp, uint64_t res_bs, uint64_t a_bs, uint64_t ai_bs, uint64_t tmp_bs,
                          uint64_t batch) {
    if (dsize == 1) {
        pgb_batch bt = {batch, res_bs, a_bs, 0};
        return vmp_apply_impl(m, res, a, pmat, 0, &bt);
    }
    const uint64_t a_size = a->size, dnum = pmat->rows, cols = a->cols, cols_out = res->cols;
    const uint64_t res_max = res->size;
    for (uint64_t di = 0; di < dsize; di++) {
        ai->size = umin64((a_size + di) / dsize, dnum);
        const int64_t cut = (int64_t)(dsize - di) - 2;
        res->size = pmat->size - (uint64_t)(cut > 0 ? cut : 0);
        pgb_batch btc = {batch, ai_bs, a_bs, 0};
        for (uint64_t j = 0; j < cols; j++) PGB_TRY(pgb_vec_znx_dft_copy_batched(m, dsize, dsize - di - 1, ai, j, a, j, &btc));
        if (di == 0) {
            pgb_batch bt = {batch, res_bs, ai_bs, 0};
            PGB_TRY(vmp_apply_impl(m, res, ai, pmat, 0, &bt));
        } else {
            tmp->size = res->size;
            pgb_batch bt = {batch, tmp_bs, ai_bs, 0};
            PGB_TRY(vmp_apply_impl(m, tmp, ai, pmat, di, &bt));
            pgb_batch bta = {batch, res_bs, tmp_bs, 0};
            for (uint64_t c = 0; c < cols_out; c++) PGB_TRY(pgb_vec_znx_dft_add_assign_batched(m, res, c, tmp, c, &bta));
        }
    }
    res->size = res_max;
    return PGB_OK;
}

// The collapsed key needs |V| < 2^118: bits(a) + bits(key) + ceil(log2(R n)) + (S - 1) K + 3 <= 118 (decided exactly on the device).  With
// dsize > 1 a flagged ciphertext costs a redo of the whole batch, so the single-kernel route is only tried when normalised operands
// (K-bit digits on both sides) would pass; long keys (S K beyond ~85 bits) go straight to the limb-wise sequence.
static bool gadget_likely_fits(uint64_t n, uint64_t R, uint64_t S, uint64_t K) {
    uint64_t rn = 0;
    while (((uint64_t)1 << rn) < R * n) rn++;
    return rn + (S - 1) * K + 3 + 2 * K <= 118;
}

// glwe_keyswitch_internal (keyswitching/glwe.rs:207-239) from the transformed input on: res_dft <- a_dft x key, left in res_dft as a big
// (ScalarBig elements, same memory).  For dsize > 1 the digit buffer ai and the temporary come from `ar` for this call only, so a caller
// that runs several products gets the same buffers each time.
static int keyswitch_core(pgb_module *m, Arena &ar, const char *what, pgb_vec_znx_dft *res_dft, uint64_t res_dft_bs, const pgb_vec_znx_dft *a_dft,
                          uint64_t a_dft_bs, const pgb_vmp_pmat *key, uint64_t dsize, uint64_t B) {
    const uint64_t n = m->n, pb = prep_bytes(m);
    const size_t mark = ar.used;
    pgb_vec_znx_dft ai = *a_dft, tmp = *res_dft;
    uint64_t ai_bs = 0, tmp_bs = 0;
    if (dsize > 1) {
        const uint64_t ai_max = umin64(div_ceil64(a_dft->size, dsize), key->rows);
        ai_bs = n * a_dft->cols * ai_max * pb;
        ai = mk(ar.take(B * ai_bs), n, a_dft->cols, ai_max);
        tmp_bs = res_dft_bs;
        tmp = mk(ar.take(B * tmp_bs), n, res_dft->cols, key->size);
        PGB_REQUIRE(ai.data && tmp.data, "%s: scratch exhausted", what);
        PGB_CHECK_CUDA(cudaMemsetAsync(ai.data, 0, B * ai_bs, m->stream));   // ai_dft.zero()       (:337)
        PGB_CHECK_CUDA(cudaMemsetAsync(tmp.data, 0, B * tmp_bs, m->stream)); // res_dft_tmp.zero()  (:342)
    }
    ar.used = mark;
    PGB_CHECK_CUDA(cudaMemsetAsync(res_dft->data, 0, B * res_dft_bs, m->stream)); // res_dft.zero() (:90)
    PGB_TRY(gadget_product(m, res_dft, a_dft, key, dsize, &ai, &tmp, res_dft_bs, a_dft_bs, ai_bs, tmp_bs, B));
    pgb_batch btc = {B, res_dft_bs, 0, 0};
    return pgb_vec_znx_idft_apply_consume_batched(m, res_dft, &btc);
}

// ---- the single-kernel gadget product ---------------------------------------------------------------------------------------------
// One product res <- a x key as the gadget kernels (fft64_gadget.cu, ntt120_gadget.cu) see it.  a is in the key's base 2^base2k; rows of
// the product are the columns row_col0 .. row_col0 + key.cols_in of a (row_col0 = 1 for the key-switch family, whose column 0 is added to
// output column 0, 0 for the external product).
struct GadgetJob {
    const pgb_vec_znx *a;
    uint64_t a_bs, row_col0;
    const pgb_vmp_pmat *key;
    uint64_t dsize, base2k;
    int small_size;  // limbs of column 0 of a added to the output
    int group_limit; // bound on the limbs of a digit group (dnum for the key-switch family, 0 = none for the external product)
    int aut_mode;    // 0: none; 1..3: X -> X^aut_p, then add / sub / sub_negate a (post_size limbs); 4: X -> X^aut_p only
    int64_t aut_p;
    int post_size;
    pgb_vec_znx *res;
    uint64_t res_bs;
    int alias; // vec_znx_alias_class(res, a): nonzero when res overlaps a
    uint64_t B;
};

// Runs the job on a single-kernel route when one fits: returns 1 when the batch is done, 0 when the caller must run the limb-wise
// sequence, < 0 on error.  Routes:
//  * FFT64, dsize <= 2: the gadget kernel, with nothing to check after the launch.
//  * NTT120, dsize == 1, no automorphism: the gadget kernel, then the ciphertexts it flagged (integers that could leave the collapsed-key
//    bound) are redone on the device by the forward transform and the fused back end of their skip list: no host round trip.  Without
//    the gadget kernel, the forward transform into a_dft and the fused back end (vmp -> idft -> CRT -> add_small -> normalize).
//  * NTT120, dsize > 1 (when gadget_likely_fits) or automorphism: the gadget kernel, then the count of flagged ciphertexts is read back;
//    any flagged one sends the whole batch to the limb-wise sequence.
// The output is staged when res overlaps a and the kernel cannot write over a: the automorphism epilogue gathers a at permuted positions,
// and after a read-back the limb-wise sequence must still find a intact.  The staging buffer is `stage` when given (used only if
// stage_cap bytes per item hold the output), else taken from `ar`; when none can be had the route is skipped.  ar supplies the flag list.
static int gadget_fused(pgb_module *m, const GadgetJob &j, Arena &ar, pgb_vec_znx_dft *a_dft, uint64_t a_dft_bs, char *stage_buf,
                        uint64_t stage_cap) {
    if (opt_on(m, PGB_OPT_NO_FUSION)) return 0;
    const pgb_vec_znx &a = *j.a, &res = *j.res;
    const pgb_vmp_pmat &key = *j.key;
    const uint64_t n = m->n, B = j.B, row_cols = key.cols_in, cols_out = key.cols_out, key_rows = key.rows * key.cols_in;
    const uint64_t R = j.dsize == 1 ? umin64(key_rows, row_cols * a.size) : row_cols * a.size;
    const int C = (int)(cols_out * key.size), S = (int)key.size, K = (int)j.base2k;
    const bool f64 = j.dsize <= 2 && fft64_gadget_supported(m, (int)R, (int)cols_out, S, K, (int)B);
    const bool gadget = f64 || ntt120_gadget_supported(m, (int)R, (int)cols_out, S, K, (int)B);
    const bool plain = j.dsize == 1 && j.aut_mode == 0, skip_list = plain && !f64, read_back = !f64 && !plain;
    if (!gadget && !(skip_list && ntt120_fused_supported(m))) return 0;
    if (read_back && j.dsize > 1 && !gadget_likely_fits(n, R, key.size, j.base2k)) return 0;
    // column 0 of a is the small term of the key-switch family's fused back end
    const char *small = j.row_col0 ? (const char *)a.data : nullptr;
    const uint64_t small_bs = j.row_col0 ? j.a_bs : 0, small_ls = j.row_col0 ? a.cols * n * 8 : 0;
    if (!gadget) {
        pgb_batch btd = {B, a_dft_bs, j.a_bs, 0};
        for (uint64_t c = 0; c < row_cols; c++) PGB_TRY(pgb_vec_znx_dft_apply_batched(m, 1, 0, a_dft, c, &a, c + j.row_col0, &btd));
        PGB_TRY(ntt120_fused_back(m, (const char *)a_dft->data, a_dft_bs, (const char *)key.data, (int)R, C, (int)cols_out, small, small_bs,
                                  small_ls, j.small_size, (char *)res.data, j.res_bs, res.cols * n * 8, (int)res.size, K, 0, (int)B,
                                  (const char *)a.data, j.a_bs, n * a.cols * a.size));
        return 1;
    }
    const size_t mark = ar.used;
    int *ok = (int *)ar.take((2 * B + 1) * sizeof(int)); // flags | count of flagged | their indices
    const bool stage = j.alias != 0 && (j.aut_mode != 0 || read_back);
    char *out = (char *)res.data;
    uint64_t out_bs = j.res_bs;
    if (stage) {
        out_bs = n * cols_out * res.size * 8;
        out = stage_buf ? (out_bs <= stage_cap ? stage_buf : nullptr) : (char *)ar.take(B * out_bs);
    }
    if (!ok || !out) {
        ar.used = mark;
        return 0;
    }
    // a plain dsize-1 product passes no digit-group geometry: its pinned-key signature then does not depend on a.size
    const int a_size = plain ? 0 : (int)a.size, g_rows = plain ? 0 : (int)key_rows, g_limit = plain ? 0 : j.group_limit;
    if (f64)
        PGB_TRY(fft64_gadget_fused(m, (const char *)a.data, j.a_bs, (int)a.cols, (int)row_cols, (int)j.row_col0, (int)R, (const char *)key.data, C,
                                   (int)cols_out, j.small_size, out, out_bs, (int)res.size, K, (int)B, (int)j.dsize, a_size, g_rows, g_limit,
                                   j.aut_mode, j.aut_p, j.post_size));
    else
        PGB_TRY(ntt120_gadget_fused(m, (const char *)a.data, j.a_bs, (int)a.cols, (int)row_cols, (int)j.row_col0, (int)R, (const char *)key.data, C,
                                    (int)cols_out, j.small_size, out, out_bs, (int)res.size, K, (int)B, ok, (int)j.dsize, a_size, g_rows, g_limit,
                                    j.aut_mode, j.aut_p, j.post_size));
    if (skip_list) {
        const uint64_t pb = prep_bytes(m);
        for (uint64_t c = 0; c < row_cols; c++) {
            LimbSet in = {(char *)a.data + limb_off(n, a.cols, c + j.row_col0, 0, 8), a.cols * n * 8, j.a_bs};
            LimbSet o = {(char *)a_dft->data + limb_off(n, row_cols, c, 0, pb), row_cols * n * pb, a_dft_bs};
            PGB_TRY(ntt120_forward_skip(m, in, o, (int)a.size, (int)B, ok, true));
        }
        PGB_TRY(ntt120_fused_back(m, (const char *)a_dft->data, a_dft_bs, (const char *)key.data, (int)R, C, (int)cols_out, small, small_bs,
                                  small_ls, j.small_size, (char *)res.data, j.res_bs, res.cols * n * 8, (int)res.size, K, 0, (int)B, nullptr, 0,
                                  0, ok, true));
        return 1;
    }
    if (read_back) {
        int nfail = 0;
        PGB_CHECK_CUDA(cudaMemcpyAsync(&nfail, ok + B, sizeof(int), cudaMemcpyDeviceToHost, m->stream));
        PGB_CHECK_CUDA(cudaStreamSynchronize(m->stream));
        if (nfail != 0) {
            ar.used = mark;
            return 0;
        }
    }
    if (stage) PGB_CHECK_CUDA(cudaMemcpy2DAsync(res.data, j.res_bs, out, out_bs, out_bs, B, cudaMemcpyDeviceToDevice, m->stream));
    return 1;
}

// ---- key-switch --------------------------------------------------------------------------------------------------------
extern "C" size_t pgb_glwe_keyswitch_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t a_base2k,
                                               const pgb_vmp_pmat *key, uint64_t key_base2k, uint64_t dsize, uint64_t batch) {
    (void)res_size;
    const uint64_t n = m->n, pb = prep_bytes(m);
    const uint64_t rank_in = key->cols_in, cols_out = key->cols_out;
    const uint64_t in_size = a_base2k == key_base2k ? a_size : conv_size(a_size, a_base2k, key_base2k);
    uint64_t t = 0;
    t += align_up(batch * n * cols_out * key->size * pb);                       // res_dft
    t += align_up(batch * n * rank_in * in_size * pb);                          // a_dft
    if (a_base2k != key_base2k) t += align_up(batch * n * (rank_in + 1) * in_size * 8); // a_conv
    if (dsize > 1) {
        t += align_up(batch * n * rank_in * div_ceil64(in_size, dsize) * pb);   // ai_dft
        t += align_up(batch * n * cols_out * key->size * pb);                   // res_dft_tmp
    }
    t += align_up((2 * batch + 1) * sizeof(int));                               // per-ciphertext route flags of the fused kernel + fail list
    return t + ALIGN;
}

extern "C" int pgb_glwe_keyswitch_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a, uint64_t a_base2k,
                                          const pgb_vmp_pmat *key, uint64_t key_base2k, uint64_t dsize, const pgb_batch *bt, void *scratch,
                                          size_t scratch_len) {
    PGB_REQUIRE(bt && bt->count >= 1 && bt->count <= 65535, "glwe_keyswitch: batch count must be in [1, 65535]");
    PGB_REQUIRE(res->n == m->n && a->n == m->n && key->n == m->n, "glwe_keyswitch: ring degree mismatch");
    PGB_REQUIRE(a->cols == key->cols_in + 1, "glwe_keyswitch: a.rank() != key.rank_in()");   // keyswitching/glwe.rs:59-65
    PGB_REQUIRE(res->cols == key->cols_out, "glwe_keyswitch: res.rank() != key.rank_out()"); // :66-72
    PGB_REQUIRE(dsize >= 1, "glwe_keyswitch: dsize must be >= 1");
    const uint64_t need = pgb_glwe_keyswitch_tmp_bytes(m, res->size, a->size, a_base2k, key, key_base2k, dsize, bt->count);
    if (scratch_len < need) {
        pgb_set_error("glwe_keyswitch: scratch of %zu bytes < required %llu", scratch_len, (unsigned long long)need);
        return PGB_ERR_SCRATCH;
    }
    const uint64_t n = m->n, pb = prep_bytes(m), B = bt->count;
    const uint64_t rank_in = key->cols_in, cols_out = key->cols_out;
    // res may BE a (glwe_keyswitch_assign, keyswitching/glwe.rs:111-165: same pointer, rank and stride); any other overlap is rejected
    const int alias = vec_znx_alias_class(res, bt->stride_res, a, bt->stride_a, B);
    if (alias < 0) {
        pgb_set_error("glwe_keyswitch: res and a overlap without being the same ciphertexts (in place needs equal pointer, rank and stride)");
        return PGB_ERR_ALIAS;
    }
    Arena ar = {(char *)scratch, scratch_len, 0};

    // (:89-90) res_dft = take_vec_znx_dft(rank_out + 1, key.size()); zero
    const uint64_t res_dft_bs = n * cols_out * key->size * pb;
    pgb_vec_znx_dft res_dft = mk(ar.take(B * res_dft_bs), n, cols_out, key->size);
    // (:92-100) cross-base2k input conversion
    pgb_vec_znx ain;
    uint64_t ain_bs;
    PGB_TRY(glwe_to_base2k(m, ar, a, bt->stride_a, a_base2k, key_base2k, B, &ain, &ain_bs));
    // glwe_keyswitch_internal (:207-239)
    const uint64_t a_dft_bs = n * rank_in * ain.size * pb;
    pgb_vec_znx_dft a_dft = mk(ar.take(B * a_dft_bs), n, rank_in, ain.size);
    if (res_base2k == key_base2k) { // one kernel per batch; in place, its output is staged in the res_dft block, still unused here
        const GadgetJob job = {&ain, ain_bs, 1, key, dsize, key_base2k, (int)umin64(ain.size, key->size), (int)key->rows, 0, 0, 0,
                               res, bt->stride_res, alias, B};
        const int done = gadget_fused(m, job, ar, &a_dft, a_dft_bs, (char *)res_dft.data, res_dft_bs);
        if (done) return done < 0 ? done : PGB_OK;
    }
    pgb_batch btd = {B, a_dft_bs, ain_bs, 0};
    for (uint64_t c = 0; c < rank_in; c++) PGB_TRY(pgb_vec_znx_dft_apply_batched(m, 1, 0, &a_dft, c, &ain, c + 1, &btd));
    PGB_TRY(keyswitch_core(m, ar, "glwe_keyswitch", &res_dft, res_dft_bs, &a_dft, a_dft_bs, key, dsize, B));
    pgb_vec_znx_big res_big = res_dft; // same memory, ScalarBig elements
    pgb_batch bts = {B, res_dft_bs, ain_bs, 0};
    PGB_TRY(big_add_small_impl(m, &res_big, 0, &ain, 0, &bts));
    // (:106-108)
    pgb_batch btn = {B, bt->stride_res, res_dft_bs, 0};
    for (uint64_t i = 0; i < res->cols; i++)
        PGB_TRY(big_normalize_impl(m, res, res_base2k, 0, i, &res_big, key_base2k, i, 0, true, &btn));
    return PGB_OK;
}

// ---- external product ------------------------------------------------------------------------------------------------------
extern "C" size_t pgb_glwe_external_product_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t a_base2k,
                                                      const pgb_vmp_pmat *ggsw, uint64_t ggsw_base2k, uint64_t dsize, uint64_t batch) {
    (void)res_size;
    const uint64_t n = m->n, pb = prep_bytes(m);
    const uint64_t cols = ggsw->cols_in;
    const uint64_t in_size = a_base2k == ggsw_base2k ? a_size : conv_size(a_size, a_base2k, ggsw_base2k);
    uint64_t t = 0;
    t += align_up(batch * n * cols * ggsw->size * pb);
    t += align_up(batch * n * cols * in_size * pb); // a_dft (dsize == 1 uses a_size limbs, dsize > 1 uses <= a_size)
    if (a_base2k != ggsw_base2k) t += align_up(batch * n * cols * in_size * 8);
    if (dsize > 1) t += align_up(batch * n * cols * ggsw->size * pb);
    t += align_up((2 * batch + 1) * sizeof(int)); // per-ciphertext route flags of the fused kernel + fail list
    return t + ALIGN;
}

extern "C" int pgb_glwe_external_product_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a,
                                                 uint64_t a_base2k, const pgb_vmp_pmat *ggsw, uint64_t ggsw_base2k, uint64_t dsize,
                                                 const pgb_batch *bt, void *scratch, size_t scratch_len) {
    PGB_REQUIRE(bt && bt->count >= 1 && bt->count <= 65535, "glwe_external_product: batch count must be in [1, 65535]");
    PGB_REQUIRE(res->n == m->n && a->n == m->n && ggsw->n == m->n, "glwe_external_product: ring degree mismatch");
    PGB_REQUIRE(a->cols == ggsw->cols_in && res->cols == ggsw->cols_out && ggsw->cols_in == ggsw->cols_out,
                "glwe_external_product: rank mismatch");                                     // external_product/glwe.rs:106-107
    PGB_REQUIRE(dsize >= 1, "glwe_external_product: dsize must be >= 1");
    const uint64_t need = pgb_glwe_external_product_tmp_bytes(m, res->size, a->size, a_base2k, ggsw, ggsw_base2k, dsize, bt->count);
    if (scratch_len < need) {
        pgb_set_error("glwe_external_product: scratch of %zu bytes < required %llu", scratch_len, (unsigned long long)need);
        return PGB_ERR_SCRATCH;
    }
    const uint64_t n = m->n, pb = prep_bytes(m), B = bt->count, cols = ggsw->cols_in;
    // res may BE a (glwe_external_product_assign, external_product/glwe.rs:143-195); any other overlap is rejected
    const int alias = vec_znx_alias_class(res, bt->stride_res, a, bt->stride_a, B);
    if (alias < 0) {
        pgb_set_error("glwe_external_product: res and a overlap without being the same ciphertexts (in place needs equal pointer and stride)");
        return PGB_ERR_ALIAS;
    }
    Arena ar = {(char *)scratch, scratch_len, 0};
    const uint64_t res_dft_bs = n * cols * ggsw->size * pb;
    pgb_vec_znx_dft res_dft = mk(ar.take(B * res_dft_bs), n, cols, ggsw->size);
    pgb_vec_znx ain;
    uint64_t ain_bs;
    PGB_TRY(glwe_to_base2k(m, ar, a, bt->stride_a, a_base2k, ggsw_base2k, B, &ain, &ain_bs));
    // glwe_external_product_internal (:197-271)
    const uint64_t a_dft_max = div_ceil64(ain.size, dsize);
    const uint64_t a_dft_bs = n * cols * a_dft_max * pb;
    pgb_vec_znx_dft a_dft = mk(ar.take(B * a_dft_bs), n, cols, a_dft_max);
    if (res_base2k == ggsw_base2k) { // as in the key-switch; no bound on the limbs of a digit group here (:233)
        const GadgetJob job = {&ain, ain_bs, 0, ggsw, dsize, ggsw_base2k, 0, 0, 0, 0, 0, res, bt->stride_res, alias, B};
        const int done = gadget_fused(m, job, ar, &a_dft, a_dft_bs, (char *)res_dft.data, res_dft_bs);
        if (done) return done < 0 ? done : PGB_OK;
    }
    void *tmp = nullptr;
    if (dsize > 1) {
        tmp = ar.take(B * res_dft_bs);
        PGB_REQUIRE(tmp, "glwe_external_product: scratch exhausted");
    }
    return external_product_limbwise(m, res, bt->stride_res, res_base2k, &ain, ain_bs, ggsw, 0, ggsw_base2k, dsize, B, &res_dft, &a_dft, tmp);
}

// glwe_external_product_internal (:197-271) as the limb-wise HAL sequence, then the normalisation into res (:138-140).  ain is already in
// ggsw_base2k; res_dft (cols, ggsw.size), a_dft (cols, ceil(ain.size / dsize)) and, for dsize > 1, `tmp` (the size of res_dft) are the
// caller's scratch.  ggsw_bs strides the GGSW per item (0: one GGSW for the whole batch).
int external_product_limbwise(pgb_module *m, pgb_vec_znx *res, uint64_t res_bs, uint64_t res_base2k, const pgb_vec_znx *ain, uint64_t ain_bs,
                              const pgb_vmp_pmat *ggsw, uint64_t ggsw_bs, uint64_t ggsw_base2k, uint64_t dsize, uint64_t B,
                              pgb_vec_znx_dft *res_dft, pgb_vec_znx_dft *a_dft, void *tmp_data) {
    const uint64_t n = m->n, pb = prep_bytes(m), cols = ggsw->cols_in, a_size = ain->size;
    const uint64_t res_dft_bs = n * cols * ggsw->size * pb, a_dft_bs = n * cols * a_dft->size * pb;
    if (dsize == 1) {
        pgb_batch btd = {B, a_dft_bs, ain_bs, 0};
        for (uint64_t j = 0; j < cols; j++) PGB_TRY(pgb_vec_znx_dft_apply_batched(m, 1, 0, a_dft, j, ain, j, &btd));
        PGB_CHECK_CUDA(cudaMemsetAsync(res_dft->data, 0, B * res_dft_bs, m->stream)); // res_dft.zero() (:123)
        pgb_batch btv = {B, res_dft_bs, a_dft_bs, ggsw_bs};
        PGB_TRY(vmp_apply_impl(m, res_dft, a_dft, ggsw, 0, &btv));
    } else {
        PGB_CHECK_CUDA(cudaMemsetAsync(res_dft->data, 0, B * res_dft_bs, m->stream)); // res_dft.zero() (:123)
        pgb_vec_znx_dft tmp = mk(tmp_data, n, cols, ggsw->size);
        // the temporary starts zeroed (a fresh allocation in the oracle's model of the scratch arena): with dsize > 1 the FFT64 vmp leaves
        // limbs past the shifted key untouched, so the result must not depend on what a reused scratch held before
        PGB_CHECK_CUDA(cudaMemsetAsync(tmp.data, 0, B * res_dft_bs, m->stream));
        // a_dft.data_mut().fill(0) (:226): FFT64 dft_apply leaves limbs past a.size untouched inside min_steps
        PGB_CHECK_CUDA(cudaMemsetAsync(a_dft->data, 0, B * a_dft_bs, m->stream));
        for (uint64_t di = 0; di < dsize; di++) {
            a_dft->size = (a_size + di) / dsize;
            const int64_t cut = (int64_t)(dsize - di) - 2;
            res_dft->size = ggsw->size - (uint64_t)(cut > 0 ? cut : 0);
            pgb_batch btd = {B, a_dft_bs, ain_bs, 0};
            for (uint64_t j = 0; j < cols; j++) PGB_TRY(pgb_vec_znx_dft_apply_batched(m, dsize, dsize - 1 - di, a_dft, j, ain, j, &btd));
            if (di == 0) {
                pgb_batch btv = {B, res_dft_bs, a_dft_bs, ggsw_bs};
                PGB_TRY(vmp_apply_impl(m, res_dft, a_dft, ggsw, 0, &btv));
            } else {
                tmp.size = res_dft->size;
                pgb_batch btv = {B, res_dft_bs, a_dft_bs, ggsw_bs};
                PGB_TRY(vmp_apply_impl(m, &tmp, a_dft, ggsw, di, &btv));
                pgb_batch bta = {B, res_dft_bs, res_dft_bs, 0};
                for (uint64_t c = 0; c < cols; c++) PGB_TRY(pgb_vec_znx_dft_add_assign_batched(m, res_dft, c, &tmp, c, &bta));
            }
        }
        res_dft->size = ggsw->size;
    }
    pgb_batch btc = {B, res_dft_bs, 0, 0};
    PGB_TRY(pgb_vec_znx_idft_apply_consume_batched(m, res_dft, &btc));
    pgb_vec_znx_big res_big = *res_dft;
    pgb_batch btn = {B, res_bs, res_dft_bs, 0};
    for (uint64_t j = 0; j < res->cols; j++)
        PGB_TRY(big_normalize_impl(m, res, res_base2k, 0, j, &res_big, ggsw_base2k, j, 0, true, &btn));
    return PGB_OK;
}

// ---- GLWE tensoring and relinearisation: the two halves of CKKS multiplication (SURVEY 8f N2) -------------------------------------
// poulpy-core/src/operations/glwe.rs:699-818 (glwe_tensor_apply), :545-610 (glwe_tensor_relinearize);
// poulpy-ckks/src/leveled/default/mul.rs:49-86 (ckks_mul_into = tensor_apply + relinearize).
static int64_t msb_mask_bottom_limb(uint64_t base2k, uint64_t k) { // operations/glwe.rs:921-926
    const uint64_t r = k % base2k;
    return r == 0 ? ~(int64_t)0 : (int64_t)(~(uint64_t)0 << (base2k - r));
}
static uint64_t normalize_input_limb_bound_with_offset(uint64_t full, uint64_t res_size, uint64_t res_base2k, uint64_t in_base2k, int64_t off) {
    int64_t ob = off % (int64_t)in_base2k; // operations/glwe.rs:928-957
    if (off < 0 && ob != 0) ob += (int64_t)in_base2k;
    return umin64(full, div_ceil64(res_size * res_base2k + (uint64_t)ob, in_base2k));
}
struct TensorPlan {
    uint64_t off_hi, dft_size;
    int64_t off_lo;
};
static TensorPlan tensor_plan(uint64_t cnv_offset, uint64_t ab_base2k, uint64_t a_size, uint64_t b_size, uint64_t res_size, uint64_t res_base2k) {
    TensorPlan t;
    if (cnv_offset < ab_base2k) { // operations/glwe.rs:753-757
        t.off_hi = 0;
        t.off_lo = -(int64_t)(ab_base2k - (cnv_offset % ab_base2k));
    } else {
        t.off_hi = cnv_offset / ab_base2k - 1;
        t.off_lo = (int64_t)(cnv_offset % ab_base2k);
    }
    t.dft_size = normalize_input_limb_bound_with_offset(a_size + b_size - t.off_hi, res_size, res_base2k, ab_base2k, t.off_lo);
    return t;
}
extern "C" size_t pgb_glwe_tensor_apply_tmp_bytes(const pgb_module *m, uint64_t rank, uint64_t res_size, uint64_t res_base2k, uint64_t a_size,
                                                  uint64_t b_size, uint64_t ab_base2k, uint64_t cnv_offset, uint64_t batch) {
    const uint64_t n = m->n, pb = prep_bytes(m), cols = rank + 1;
    const TensorPlan t = tensor_plan(cnv_offset, ab_base2k, a_size, b_size, res_size, res_base2k);
    return align_up(batch * n * cols * a_size * pb) + align_up(batch * n * cols * b_size * pb) + align_up(batch * n * t.dft_size * pb) +
           align_up(batch * n * res_size * 8) + ALIGN;
}
// res: `count` GLWETensor VecZnx with (rank+1)(rank+2)/2 columns (stride bt->stride_res); a / b: GLWE VecZnx (strides stride_a / stride_b)
extern "C" int pgb_glwe_tensor_apply_batched(pgb_module *m, uint64_t cnv_offset, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a,
                                             uint64_t a_effective_k, const pgb_vec_znx *b, uint64_t b_effective_k, uint64_t ab_base2k,
                                             const pgb_batch *bt, void *scratch, size_t scratch_len) {
    PGB_REQUIRE(bt && bt->count >= 1 && bt->count <= 65535, "glwe_tensor_apply: batch count must be in [1, 65535]");
    PGB_REQUIRE(res->n == m->n && a->n == m->n && b->n == m->n, "glwe_tensor_apply: ring degree mismatch");
    const uint64_t n = m->n, pb = prep_bytes(m), B = bt->count, cols = a->cols;
    PGB_REQUIRE(b->cols == cols && res->cols == cols * (cols + 1) / 2, "glwe_tensor_apply: res must have (rank+1)(rank+2)/2 columns");
    PGB_REQUIRE(div_ceil64(a_effective_k, ab_base2k) == a->size && div_ceil64(b_effective_k, ab_base2k) == b->size,
                "glwe_tensor_apply: effective_k does not match the operand sizes"); // operations/glwe.rs:727-728
    const size_t need = pgb_glwe_tensor_apply_tmp_bytes(m, cols - 1, res->size, res_base2k, a->size, b->size, ab_base2k, cnv_offset, B);
    if (scratch_len < need) {
        pgb_set_error("glwe_tensor_apply: scratch of %zu bytes < required %zu", scratch_len, need);
        return PGB_ERR_SCRATCH;
    }
    const TensorPlan t = tensor_plan(cnv_offset, ab_base2k, a->size, b->size, res->size, res_base2k);
    Arena ar = {(char *)scratch, scratch_len, 0};
    const uint64_t ap_bs = n * cols * a->size * pb, bp_bs = n * cols * b->size * pb, rd_bs = n * t.dft_size * pb, tmp_bs = n * res->size * 8;
    pgb_vec_znx_dft a_prep = mk(ar.take(B * ap_bs), n, cols, a->size), b_prep = mk(ar.take(B * bp_bs), n, cols, b->size);
    pgb_vec_znx_dft res_dft = mk(ar.take(B * rd_bs), n, 1, t.dft_size);
    pgb_vec_znx tmp = mk(ar.take(B * tmp_bs), n, 1, res->size);
    pgb_batch bta = {B, ap_bs, bt->stride_a, 0}, btb = {B, bp_bs, bt->stride_b, 0};
    PGB_TRY(cnv_prepare_impl(m, &a_prep, a, msb_mask_bottom_limb(ab_base2k, a_effective_k), &bta)); // :736-740
    PGB_TRY(cnv_prepare_impl(m, &b_prep, b, msb_mask_bottom_limb(ab_base2k, b_effective_k), &btb));
    const uint64_t res_ls = res->cols * n * 8;
    auto tensor_col = [&](uint64_t c) { LimbSet s = {(char *)res->data + c * n * 8, res_ls, bt->stride_res}; return s; };
    const LimbSet T = {(char *)tmp.data, n * 8, tmp_bs};
    auto product = [&](uint64_t i, uint64_t j) -> int { // tmp <- normalize(idft(cnv(a_prep, b_prep; i, j)))
        pgb_batch btc = {B, rd_bs, ap_bs, bp_bs};
        PGB_TRY(pgb_cnv_pairwise_apply_dft_batched(m, t.off_hi, &res_dft, 0, &a_prep, &b_prep, i, j, &btc));
        pgb_batch bti = {B, rd_bs, 0, 0};
        PGB_TRY(pgb_vec_znx_idft_apply_consume_batched(m, &res_dft, &bti));
        pgb_batch btn = {B, tmp_bs, rd_bs, 0};
        return big_normalize_impl(m, &tmp, res_base2k, t.off_lo, 0, &res_dft, ab_base2k, 0, 0, true, &btn);
    };
    const uint32_t rs = (uint32_t)res->size;
    for (uint64_t i = 0; i < cols; i++) { // :773-797
        const uint64_t col_i = i * cols - (i * (i + 1) / 2);
        PGB_TRY(product(i, i));
        PGB_TRY(znx_ew(m, 3, tensor_col(col_i + i), T, 0, nullptr, 0, rs, (uint32_t)B)); // vec_znx_copy
        for (uint64_t j = 0; j < cols; j++) {
            if (j == i) continue;
            if (j < i) {
                const uint64_t col_j = j * cols - (j * (j + 1) / 2);
                PGB_TRY(znx_ew(m, 1, tensor_col(col_j + i), T, 0, nullptr, 0, rs, (uint32_t)B)); // vec_znx_sub_assign
            } else {
                PGB_TRY(znx_ew(m, 4, tensor_col(col_i + j), T, 0, nullptr, 0, rs, (uint32_t)B)); // vec_znx_negate
            }
        }
    }
    for (uint64_t i = 0; i < cols; i++) { // :799-816
        const uint64_t col_i = i * cols - (i * (i + 1) / 2);
        for (uint64_t j = i + 1; j < cols; j++) {
            PGB_TRY(product(i, j));
            PGB_TRY(znx_ew(m, 0, tensor_col(col_i + j), T, 0, nullptr, 0, rs, (uint32_t)B)); // vec_znx_add_assign
        }
    }
    return PGB_OK;
}

extern "C" size_t pgb_glwe_tensor_relinearize_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t a_base2k,
                                                        const pgb_vmp_pmat *tsk, uint64_t key_base2k, uint64_t dsize, uint64_t batch) {
    (void)res_size;
    const uint64_t n = m->n, pb = prep_bytes(m), cols = tsk->cols_out, pairs = tsk->cols_in;
    const uint64_t a_dft_size = div_ceil64(a_size * a_base2k, key_base2k);
    uint64_t t = align_up(batch * n * pairs * a_dft_size * pb) + align_up(batch * n * a_dft_size * 8) + align_up(batch * n * cols * tsk->size * pb);
    if (dsize > 1) t += align_up(batch * n * pairs * div_ceil64(a_dft_size, dsize) * pb) + align_up(batch * n * cols * tsk->size * pb);
    return t + ALIGN;
}
// a: `count` GLWETensor VecZnx (cols + pairs columns, stride bt->stride_a); tsk: prepared tensor key VmpPMat(dnum, pairs, cols, size)
extern "C" int pgb_glwe_tensor_relinearize_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a, uint64_t a_base2k,
                                                   const pgb_vmp_pmat *tsk, uint64_t key_base2k, uint64_t dsize, const pgb_batch *bt,
                                                   void *scratch, size_t scratch_len) {
    PGB_REQUIRE(bt && bt->count >= 1 && bt->count <= 65535, "glwe_tensor_relinearize: batch count must be in [1, 65535]");
    PGB_REQUIRE(res->n == m->n && a->n == m->n && tsk->n == m->n, "glwe_tensor_relinearize: ring degree mismatch");
    const uint64_t n = m->n, pb = prep_bytes(m), B = bt->count, cols = tsk->cols_out, pairs = tsk->cols_in;
    PGB_REQUIRE(res->cols == cols && a->cols == cols + pairs, "glwe_tensor_relinearize: rank mismatch"); // :571-572
    PGB_REQUIRE(dsize >= 1, "glwe_tensor_relinearize: dsize must be >= 1");
    const size_t need = pgb_glwe_tensor_relinearize_tmp_bytes(m, res->size, a->size, a_base2k, tsk, key_base2k, dsize, B);
    if (scratch_len < need) {
        pgb_set_error("glwe_tensor_relinearize: scratch of %zu bytes < required %zu", scratch_len, need);
        return PGB_ERR_SCRATCH;
    }
    Arena ar = {(char *)scratch, scratch_len, 0};
    const uint64_t a_dft_size = div_ceil64(a->size * a_base2k, key_base2k);
    const uint64_t a_dft_bs = n * pairs * a_dft_size * pb, conv_bs = n * a_dft_size * 8, res_dft_bs = n * cols * tsk->size * pb;
    pgb_vec_znx_dft a_dft = mk(ar.take(B * a_dft_bs), n, pairs, a_dft_size);
    pgb_vec_znx a_conv = mk(ar.take(B * conv_bs), n, 1, a_dft_size);
    pgb_vec_znx_dft res_dft = mk(ar.take(B * res_dft_bs), n, cols, tsk->size);
    for (uint64_t i = 0; i < pairs; i++) { // :579-589
        pgb_batch btd = {B, a_dft_bs, bt->stride_a, 0};
        if (a_base2k != key_base2k) {
            pgb_batch btn = {B, conv_bs, bt->stride_a, 0};
            PGB_TRY(big_normalize_impl(m, &a_conv, key_base2k, 0, 0, a, a_base2k, cols + i, 0, false, &btn));
            btd.stride_a = conv_bs;
            PGB_TRY(pgb_vec_znx_dft_apply_batched(m, 1, 0, &a_dft, i, &a_conv, 0, &btd));
        } else {
            PGB_TRY(pgb_vec_znx_dft_apply_batched(m, 1, 0, &a_dft, i, a, cols + i, &btd));
        }
    }
    PGB_TRY(keyswitch_core(m, ar, "glwe_tensor_relinearize", &res_dft, res_dft_bs, &a_dft, a_dft_bs, tsk, dsize, B)); // :593
    pgb_vec_znx_big res_big = res_dft;
    for (uint64_t i = 0; i < cols; i++) { // :596-606 (sic: the reference tests res_base2k == key_base2k)
        if (res_base2k == key_base2k) {
            pgb_batch bts = {B, res_dft_bs, bt->stride_a, 0};
            PGB_TRY(big_add_small_impl(m, &res_big, i, a, i, &bts));
        } else {
            pgb_batch btn = {B, conv_bs, bt->stride_a, 0};
            PGB_TRY(big_normalize_impl(m, &a_conv, key_base2k, 0, 0, a, a_base2k, i, 0, false, &btn));
            pgb_batch bts = {B, res_dft_bs, conv_bs, 0};
            PGB_TRY(big_add_small_impl(m, &res_big, i, &a_conv, 0, &bts));
        }
    }
    pgb_batch btn = {B, bt->stride_res, res_dft_bs, 0};
    for (uint64_t i = 0; i < res->cols; i++) PGB_TRY(big_normalize_impl(m, res, res_base2k, 0, i, &res_big, key_base2k, i, 0, true, &btn));
    return PGB_OK;
}

// The automorphism family on the single-kernel route (gadget_fused with the kernels' automorphism epilogue): key-switch, X -> X^p and the
// addition / subtraction of the input in one launch per batch.  aut_mode 1..3 = op 0..2 of pgb_glwe_automorphism_op_batched, 4 = plain
// glwe_automorphism.  Returns as gadget_fused; `ar` supplies the flag list and, when res overlaps a, the staging buffer of the outputs.
static int automorphism_fused(pgb_module *m, int aut_mode, pgb_vec_znx *res, uint64_t res_bs, const pgb_vec_znx *a, uint64_t a_bs,
                              const pgb_vmp_pmat *key, uint64_t base2k, int64_t p, uint64_t dsize, uint64_t B, Arena &ar) {
    const int small = (int)umin64(a->size, key->size);
    const GadgetJob job = {a, a_bs, 1, key, dsize, base2k, small, (int)key->rows, aut_mode, p, aut_mode == 4 ? 0 : small, res, res_bs,
                           vec_znx_alias_class(res, res_bs, a, a_bs, B), B};
    return gadget_fused(m, job, ar, nullptr, 0, nullptr, 0);
}

// ---- glwe_automorphism (poulpy-core/src/automorphism/glwe_ct.rs:51-72; SURVEY 8f N4): key-switch with the automorphism key, then
// X -> X^p on every column.  The key-switch lands in scratch so that the permutation is out of place.
extern "C" size_t pgb_glwe_automorphism_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t a_base2k,
                                                  const pgb_vmp_pmat *key, uint64_t key_base2k, uint64_t dsize, uint64_t batch) {
    return align_up(batch * m->n * key->cols_out * res_size * 8) + pgb_glwe_keyswitch_tmp_bytes(m, res_size, a_size, a_base2k, key, key_base2k, dsize, batch) +
           align_up((2 * batch + 1) * sizeof(int)) + ALIGN;
}
extern "C" int pgb_glwe_automorphism_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a, uint64_t a_base2k,
                                             const pgb_vmp_pmat *key, uint64_t key_base2k, int64_t p, uint64_t dsize, const pgb_batch *bt,
                                             void *scratch, size_t scratch_len) {
    PGB_REQUIRE(bt && bt->count >= 1 && bt->count <= 65535, "glwe_automorphism: batch count must be in [1, 65535]");
    PGB_REQUIRE(res->n == m->n && res->cols == key->cols_out, "glwe_automorphism: res does not match the key");
    const size_t need = pgb_glwe_automorphism_tmp_bytes(m, res->size, a->size, a_base2k, key, key_base2k, dsize, bt->count);
    if (scratch_len < need) {
        pgb_set_error("glwe_automorphism: scratch of %zu bytes < required %zu", scratch_len, need);
        return PGB_ERR_SCRATCH;
    }
    const uint64_t n = m->n, B = bt->count, tmp_bs = n * res->cols * res->size * 8;
    Arena ar = {(char *)scratch, scratch_len, 0};
    if (res_base2k == key_base2k && a_base2k == key_base2k && a->cols == key->cols_in + 1) {
        const int done = automorphism_fused(m, 4, res, bt->stride_res, a, bt->stride_a, key, key_base2k, p, dsize, B, ar);
        if (done < 0) return done;
        if (done) return PGB_OK;
    }
    pgb_vec_znx tmp = mk(ar.take(B * tmp_bs), n, res->cols, res->size);
    pgb_batch btk = {B, tmp_bs, bt->stride_a, 0};
    PGB_TRY(pgb_glwe_keyswitch_batched(m, &tmp, res_base2k, a, a_base2k, key, key_base2k, dsize, &btk, ar.rest(), ar.rest_len()));
    pgb_batch bta = {B, bt->stride_res, tmp_bs, 0};
    for (uint64_t i = 0; i < res->cols; i++) PGB_TRY(pgb_vec_znx_automorphism_batched(m, p, res, i, &tmp, i, &bta));
    return PGB_OK;
}

// ---- glwe_automorphism_add_assign (poulpy-core/src/automorphism/glwe_ct.rs:142-183) and glwe_trace_assign
// (poulpy-core/src/glwe_trace.rs:129-175; SURVEY 8f N4), batched and device resident.  The limb-wise HAL sequence of the reference:
//   res_big = glwe_keyswitch_internal(res_dft, res, key); per column: big_automorphism(p), big_add_small_assign(res column),
//   big_normalize back into res.  The permutation is out of place into a second big buffer instead of through an n-element tmp.
extern "C" size_t pgb_glwe_automorphism_add_assign_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t res_base2k, const pgb_vmp_pmat *key,
                                                             uint64_t key_base2k, uint64_t dsize, uint64_t batch) {
    const uint64_t n = m->n, pb = prep_bytes(m), bb = big_bytes(m);
    const uint64_t rank_in = key->cols_in, cols = key->cols_out;
    const uint64_t in_size = res_base2k == key_base2k ? res_size : conv_size(res_size, res_base2k, key_base2k);
    uint64_t t = 0;
    t += align_up(batch * n * cols * key->size * pb);                                   // res_dft / res_big
    t += align_up(batch * n * cols * key->size * bb);                                   // permuted big
    t += align_up(batch * n * rank_in * in_size * pb);                                  // a_dft
    if (res_base2k != key_base2k) t += align_up(batch * n * cols * in_size * 8);        // res_conv
    if (dsize > 1) t += align_up(batch * n * rank_in * div_ceil64(in_size, dsize) * pb) + align_up(batch * n * cols * key->size * pb);
    const uint64_t fused = align_up((2 * batch + 1) * sizeof(int)) + align_up(batch * n * cols * res_size * 8); // flags + in-place staging
    return (t > fused ? t : fused) + ALIGN;
}
// glwe_automorphism_add / _sub / _sub_negate (automorphism/glwe_ct.rs:95-275): res = normalize(aut_p(ks(a)) (+|-) a) resp. normalize(a -
// aut_p(ks(a))), out of place (res == a gives the _assign forms); op = 0 add, 1 sub, 2 sub_negate.  a and res share a_base2k / sizes here
// (what the trace and the packing use); bt->stride_a is the stride of a.
extern "C" int pgb_glwe_automorphism_op_batched(pgb_module *m, int op, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a,
                                                const pgb_vmp_pmat *key, uint64_t key_base2k, int64_t p, uint64_t dsize, const pgb_batch *bt,
                                                void *scratch, size_t scratch_len);
extern "C" int pgb_glwe_automorphism_add_assign_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vmp_pmat *key,
                                                        uint64_t key_base2k, int64_t p, uint64_t dsize, const pgb_batch *bt, void *scratch,
                                                        size_t scratch_len) {
    pgb_batch b2 = {bt->count, bt->stride_res, bt->stride_res, 0};
    return pgb_glwe_automorphism_op_batched(m, 0, res, res_base2k, res, key, key_base2k, p, dsize, &b2, scratch, scratch_len);
}
extern "C" int pgb_glwe_automorphism_op_batched(pgb_module *m, int op, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a,
                                                const pgb_vmp_pmat *key, uint64_t key_base2k, int64_t p, uint64_t dsize, const pgb_batch *bt,
                                                void *scratch, size_t scratch_len) {
    PGB_REQUIRE(bt && bt->count >= 1 && bt->count <= 65535, "glwe_automorphism_op: batch count must be in [1, 65535]");
    PGB_REQUIRE(op >= 0 && op <= 2, "glwe_automorphism_op: op must be 0 (add), 1 (sub) or 2 (sub_negate)");
    PGB_REQUIRE(res->n == m->n && key->n == m->n && a->n == m->n, "glwe_automorphism_op: ring degree mismatch");
    PGB_REQUIRE(res->cols == key->cols_in + 1 && res->cols == key->cols_out && a->cols == res->cols, "glwe_automorphism_op: rank mismatch");
    PGB_REQUIRE(a->size == res->size, "glwe_automorphism_op: a and res must have the same size");
    PGB_REQUIRE(dsize >= 1, "glwe_automorphism_op: dsize must be >= 1");
    const size_t need = pgb_glwe_automorphism_add_assign_tmp_bytes(m, res->size, res_base2k, key, key_base2k, dsize, bt->count);
    if (scratch_len < need) {
        pgb_set_error("glwe_automorphism_op: scratch of %zu bytes < required %zu", scratch_len, need);
        return PGB_ERR_SCRATCH;
    }
    const uint64_t n = m->n, pb = prep_bytes(m), bb = big_bytes(m), B = bt->count, rank_in = key->cols_in, cols = key->cols_out;
    Arena ar = {(char *)scratch, scratch_len, 0};
    if (res_base2k == key_base2k) {
        const int done = automorphism_fused(m, op + 1, res, bt->stride_res, a, bt->stride_a, key, key_base2k, p, dsize, B, ar);
        if (done < 0) return done;
        if (done) return PGB_OK;
    }
    const uint64_t res_dft_bs = n * cols * key->size * pb, big2_bs = n * cols * key->size * bb;
    pgb_vec_znx_dft res_dft = mk(ar.take(B * res_dft_bs), n, cols, key->size);
    pgb_vec_znx_big big2 = mk(ar.take(B * big2_bs), n, cols, key->size);
    pgb_vec_znx ain; // (:161-168) res_conv = glwe_normalize(res) at the key's base2k
    uint64_t ain_bs;
    PGB_TRY(glwe_to_base2k(m, ar, a, bt->stride_a, res_base2k, key_base2k, B, &ain, &ain_bs));
    // glwe_keyswitch_internal (keyswitching/glwe.rs:207-239)
    const uint64_t a_dft_bs = n * rank_in * ain.size * pb;
    pgb_vec_znx_dft a_dft = mk(ar.take(B * a_dft_bs), n, rank_in, ain.size);
    pgb_batch btd = {B, a_dft_bs, ain_bs, 0};
    for (uint64_t c = 0; c < rank_in; c++) PGB_TRY(pgb_vec_znx_dft_apply_batched(m, 1, 0, &a_dft, c, &ain, c + 1, &btd));
    PGB_TRY(keyswitch_core(m, ar, "glwe_automorphism_op", &res_dft, res_dft_bs, &a_dft, a_dft_bs, key, dsize, B));
    pgb_vec_znx_big res_big = res_dft;
    pgb_batch bts = {B, res_dft_bs, ain_bs, 0};
    PGB_TRY(big_add_small_impl(m, &res_big, 0, &ain, 0, &bts));
    for (uint64_t i = 0; i < res->cols; i++) { // (:170-181)
        pgb_batch bta = {B, big2_bs, res_dft_bs, 0};
        PGB_TRY(big_automorphism_impl(m, p, &big2, i, &res_big, i, &bta));
        pgb_batch bt2 = {B, big2_bs, ain_bs, 0};
        PGB_TRY(big_small_op_impl(m, op == 0 ? BIG_ADD_SMALL : (op == 1 ? BIG_SUB_SMALL : BIG_SUB_SMALL_NEG), &big2, i, &ain, i, &bt2));
        pgb_batch btn = {B, bt->stride_res, big2_bs, 0};
        PGB_TRY(big_normalize_impl(m, res, res_base2k, 0, i, &big2, key_base2k, i, 0, true, &btn));
    }
    return PGB_OK;
}

// trace_galois_elements (glwe_trace.rs:34-44): -1 for i = 0, GALOISGENERATOR^(2^(i-1)) mod 2n otherwise (layouts/module.rs:214-226)
extern "C" int64_t pgb_trace_galois_element(const pgb_module *m, uint64_t i) {
    if (i == 0) return -1;
    uint64_t r = 1, x = 5, e = (uint64_t)1 << (i - 1);
    while (e) {
        if (e & 1) r *= x;
        x *= x;
        e >>= 1;
    }
    return (int64_t)(r & (2 * m->n - 1));
}
extern "C" size_t pgb_glwe_trace_assign_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t res_base2k, const pgb_vmp_pmat *key,
                                                  uint64_t key_base2k, uint64_t dsize, uint64_t batch) {
    const uint64_t in_size = res_base2k == key_base2k ? res_size : conv_size(res_size, res_base2k, key_base2k);
    size_t t = pgb_glwe_automorphism_add_assign_tmp_bytes(m, in_size, key_base2k, key, key_base2k, dsize, batch);
    if (res_base2k != key_base2k) t += align_up(batch * m->n * key->cols_out * in_size * 8);
    t += align_up(batch * m->n * key->cols_out * in_size * 8); // second GLWE buffer: the rounds alternate between two buffers
    return t + ALIGN;
}
// keys: host array of log_n prepared automorphism keys (same shape), keys[i] for pgb_trace_galois_element(i); entries below `skip` unread
extern "C" int pgb_glwe_trace_assign_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, uint64_t skip, const pgb_vmp_pmat *keys,
                                             uint64_t nkeys, uint64_t key_base2k, uint64_t dsize, const pgb_batch *bt, void *scratch,
                                             size_t scratch_len) {
    PGB_REQUIRE(bt && bt->count >= 1 && bt->count <= 65535, "glwe_trace: batch count must be in [1, 65535]");
    PGB_REQUIRE(res->n == m->n, "glwe_trace: ring degree mismatch");
    PGB_REQUIRE(skip <= (uint64_t)m->log_n, "glwe_trace: skip > log_n");                      // glwe_trace.rs:144
    PGB_REQUIRE(nkeys >= (uint64_t)m->log_n, "glwe_trace: needs log_n automorphism keys");
    if (skip == (uint64_t)m->log_n) return PGB_OK;
    const pgb_vmp_pmat *k0 = &keys[skip];
    const size_t need = pgb_glwe_trace_assign_tmp_bytes(m, res->size, res_base2k, k0, key_base2k, dsize, bt->count);
    if (scratch_len < need) {
        pgb_set_error("glwe_trace: scratch of %zu bytes < required %zu", scratch_len, need);
        return PGB_ERR_SCRATCH;
    }
    const uint64_t n = m->n, B = bt->count;
    Arena ar = {(char *)scratch, scratch_len, 0};
    pgb_vec_znx cur; // (:156-165) work on a copy at the key's base2k
    uint64_t cur_bs;
    PGB_TRY(glwe_to_base2k(m, ar, res, bt->stride_res, res_base2k, key_base2k, B, &cur, &cur_bs));
    // The rounds run out of place, alternating between `cur` and a second buffer (glwe_automorphism_add_assign is res = aut(ks(res)) +
    // res; the single-kernel route cannot run in place), and the result is copied back if it ends in the second one.
    const uint64_t alt_bs = n * cur.cols * cur.size * 8;
    pgb_vec_znx alt = mk(ar.take(B * alt_bs), n, cur.cols, cur.size);
    char *sc = ar.rest();
    const size_t sc_len = ar.rest_len();
    pgb_vec_znx home = cur;
    const uint64_t home_bs = cur_bs;
    uint64_t alt_stride = alt_bs;
    for (uint64_t i = skip; i < (uint64_t)m->log_n; i++) { // (:166-177)
        pgb_batch btc = {B, cur_bs, 0, 0};
        { // glwe_rsh(1) on every column: the columns of a limb are adjacent, so one launch shifts cols * n words per limb
            PGB_REQUIRE(key_base2k >= 1 && key_base2k <= 63 && cur.size >= 1, "glwe_trace: base2k must be in [1, 63]");
            LimbSet RS = {(char *)cur.data, cur.cols * n * 8, btc.stride_res};
            PGB_TRY(znx_rsh_assign(m, RS, (int)cur.size, (int)key_base2k, 1, (uint32_t)B, (uint32_t)(cur.cols * n)));
        }
        pgb_batch bto = {B, alt_stride, cur_bs, 0};
        PGB_TRY(pgb_glwe_automorphism_op_batched(m, 0, &alt, key_base2k, &cur, &keys[i], key_base2k, pgb_trace_galois_element(m, i), dsize, &bto,
                                                 sc, sc_len));
        pgb_vec_znx tv = cur;
        cur = alt;
        alt = tv;
        const uint64_t ts = cur_bs;
        cur_bs = alt_stride;
        alt_stride = ts;
    }
    if (cur.data != home.data) {
        PGB_CHECK_CUDA(cudaMemcpy2DAsync(home.data, home_bs, cur.data, cur_bs, alt_bs, B, cudaMemcpyDeviceToDevice, m->stream));
        cur = home;
        cur_bs = home_bs;
    }
    if (res_base2k != key_base2k) {
        pgb_batch btn = {B, bt->stride_res, cur_bs, 0};
        for (uint64_t i = 0; i < res->cols; i++) PGB_TRY(big_normalize_impl(m, res, res_base2k, 0, i, &cur, key_base2k, i, 0, false, &btn));
    }
    return PGB_OK;
}

// ---- ggsw_expand_row (poulpy-core/src/conversion/gglwe_to_ggsw.rs:116-268; SURVEY 8f N4): the GLWEs of columns 1..rank of a GGSW from
// its column-0 GLWEs and the tensor keys GGLWE(s[c] * s) -- the last step of circuit bootstrapping.  Per row: the mask of the column-0
// GLWE goes to the DFT domain once, then every column is a gadget product with tsk[col-1], the column-0 body added on output column `col`
// (vec_znx_big_add_small_assign) and the normalisation of all output columns.
extern "C" size_t pgb_ggsw_expand_row_tmp_bytes(const pgb_module *m, uint64_t rank, uint64_t size, uint64_t res_base2k, const pgb_vmp_pmat *tsk,
                                                uint64_t tsk_base2k, uint64_t dsize, uint64_t batch) {
    const uint64_t n = m->n, pb = prep_bytes(m), cols = rank + 1;
    const uint64_t conv = res_base2k == tsk_base2k ? size : conv_size(size, res_base2k, tsk_base2k);
    uint64_t t = align_up(batch * n * rank * conv * pb) + align_up(batch * n * conv * 8) + align_up(batch * n * cols * tsk->size * pb);
    if (dsize > 1) t += align_up(batch * n * rank * div_ceil64(conv, dsize) * pb) + align_up(batch * n * cols * tsk->size * pb);
    return t + ALIGN;
}
// ggsw: `count` MatZnx(dnum, rank+1, rank+1, size) (stride bt->stride_res bytes) with the column-0 GLWEs filled; tsk: HOST array of `rank`
// prepared keys VmpPMat(dnum_tsk, rank, rank+1, size_tsk)
extern "C" int pgb_ggsw_expand_row_batched(pgb_module *m, pgb_mat_znx *ggsw, uint64_t res_base2k, const pgb_vmp_pmat *tsk, uint64_t ntsk,
                                           uint64_t tsk_base2k, uint64_t dsize, const pgb_batch *bt, void *scratch, size_t scratch_len) {
    PGB_REQUIRE(bt && bt->count >= 1 && bt->count <= 65535, "ggsw_expand_row: batch count must be in [1, 65535]");
    PGB_REQUIRE(ggsw->n == m->n && ggsw->cols_in == ggsw->cols_out && ggsw->cols_in >= 1, "ggsw_expand_row: not a GGSW of this ring");
    const uint64_t n = m->n, pb = prep_bytes(m), B = bt->count, cols = ggsw->cols_in, rank = cols - 1, size = ggsw->size, dnum = ggsw->rows;
    if (rank == 0) return PGB_OK;
    PGB_REQUIRE(ntsk >= rank, "ggsw_expand_row: needs one tensor key per mask column");
    for (uint64_t c = 0; c < rank; c++)
        PGB_REQUIRE(tsk[c].n == n && tsk[c].cols_in == rank && tsk[c].cols_out == cols && tsk[c].size == tsk[0].size && tsk[c].rows == tsk[0].rows,
                    "ggsw_expand_row: tensor key %llu has the wrong shape", (unsigned long long)c);
    PGB_REQUIRE(dsize >= 1, "ggsw_expand_row: dsize must be >= 1");
    const size_t need = pgb_ggsw_expand_row_tmp_bytes(m, rank, size, res_base2k, &tsk[0], tsk_base2k, dsize, B);
    if (scratch_len < need) {
        pgb_set_error("ggsw_expand_row: scratch of %zu bytes < required %zu", scratch_len, need);
        return PGB_ERR_SCRATCH;
    }
    Arena ar = {(char *)scratch, scratch_len, 0};
    const uint64_t conv = res_base2k == tsk_base2k ? size : conv_size(size, res_base2k, tsk_base2k);
    const uint64_t a_dft_bs = n * rank * conv * pb, a0_bs = n * conv * 8, res_dft_bs = n * cols * tsk[0].size * pb, glwe_bytes = n * cols * size * 8;
    pgb_vec_znx_dft a_dft = mk(ar.take(B * a_dft_bs), n, rank, conv);
    pgb_vec_znx a_0 = mk(ar.take(B * a0_bs), n, 1, conv);
    pgb_vec_znx_dft res_dft = mk(ar.take(B * res_dft_bs), n, cols, tsk[0].size);
    for (uint64_t row = 0; row < dnum; row++) {
        pgb_vec_znx mi = mk((char *)ggsw->data + (row * cols + 0) * glwe_bytes, n, cols, size); // res.at(row, 0)
        const pgb_vec_znx *small = &mi; // column 0 of the row's GLWE joins output column `col`
        uint64_t small_bs = bt->stride_res;
        if (res_base2k == tsk_base2k) { // (:145-149)
            pgb_batch btd = {B, a_dft_bs, bt->stride_res, 0};
            for (uint64_t c = 0; c < rank; c++) PGB_TRY(pgb_vec_znx_dft_apply_batched(m, 1, 0, &a_dft, c, &mi, c + 1, &btd));
        } else { // (:150-156)
            pgb_batch btn = {B, a0_bs, bt->stride_res, 0}, btd = {B, a_dft_bs, a0_bs, 0};
            for (uint64_t c = 0; c < rank; c++) {
                PGB_TRY(big_normalize_impl(m, &a_0, tsk_base2k, 0, 0, &mi, res_base2k, c + 1, 0, false, &btn));
                PGB_TRY(pgb_vec_znx_dft_apply_batched(m, 1, 0, &a_dft, c, &a_0, 0, &btd));
            }
            PGB_TRY(big_normalize_impl(m, &a_0, tsk_base2k, 0, 0, &mi, res_base2k, 0, 0, false, &btn));
            small = &a_0;
            small_bs = a0_bs;
        }
        for (uint64_t col = 1; col < cols; col++) { // ggsw_expand_rows_internal (:182-268)
            PGB_TRY(keyswitch_core(m, ar, "ggsw_expand_row", &res_dft, res_dft_bs, &a_dft, a_dft_bs, &tsk[col - 1], dsize, B));
            pgb_vec_znx_big res_big = res_dft;
            pgb_batch bts = {B, res_dft_bs, small_bs, 0};
            PGB_TRY(big_add_small_impl(m, &res_big, col, small, 0, &bts));
            pgb_vec_znx out = mk((char *)ggsw->data + (row * cols + col) * glwe_bytes, n, cols, size); // res.at(row, col)
            pgb_batch btn = {B, bt->stride_res, res_dft_bs, 0};
            for (uint64_t j = 0; j < cols; j++) PGB_TRY(big_normalize_impl(m, &out, res_base2k, 0, j, &res_big, tsk_base2k, j, 0, true, &btn));
        }
    }
    return PGB_OK;
}

// ---- host-buffer front ends ---------------------------------------------------------------------------------------------------
// Chunked three-stage pipeline (H2D on aux stream 0, compute on the module stream, D2H on aux stream 1), double buffered.
int ensure_ws(pgb_module *m, size_t len) {
    PGB_CHECK_CUDA(cudaSetDevice(m->device));
    if (m->ws_len >= len) return PGB_OK;
    if (m->ws) cudaFree(m->ws);
    m->ws = nullptr;
    m->ws_len = 0;
    PGB_CHECK_CUDA(cudaMalloc(&m->ws, len));
    m->ws_len = len;
    return PGB_OK;
}
static int ensure_pinned(pgb_module *m, size_t len) {
    if (m->pinned_len >= len) return PGB_OK;
    for (int i = 0; i < 4; i++) {
        if (m->pinned[i]) cudaFreeHost(m->pinned[i]);
        m->pinned[i] = nullptr;
    }
    m->pinned_len = 0;
    for (int i = 0; i < 4; i++) PGB_CHECK_CUDA(cudaHostAlloc(&m->pinned[i], len, cudaHostAllocDefault));
    m->pinned_len = len;
    return PGB_OK;
}

typedef int (*core_fn)(pgb_module *, pgb_vec_znx *, uint64_t, const pgb_vec_znx *, uint64_t, const pgb_vmp_pmat *, uint64_t, uint64_t,
                       const pgb_batch *, void *, size_t);

bool is_pinned(const void *p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost;
}

// Chunk c uses slot s = c & 1 of the double-buffered device (and, for pageable callers, pinned) buffers.
//   s_in : H2D(c)            waits compute(c-2) (d_in[s] free)
//   s_c  : compute(c)        waits H2D(c) and D2H(c-2) (d_out[s] free)
//   s_out: D2H(c)            waits compute(c)
static int host_pipeline(pgb_module *m, bool ext, int64_t *res_host, uint64_t res_cols, uint64_t res_size, uint64_t res_base2k,
                         const int64_t *a_host, uint64_t a_cols, uint64_t a_size, uint64_t a_base2k, const pgb_vmp_pmat *key,
                         uint64_t key_base2k, uint64_t dsize, uint64_t count) {
    if (count == 0) return PGB_OK;
    const uint64_t n = m->n;
    const uint64_t a_bytes = n * a_cols * a_size * 8, r_bytes = n * res_cols * res_size * 8;
    // small chunks keep the three stages overlapped and the fill / drain of the pipeline short; 32 MB of staging per slot measured best
    // (scripts/e2e_probe.py: 229 k key-switches/s against a 250 k ceiling of this box's pinned H2D rate, 49 GB/s)
    const uint64_t stage_bytes = (uint64_t)(m->opt[PGB_OPT_HOST_CHUNK_MB] > 0 ? m->opt[PGB_OPT_HOST_CHUNK_MB] : 32) << 20;
    const uint64_t chunk = umin64(count, umin64(2048, (a_bytes > r_bytes ? stage_bytes / a_bytes : stage_bytes / r_bytes) + 1));
    const size_t tmp = ext ? pgb_glwe_external_product_tmp_bytes(m, res_size, a_size, a_base2k, key, key_base2k, dsize, chunk)
                           : pgb_glwe_keyswitch_tmp_bytes(m, res_size, a_size, a_base2k, key, key_base2k, dsize, chunk);
    const size_t in_dev = align_up(chunk * a_bytes), out_dev = align_up(chunk * r_bytes);
    PGB_TRY(ensure_ws(m, 2 * (in_dev + out_dev) + align_up(tmp) + ALIGN));
    const bool direct = is_pinned(a_host) && is_pinned(res_host);
    if (!direct) PGB_TRY(ensure_pinned(m, (size_t)(chunk * (a_bytes > r_bytes ? a_bytes : r_bytes))));
    char *ws = (char *)m->ws;
    char *d_in[2] = {ws, ws + in_dev};
    char *d_out[2] = {ws + 2 * in_dev, ws + 2 * in_dev + out_dev};
    char *d_tmp = ws + 2 * (in_dev + out_dev);
    cudaStream_t s_in = m->aux_stream[0], s_out = m->aux_stream[1], s_c = m->stream;
    cudaEvent_t *ev_in = &m->ev[0], *ev_c = &m->ev[2], *ev_out = &m->ev[4];
    const uint64_t nchunks = div_ceil64(count, chunk);
    core_fn fn = ext ? (core_fn)pgb_glwe_external_product_batched : (core_fn)pgb_glwe_keyswitch_batched;
    for (uint64_t c = 0; c < nchunks; c++) {
        const int s = (int)(c & 1);
        const uint64_t first = c * chunk, cnt = umin64(chunk, count - first);
        const char *src = (const char *)a_host + first * a_bytes;
        char *dst = (char *)res_host + first * r_bytes;
        if (c >= 2) {
            PGB_CHECK_CUDA(cudaStreamWaitEvent(s_in, ev_c[s], 0));
            if (!direct) { // pinned slot s is reused: drain chunk c-2 to the caller first
                PGB_CHECK_CUDA(cudaEventSynchronize(ev_out[s]));
                memcpy((char *)res_host + (first - 2 * chunk) * r_bytes, m->pinned[2 + s], (size_t)(chunk * r_bytes));
            }
        }
        if (!direct) {
            memcpy(m->pinned[s], src, (size_t)(cnt * a_bytes));
            src = (const char *)m->pinned[s];
            dst = (char *)m->pinned[2 + s];
        }
        PGB_CHECK_CUDA(cudaMemcpyAsync(d_in[s], src, cnt * a_bytes, cudaMemcpyHostToDevice, s_in));
        PGB_CHECK_CUDA(cudaEventRecord(ev_in[s], s_in));
        PGB_CHECK_CUDA(cudaStreamWaitEvent(s_c, ev_in[s], 0));
        if (c >= 2) PGB_CHECK_CUDA(cudaStreamWaitEvent(s_c, ev_out[s], 0));
        pgb_vec_znx av = {d_in[s], n, a_cols, a_size, a_size}, rv = {d_out[s], n, res_cols, res_size, res_size};
        pgb_batch bt = {cnt, r_bytes, a_bytes, 0};
        PGB_TRY(fn(m, &rv, res_base2k, &av, a_base2k, key, key_base2k, dsize, &bt, d_tmp, m->ws_len - (size_t)(d_tmp - ws)));
        PGB_CHECK_CUDA(cudaEventRecord(ev_c[s], s_c));
        PGB_CHECK_CUDA(cudaStreamWaitEvent(s_out, ev_c[s], 0));
        PGB_CHECK_CUDA(cudaMemcpyAsync(dst, d_out[s], cnt * r_bytes, cudaMemcpyDeviceToHost, s_out));
        PGB_CHECK_CUDA(cudaEventRecord(ev_out[s], s_out));
    }
    PGB_CHECK_CUDA(cudaStreamSynchronize(s_out));
    if (!direct) {
        for (uint64_t c = nchunks >= 2 ? nchunks - 2 : 0; c < nchunks; c++) {
            const int s = (int)(c & 1);
            const uint64_t first = c * chunk, cnt = umin64(chunk, count - first);
            memcpy((char *)res_host + first * r_bytes, m->pinned[2 + s], (size_t)(cnt * r_bytes));
        }
    }
    PGB_CHECK_CUDA(cudaStreamSynchronize(s_c));
    PGB_CHECK_CUDA(cudaStreamSynchronize(s_in));
    return PGB_OK;
}

extern "C" int pgb_glwe_keyswitch_host(pgb_module *m, int64_t *res_host, uint64_t res_size, uint64_t res_base2k, const int64_t *a_host,
                                       uint64_t a_size, uint64_t a_base2k, uint64_t rank_in, uint64_t rank_out, const pgb_vmp_pmat *key,
                                       uint64_t key_base2k, uint64_t dsize, uint64_t count) {
    PGB_REQUIRE(key->cols_in == rank_in && key->cols_out == rank_out + 1, "glwe_keyswitch_host: key shape does not match the ranks");
    return host_pipeline(m, false, res_host, rank_out + 1, res_size, res_base2k, a_host, rank_in + 1, a_size, a_base2k, key, key_base2k,
                         dsize, count);
}
extern "C" int pgb_glwe_external_product_host(pgb_module *m, int64_t *res_host, uint64_t res_size, uint64_t res_base2k,
                                              const int64_t *a_host, uint64_t a_size, uint64_t a_base2k, uint64_t rank,
                                              const pgb_vmp_pmat *ggsw, uint64_t ggsw_base2k, uint64_t dsize, uint64_t count) {
    PGB_REQUIRE(ggsw->cols_in == rank + 1 && ggsw->cols_out == rank + 1, "glwe_external_product_host: ggsw shape does not match the rank");
    return host_pipeline(m, true, res_host, rank + 1, res_size, res_base2k, a_host, rank + 1, a_size, a_base2k, ggsw, ggsw_base2k, dsize,
                         count);
}

// ---- one host call, several devices (Module is Sync + Send in the reference, poulpy-hal/src/layouts/module.rs:103-104: a Rust caller may
// drive one Module per GPU from one thread pool).  The batch is split contiguously over the modules (the first count % n_modules shards get
// one extra ciphertext, as poulpy_b200/sharding.py: shard_range), every shard runs the host pipeline of its module on its own host thread
// and device, and the call returns when every shard of res_host is complete.  keys[i] is the replica of the prepared key on modules[i]'s
// device (prepared keys are per-device memory).  No collective: the shards are independent (SURVEY 8e).
extern "C" int pgb_glwe_keyswitch_host_sharded(pgb_module *const *modules, const pgb_vmp_pmat *keys, uint64_t n_modules, int64_t *res_host,
                                               uint64_t res_size, uint64_t res_base2k, const int64_t *a_host, uint64_t a_size,
                                               uint64_t a_base2k, uint64_t rank_in, uint64_t rank_out, uint64_t key_base2k, uint64_t dsize,
                                               uint64_t count) {
    PGB_REQUIRE(modules && keys && n_modules >= 1, "glwe_keyswitch_host_sharded: no modules");
    for (uint64_t i = 0; i < n_modules; i++) {
        PGB_REQUIRE(modules[i] && modules[i]->n == modules[0]->n && modules[i]->flavour == modules[0]->flavour,
                    "glwe_keyswitch_host_sharded: modules must share n and flavour");
        for (uint64_t j = 0; j < i; j++) PGB_REQUIRE(modules[i] != modules[j], "glwe_keyswitch_host_sharded: a module may appear only once");
    }
    const uint64_t n = modules[0]->n;
    const uint64_t a_item = n * (rank_in + 1) * a_size, r_item = n * (rank_out + 1) * res_size; // i64 words per ciphertext
    std::vector<int> status(n_modules, PGB_OK);
    std::vector<std::string> message(n_modules);
    std::vector<std::thread> workers;
    const uint64_t base = count / n_modules, extra = count % n_modules;
    uint64_t first = 0;
    for (uint64_t i = 0; i < n_modules; i++) {
        const uint64_t cnt = base + (i < extra ? 1 : 0), start = first;
        first += cnt;
        if (cnt == 0) continue;
        workers.emplace_back([=, &status, &message]() {
            cudaSetDevice(modules[i]->device);
            status[i] = pgb_glwe_keyswitch_host(modules[i], res_host + start * r_item, res_size, res_base2k, a_host + start * a_item, a_size,
                                                a_base2k, rank_in, rank_out, &keys[i], key_base2k, dsize, cnt);
            if (status[i] != PGB_OK) message[i] = pgb_last_error(); // the message lives in the worker's thread-local slot
        });
    }
    for (auto &w : workers) w.join();
    for (uint64_t i = 0; i < n_modules; i++)
        if (status[i] != PGB_OK) {
            pgb_set_error("glwe_keyswitch_host_sharded: shard %llu (device %d): %s", (unsigned long long)i, modules[i]->device, message[i].c_str());
            return status[i];
        }
    return PGB_OK;
}
