// lwe.cu -- the conversions between the blind rotation's GLWE output and the LWE the next gate reads, batched and device resident:
// sample extraction and GLWE -> LWE (poulpy-core/src/conversion/glwe_to_lwe.rs), LWE key-switching (keyswitching/lwe.rs) and LWE -> GLWE
// (conversion/lwe_to_glwe.rs).
//
// An LWE is a one-column VecZnx of n_lwe + 1 coefficients per limb, (b, a_0, .., a_{n_lwe-1}), phase b + <a, s_lwe>.  Under the GLWE
// embedding s_glwe(X) = s_lwe(X^-1) (zero padded to N) coefficient 0 of c0 + c1 s_glwe is c0[0] + <c1[0..n_lwe), s_lwe>, so both layout
// changes are plain copies.  All arithmetic is pgb_glwe_keyswitch_batched on rank-1 GLWEs staged in the caller's scratch; the two kernels
// here only move 8-byte words.  An LWE row is (n_lwe + 1) * 8 bytes, for the usual n_lwe an odd multiple of 8: every LWE access is one
// 8-byte word per thread, never a 16-byte vector or a bulk copy.
#include "internal.h"

// ---- kernels: one thread per output coefficient, grid (coefficient, limb, ciphertext) ----------------------------------------------------
struct LweEmbedArgs {
    const char *lwe; uint64_t lwe_bs; // item b at lwe + b * lwe_bs, limb j at + j * (n_in + 1) words
    char *glwe; uint64_t glwe_bs;     // rank-1 GLWE VecZnx(n, 2, size): limb j, column c at + (2 j + c) * n words
    uint32_t n, n_in;
};
// Every coefficient of the staged GLWE is written, the zeros included: the scratch it lives in is shared and dirty.
__global__ void __launch_bounds__(256) lwe_embed_kernel(LweEmbedArgs p) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; // column * n + coefficient
    if (t >= 2 * p.n) return;
    const uint32_t j = blockIdx.y;
    const long long *src = reinterpret_cast<const long long *>(p.lwe + (size_t)blockIdx.z * p.lwe_bs) + (size_t)j * (p.n_in + 1);
    long long v = 0;
    if (t == 0) v = src[0];
    else if (t >= p.n && t - p.n < p.n_in) v = src[1 + (t - p.n)];
    reinterpret_cast<long long *>(p.glwe + (size_t)blockIdx.z * p.glwe_bs)[(size_t)j * 2 * p.n + t] = v;
}

struct LweExtractArgs {
    const char *glwe; uint64_t glwe_bs; // rank-1 GLWE VecZnx(n, 2, >= copy limbs)
    char *lwe; uint64_t lwe_bs;         // LWE VecZnx(len, 1, gridDim.y limbs)
    uint32_t n, len, copy;              // len = n_lwe + 1; limbs j < copy are copied, the others zeroed
};
__global__ void __launch_bounds__(256) lwe_extract_kernel(LweExtractArgs p) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= p.len) return;
    const uint32_t j = blockIdx.y;
    long long v = 0;
    if (j < p.copy)
        v = reinterpret_cast<const long long *>(p.glwe + (size_t)blockIdx.z * p.glwe_bs)[(size_t)j * 2 * p.n + (t == 0 ? 0 : p.n + t - 1)];
    reinterpret_cast<long long *>(p.lwe + (size_t)blockIdx.z * p.lwe_bs)[(size_t)j * p.len + t] = v;
}

static int launch_embed(pgb_module *m, char *glwe, uint64_t glwe_bs, const pgb_vec_znx *a, uint64_t a_bs, uint64_t B) {
    LweEmbedArgs p = {(const char *)a->data, a_bs, glwe, glwe_bs, (uint32_t)m->n, (uint32_t)(a->n - 1)};
    { ProfScope _ps(m, PROF_OTHER);
    lwe_embed_kernel<<<dim3((uint32_t)((2 * m->n + 255) / 256), (uint32_t)a->size, (uint32_t)B), 256, 0, m->stream>>>(p);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

static int launch_extract(pgb_module *m, pgb_vec_znx *res, uint64_t res_bs, const char *glwe, uint64_t glwe_bs, uint64_t glwe_size, uint64_t B) {
    LweExtractArgs p = {glwe, glwe_bs, (char *)res->data, res_bs, (uint32_t)m->n, (uint32_t)res->n, (uint32_t)umin64(res->size, glwe_size)};
    { ProfScope _ps(m, PROF_OTHER);
    lwe_extract_kernel<<<dim3((uint32_t)((res->n + 255) / 256), (uint32_t)res->size, (uint32_t)B), 256, 0, m->stream>>>(p);
    }
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

// ---- shape checks (all of them before the first launch) ----------------------------------------------------------------------------------
static int check_batch(const char *what, const pgb_batch *bt) {
    PGB_REQUIRE(bt && bt->count >= 1 && bt->count <= 65535, "%s: batch count must be in [1, 65535]", what);
    return PGB_OK;
}
// size in [1, 65535] (a grid dimension), data non-null, data and stride multiples of `align` bytes, stride at least one item.  LWEs need 8;
// GLWEs need 16: the key-switch kernels read them with 16-byte loads and 16-byte L2 bulk prefetches
static int check_layout(const char *what, const char *name, const pgb_vec_znx *v, uint64_t stride, uint64_t count, uint64_t align) {
    PGB_REQUIRE(v->size >= 1 && v->size <= 65535, "%s: %s has %llu limbs (must be in [1, 65535])", what, name, (unsigned long long)v->size);
    PGB_REQUIRE(v->data != nullptr && (uintptr_t)v->data % align == 0, "%s: %s data must be non-null and %llu-byte aligned", what, name,
                (unsigned long long)align);
    const uint64_t item = v->n * v->cols * v->size * 8;
    PGB_REQUIRE(stride % align == 0 && (count == 1 || stride >= item),
                "%s: %s batch stride %llu must be a multiple of %llu and at least one item (%llu bytes)", what, name, (unsigned long long)stride,
                (unsigned long long)align, (unsigned long long)item);
    return PGB_OK;
}
// LWE descriptors have n = n_lwe + 1, not the module's n
static int check_lwe(const char *what, const char *name, const pgb_module *m, const pgb_vec_znx *v, uint64_t stride, uint64_t count) {
    PGB_REQUIRE(v->cols == 1 && v->n >= 2 && v->n - 1 <= m->n,
                "%s: %s must be a one-column VecZnx of n_lwe + 1 coefficients with 1 <= n_lwe <= N = %llu (got n = %llu, cols = %llu)", what, name,
                (unsigned long long)m->n, (unsigned long long)v->n, (unsigned long long)v->cols);
    return check_layout(what, name, v, stride, count, 8);
}
static int check_glwe(const char *what, const char *name, const pgb_module *m, const pgb_vec_znx *v, uint64_t cols, uint64_t stride, uint64_t count) {
    PGB_REQUIRE(v->n == m->n, "%s: %s has ring degree %llu, the module %llu", what, name, (unsigned long long)v->n, (unsigned long long)m->n);
    PGB_REQUIRE(v->cols == cols, "%s: %s has %llu columns, %llu expected (rank %llu)", what, name, (unsigned long long)v->cols,
                (unsigned long long)cols, (unsigned long long)(cols - 1));
    return check_layout(what, name, v, stride, count, 16);
}
static int check_key(const char *what, const pgb_module *m, const pgb_vmp_pmat *key, uint64_t cols_in, uint64_t cols_out, uint64_t dsize) {
    PGB_REQUIRE(key && key->data && key->n == m->n && key->rows >= 1 && key->size >= 1, "%s: the key must be a non-empty VmpPMat of ring degree %llu",
                what, (unsigned long long)m->n);
    PGB_REQUIRE(key->cols_in == cols_in && key->cols_out == cols_out, "%s: key is VmpPMat(cols_in %llu, cols_out %llu), (%llu, %llu) expected", what,
                (unsigned long long)key->cols_in, (unsigned long long)key->cols_out, (unsigned long long)cols_in, (unsigned long long)cols_out);
    PGB_REQUIRE(dsize >= 1, "%s: dsize must be >= 1", what);
    return PGB_OK;
}
// the staged GLWEs start the scratch, and the inner key-switch carves its buffers at 256-byte offsets from there
static int check_scratch(const char *what, const void *scratch, size_t have, uint64_t need) {
    PGB_REQUIRE(scratch != nullptr && (uintptr_t)scratch % 256 == 0, "%s: scratch must be non-null and 256-byte aligned", what);
    if (have < need) {
        pgb_set_error("%s: scratch of %zu bytes < required %llu", what, have, (unsigned long long)need);
        return PGB_ERR_SCRATCH;
    }
    return PGB_OK;
}

// ---- LWE::sample_extract (conversion/glwe_to_lwe.rs) ----------------------------------------------------------------------------------------
// res[i][0] = a[0][i][0], res[i][1..=n_lwe] = a[1][i][0..n_lwe) for i < min(res.size, a.size); every other limb of res is zeroed
extern "C" int pgb_lwe_sample_extract_batched(pgb_module *m, pgb_vec_znx *res, const pgb_vec_znx *a, const pgb_batch *bt) {
    const char *what = "lwe_sample_extract";
    PGB_TRY(check_batch(what, bt));
    const uint64_t B = bt->count;
    PGB_TRY(check_lwe(what, "res", m, res, bt->stride_res, B));
    PGB_TRY(check_glwe(what, "a", m, a, 2, bt->stride_a, B));
    PGB_REQUIRE_DISJOINT(res, bt->stride_res, a, bt->stride_a, B, 8, what);
    return launch_extract(m, res, bt->stride_res, (const char *)a->data, bt->stride_a, a->size, B);
}

// ---- LWE::keyswitch (keyswitching/lwe.rs): embed -> glwe_keyswitch -> extract ---------------------------------------------------------
extern "C" size_t pgb_lwe_keyswitch_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t a_base2k, const pgb_vmp_pmat *key,
                                              uint64_t key_base2k, uint64_t dsize, uint64_t batch) {
    return align_up(batch * m->n * 2 * a_size * 8) + align_up(batch * m->n * 2 * res_size * 8) +
           pgb_glwe_keyswitch_tmp_bytes(m, res_size, a_size, a_base2k, key, key_base2k, dsize, batch);
}
extern "C" int pgb_lwe_keyswitch_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a, uint64_t a_base2k,
                                         const pgb_vmp_pmat *key, uint64_t key_base2k, uint64_t dsize, const pgb_batch *bt, void *scratch,
                                         size_t scratch_len) {
    const char *what = "lwe_keyswitch";
    PGB_TRY(check_batch(what, bt));
    const uint64_t B = bt->count, n = m->n;
    PGB_TRY(check_lwe(what, "res", m, res, bt->stride_res, B));
    PGB_TRY(check_lwe(what, "a", m, a, bt->stride_a, B));
    PGB_TRY(check_key(what, m, key, 1, 2, dsize));
    PGB_REQUIRE_DISJOINT(res, bt->stride_res, a, bt->stride_a, B, 8, what);
    PGB_TRY(check_scratch(what, scratch, scratch_len, pgb_lwe_keyswitch_tmp_bytes(m, res->size, a->size, a_base2k, key, key_base2k, dsize, B)));
    const uint64_t in_bs = n * 2 * a->size * 8, out_bs = n * 2 * res->size * 8;
    Arena ar = {(char *)scratch, scratch_len, 0};
    char *in = (char *)ar.take(B * in_bs), *out = (char *)ar.take(B * out_bs);
    pgb_vec_znx gin = mk(in, n, 2, a->size), gout = mk(out, n, 2, res->size);
    PGB_TRY(launch_embed(m, in, in_bs, a, bt->stride_a, B));
    pgb_batch btk = {B, out_bs, in_bs, 0};
    PGB_TRY(pgb_glwe_keyswitch_batched(m, &gout, res_base2k, &gin, a_base2k, key, key_base2k, dsize, &btk, ar.rest(), ar.rest_len()));
    return launch_extract(m, res, bt->stride_res, out, out_bs, res->size, B);
}

// ---- LWE::from_glwe (conversion/glwe_to_lwe.rs): glwe_keyswitch to rank 1 -> extract -------------------------------------------------------
extern "C" size_t pgb_glwe_to_lwe_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t a_base2k, const pgb_vmp_pmat *key,
                                            uint64_t key_base2k, uint64_t dsize, uint64_t batch) {
    return align_up(batch * m->n * 2 * res_size * 8) + pgb_glwe_keyswitch_tmp_bytes(m, res_size, a_size, a_base2k, key, key_base2k, dsize, batch);
}
extern "C" int pgb_glwe_to_lwe_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a, uint64_t a_base2k,
                                       const pgb_vmp_pmat *key, uint64_t key_base2k, uint64_t dsize, const pgb_batch *bt, void *scratch,
                                       size_t scratch_len) {
    const char *what = "glwe_to_lwe";
    PGB_TRY(check_batch(what, bt));
    const uint64_t B = bt->count, n = m->n;
    PGB_TRY(check_lwe(what, "res", m, res, bt->stride_res, B));
    PGB_REQUIRE(a->cols >= 2, "%s: a must be a GLWE of rank >= 1", what);
    PGB_TRY(check_glwe(what, "a", m, a, a->cols, bt->stride_a, B));
    PGB_TRY(check_key(what, m, key, a->cols - 1, 2, dsize));
    PGB_REQUIRE_DISJOINT(res, bt->stride_res, a, bt->stride_a, B, 8, what);
    PGB_TRY(check_scratch(what, scratch, scratch_len, pgb_glwe_to_lwe_tmp_bytes(m, res->size, a->size, a_base2k, key, key_base2k, dsize, B)));
    const uint64_t out_bs = n * 2 * res->size * 8;
    Arena ar = {(char *)scratch, scratch_len, 0};
    char *out = (char *)ar.take(B * out_bs);
    pgb_vec_znx gout = mk(out, n, 2, res->size);
    pgb_batch btk = {B, out_bs, bt->stride_a, 0};
    PGB_TRY(pgb_glwe_keyswitch_batched(m, &gout, res_base2k, a, a_base2k, key, key_base2k, dsize, &btk, ar.rest(), ar.rest_len()));
    return launch_extract(m, res, bt->stride_res, out, out_bs, res->size, B);
}

// ---- GLWE::from_lwe (conversion/lwe_to_glwe.rs): embed -> glwe_keyswitch to rank k ------------------------------------------------------------
extern "C" size_t pgb_lwe_to_glwe_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t a_base2k, const pgb_vmp_pmat *key,
                                            uint64_t key_base2k, uint64_t dsize, uint64_t batch) {
    return align_up(batch * m->n * 2 * a_size * 8) + pgb_glwe_keyswitch_tmp_bytes(m, res_size, a_size, a_base2k, key, key_base2k, dsize, batch);
}
extern "C" int pgb_lwe_to_glwe_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a, uint64_t a_base2k,
                                       const pgb_vmp_pmat *key, uint64_t key_base2k, uint64_t dsize, const pgb_batch *bt, void *scratch,
                                       size_t scratch_len) {
    const char *what = "lwe_to_glwe";
    PGB_TRY(check_batch(what, bt));
    const uint64_t B = bt->count, n = m->n;
    PGB_TRY(check_lwe(what, "a", m, a, bt->stride_a, B));
    PGB_REQUIRE(res->cols >= 2, "%s: res must be a GLWE of rank >= 1", what);
    PGB_TRY(check_glwe(what, "res", m, res, res->cols, bt->stride_res, B));
    PGB_TRY(check_key(what, m, key, 1, res->cols, dsize));
    PGB_REQUIRE_DISJOINT(res, bt->stride_res, a, bt->stride_a, B, 8, what);
    PGB_TRY(check_scratch(what, scratch, scratch_len, pgb_lwe_to_glwe_tmp_bytes(m, res->size, a->size, a_base2k, key, key_base2k, dsize, B)));
    const uint64_t in_bs = n * 2 * a->size * 8;
    Arena ar = {(char *)scratch, scratch_len, 0};
    char *in = (char *)ar.take(B * in_bs);
    pgb_vec_znx gin = mk(in, n, 2, a->size);
    PGB_TRY(launch_embed(m, in, in_bs, a, bt->stride_a, B));
    pgb_batch btk = {B, bt->stride_res, in_bs, 0};
    return pgb_glwe_keyswitch_batched(m, res, res_base2k, &gin, a_base2k, key, key_base2k, dsize, &btk, ar.rest(), ar.rest_len());
}
