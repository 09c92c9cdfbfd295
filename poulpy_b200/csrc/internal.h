// internal.h -- declarations shared between the translation units of libpoulpy_b200.so (not part of the ABI).
#pragma once
#include "common.cuh"

static inline uint64_t prep_bytes(const pgb_module *m) { return m->flavour == PGB_NTT120 ? 16 : 8; }
static inline uint64_t big_bytes(const pgb_module *m) { return m->flavour == PGB_NTT120 ? 16 : 8; }

// ---- scratch arena: every buffer carved from a caller's scratch starts at a 256-byte aligned offset -----------------------------------
static const uint64_t ALIGN = 256;
static inline uint64_t align_up(uint64_t x) { return (x + ALIGN - 1) / ALIGN * ALIGN; }
struct Arena {
    char *base;
    size_t len, used;
    void *take(size_t bytes) { // null when the buffer does not fit
        size_t off = align_up(used);
        if (off + bytes > len) return nullptr;
        used = off + bytes;
        return base + off;
    }
    // what is left after the buffers taken so far, for a nested call that carves its own scratch
    char *rest() const { return base + align_up(used); }
    size_t rest_len() const { return len - align_up(used); }
};
static inline pgb_vec_znx mk(void *data, uint64_t n, uint64_t cols, uint64_t size) {
    pgb_vec_znx v = {data, n, cols, size, size};
    return v;
}

// ---- aliasing (poulpy-hal/docs/backend_safety_contract.md "Aliasing": never UB, detect and reject) ----------------------------------
// byte extent of `count` items of `item` bytes laid out `stride` bytes apart (stride 0 = one shared item)
static inline uint64_t batch_extent(uint64_t item, uint64_t stride, uint64_t count) { return (count ? (count - 1) * stride : 0) + item; }
static inline bool ranges_overlap(const void *a, uint64_t alen, const void *b, uint64_t blen) {
    const char *a0 = (const char *)a, *b0 = (const char *)b;
    return alen && blen && a0 < b0 + blen && b0 < a0 + alen;
}
// 0: disjoint; 1: res IS a (same pointer, column count and batch stride, so limb (j, col) has one address on both sides: the reference's
// `_assign` forms); -1: any other overlap
static inline int vec_znx_alias_class(const pgb_vec_znx *res, uint64_t res_stride, const pgb_vec_znx *a, uint64_t a_stride, uint64_t count,
                                      uint64_t scalar_bytes = 8) {
    const uint64_t ri = res->n * res->cols * res->size * scalar_bytes, ai = a->n * a->cols * a->size * scalar_bytes;
    if (!ranges_overlap(res->data, batch_extent(ri, res_stride, count), a->data, batch_extent(ai, a_stride, count))) return 0;
    if (res->data == a->data && res->cols == a->cols && (count <= 1 || res_stride == a_stride)) return 1;
    return -1;
}
#define PGB_REQUIRE_DISJOINT(res, res_stride, a, a_stride, count, scalar_bytes, what)                                       \
    do {                                                                                                                   \
        if (vec_znx_alias_class((res), (res_stride), (a), (a_stride), (count), (scalar_bytes)) != 0) {                       \
            pgb_set_error("%s: res and a must not overlap", (what));                                                        \
            return PGB_ERR_ALIAS;                                                                                          \
        }                                                                                                                  \
    } while (0)

enum { EW_ADD = 0, EW_SUB = 1, EW_NEG = 2, EW_COPY = 3, EW_ZERO = 4, EW_MUL = 5 };
enum { BIG_ADD_SMALL = 0, BIG_FROM_SMALL = 1, BIG_ZERO = 2, BIG_SUB_SMALL = 3, BIG_SUB_SMALL_NEG = 4, BIG_NEG = 5 };

// ntt120_dft.cu
int ntt120_module_init(pgb_module *m);
int ntt120_forward(pgb_module *m, LimbSet in, LimbSet out, int jobs_per_batch, int batch, long long and_mask = -1);
// same, skipping the batch items b with skip[b] != 0 (device array); single-CTA sizes only.  skip_list: skip[batch] holds the number of
// items that are NOT skipped and skip[batch + 1 ..] their indices (the gadget kernel's fail list), so a small grid strides over those only
int ntt120_forward_skip(pgb_module *m, LimbSet in, LimbSet out, int jobs_per_batch, int batch, const int *skip, bool skip_list = false);
int ntt120_inverse_big(pgb_module *m, LimbSet in, LimbSet out, int jobs_per_batch, int batch);
bool ntt120_fused_supported(const pgb_module *m);
int ntt120_fused_back(pgb_module *m, const char *a_dft, uint64_t a_bs, const char *pmat, int R, int C, int cols_out, const char *small,
                      uint64_t small_bs, uint64_t small_limb_stride, int small_size, char *res, uint64_t res_bs, uint64_t res_limb_stride,
                      int res_size, int base2k, int64_t res_offset, int batch, const char *glwe, uint64_t glwe_bs, uint64_t glwe_words,
                      const int *skip = nullptr, bool skip_list = false, bool direct = false, bool small_all_cols = false,
                      uint64_t pmat_bs = 0, uint32_t pmat_div = 1);
// direct: a_dft already holds the C = cols_out * size product polys (limb-major, column-minor), pmat / R are ignored: inverse transform +
// CRT + add_small + normalize only; small_all_cols: `small` is added on every output column (CGGI: acc += ...), not only on column 0;
// pmat_bs: item b multiplies by the matrix at pmat + (b / pmat_div) * pmat_bs (0 = one matrix for the whole batch; the collapsed-key
// path needs 0); pmat_div > 1 gives pmat_div consecutive items one matrix (the levels of the CMux tree and of a BDD)
// max bit length of the integer coefficients of `polys` DFT polys -> *bits_dev (coef_ws: polys * 16n bytes of device scratch)
int ntt120_key_max_bits(pgb_module *m, const char *pmat, int polys, char *coef_ws, int *bits_dev);
// ntt120_gadget.cu
bool ntt120_gadget_supported(const pgb_module *m, int R, int cols_out, int S, int base2k, int batch);
int ntt120_gadget_fused(pgb_module *m, const char *in, uint64_t in_bs, int in_cols, int row_cols, int row_col0, int R, const char *pmat,
                        int C, int cols_out, int small_size, char *res, uint64_t res_bs, int res_size, int base2k, int batch, int *ok_out,
                        int dsize = 1, int a_size = 0, int key_rows = 0, int group_limit = 0, int aut_mode = 0, int64_t aut_p = 0,
                        int post_size = 0);
// fft64.cu: inverse transform + round + add of the column's own limbs + same-base2k normalisation of every (ciphertext, column), in place
bool fft64_fused_back_supported(const pgb_module *m, int S);
int fft64_fused_back(pgb_module *m, const char *in, uint64_t in_bs, int cols, int S, char *res, uint64_t res_bs, int res_size, int base2k, int batch);
// fft64_gadget.cu
bool fft64_gadget_supported(const pgb_module *m, int R, int cols_out, int S, int base2k, int batch);
int fft64_gadget_fused(pgb_module *m, const char *in, uint64_t in_bs, int in_cols, int row_cols, int row_col0, int R, const char *pmat, int C,
                       int cols_out, int small_size, char *res, uint64_t res_bs, int res_size, int base2k, int batch, int dsize = 1, int a_size = 0,
                       int key_rows = 0, int group_limit = 0, int aut_mode = 0, int64_t aut_p = 0, int post_size = 0);
// ntt120_ops.cu
int ntt120_vmp(pgb_module *m, const char *a, uint64_t a_bs, char *res, uint64_t res_bs, const char *pm, uint64_t pm_bs,
               uint32_t row_max, uint32_t C, uint32_t col0, uint32_t ncols_out, uint32_t batch, uint32_t pm_div = 1);
int ntt120_vmp_odd_last(pgb_module *m, const char *a, uint64_t a_bs, char *res_poly, uint64_t res_bs, const char *pm, uint64_t pm_bs,
                        uint32_t row_max, uint32_t C, uint32_t last, uint32_t batch, uint32_t pm_div = 1);
int ntt120_ew(pgb_module *m, int op, LimbSet dst, LimbSet a, LimbSet b, uint32_t jobs, uint32_t batch);
// fft64.cu
int fft64_module_init(pgb_module *m);
int fft64_forward(pgb_module *m, LimbSet in, LimbSet out, int jobs_per_batch, int batch, long long and_mask = -1);
int fft64_inverse_big(pgb_module *m, LimbSet in, LimbSet out, int jobs_per_batch, int batch);
int fft64_vmp(pgb_module *m, const char *a, uint64_t a_bs, char *res, uint64_t res_bs, const char *pm, uint64_t pm_bs,
              uint32_t row_max, uint32_t C, uint32_t col0, uint32_t ncols_out, uint32_t batch, uint32_t pm_div = 1);
int fft64_ew(pgb_module *m, int op, LimbSet dst, LimbSet a, LimbSet b, uint32_t jobs, uint32_t batch);
// cggi_fused.cu
bool cggi_fused_supported(const pgb_module *m, uint64_t cols, uint64_t dnum, uint64_t brk_size);
int cggi_fused_fft64(pgb_module *m, long long *res, uint64_t res_stride_words, const long long *lwe, uint64_t lwe_stride, const double *brk,
                     uint64_t brk_doubles, const double *xpa, int n_lwe, int block_size, int base2k, int cols, int dnum, int brk_size,
                     int out_size, int batch);
// cggi_ntt_fused.cu: whole-rotation NTT120 kernel with two primes when the device-measured bound allows; *handled = false -> caller runs
// the four-prime limb-wise path (after re-initialising res)
bool cggi_ntt_fused_supported(const pgb_module *m, uint64_t cols, uint64_t dnum, uint64_t brk_size, uint64_t block_size);
int cggi_fused_ntt120(pgb_module *m, long long *res, uint64_t res_stride_words, const long long *lwe, uint64_t lwe_stride, const char *brk,
                      uint64_t brk_bytes, const char *xpa, int n_lwe, int block_size, int base2k, int cols, int dnum, int brk_size,
                      int out_size, int batch, const long long *lut, uint64_t lut_words, bool *handled);
// big.cu
int big_normalize(pgb_module *m, bool big_is_i128, LimbSet res, int res_size, int res_k, int64_t res_offset, LimbSet a, int a_size,
                  int a_k, int op, uint32_t batch);
int big_ew(pgb_module *m, bool big_is_i128, int op, LimbSet dst, LimbSet a, uint32_t jobs, uint32_t batch);
int znx_rotate(pgb_module *m, LimbSet dst, LimbSet a, long long p, const long long *p_dev, uint32_t p_stride, uint32_t jobs, uint32_t batch);
int znx_ew(pgb_module *m, int op, LimbSet dst, LimbSet a, long long p, const long long *p_dev, uint32_t p_stride, uint32_t jobs, uint32_t batch);
int znx_automorphism(pgb_module *m, LimbSet dst, LimbSet a, long long p, uint32_t jobs, uint32_t batch, bool big_is_i128 = false);
int znx_rsh_assign(pgb_module *m, LimbSet r, int size, int base2k, int k, uint32_t batch, uint32_t words = 0);
int raw_limbs(pgb_module *m, bool zero, LimbSet dst, LimbSet a, uint64_t limb_bytes, uint32_t jobs, uint32_t batch);
// cnv.cu
int cnv_apply(pgb_module *m, LimbSet res, int res_size, LimbSet a, LimbSet a2, int a_size, LimbSet b, LimbSet b2, int b_size, uint64_t cnv_offset,
              uint32_t batch);
int cnv_by_const(pgb_module *m, LimbSet res, int res_size, LimbSet a, int a_size, const long long *b_dev, int b_size, uint64_t cnv_offset,
                 uint32_t batch);
int cnv_prepare_impl(pgb_module *m, pgb_vec_znx_dft *res, const pgb_vec_znx *a, int64_t mask, const pgb_batch *bt);
// key_cache.cu: cached gadget-kernel forms of pinned keys.  sig = what the cached bytes depend on besides the key itself
enum { KEY_SIG_WORDS = 10 };
bool key_is_pinned(const pgb_module *m, const void *key);
void *key_cache_find(pgb_module *m, const void *key, const uint64_t *sig);
int key_cache_insert(pgb_module *m, const void *key, uint64_t key_len, const uint64_t *sig, size_t bytes, void **out);
int64_t *key_cache_host_slot(pgb_module *m, const void *key, uint64_t key_len, const uint64_t *sig);
void key_cache_invalidate(pgb_module *m, const void *p, uint64_t len);
void key_cache_destroy(pgb_module *m);
// core.cu: lazily grown device workspace of the host front ends; whether a host pointer is page-locked
int ensure_ws(pgb_module *m, size_t len);
bool is_pinned(const void *p);
// core.cu: the limb-wise external product (item b's GGSW at ggsw + (b / ggsw_div) * ggsw_bs, ggsw_bs = 0: shared) and its
// normalisation into res; the input ain is in ggsw_base2k, res_dft / a_dft / tmp (dsize > 1 only) are scratch of the external product's layout
int external_product_limbwise(pgb_module *m, pgb_vec_znx *res, uint64_t res_bs, uint64_t res_base2k, const pgb_vec_znx *ain, uint64_t ain_bs,
                              const pgb_vmp_pmat *ggsw, uint64_t ggsw_bs, uint32_t ggsw_div, uint64_t ggsw_base2k, uint64_t dsize, uint64_t B,
                              pgb_vec_znx_dft *res_dft, pgb_vec_znx_dft *a_dft, void *tmp);
// core.cu: the input of a gadget product in the key's base: a itself when the bases agree, otherwise every column of a normalised from
// base 2^from into base 2^to (ceil(a.size * from / to) limbs), in a buffer taken from `ar`
int glwe_to_base2k(pgb_module *m, Arena &ar, const pgb_vec_znx *a, uint64_t a_bs, uint64_t from, uint64_t to, uint64_t B, pgb_vec_znx *out,
                   uint64_t *out_bs);
// api.cu (used by core.cu); item b's matrix at pmat + (b / pm_div) * bt->stride_b
int vmp_apply_impl(pgb_module *m, pgb_vec_znx_dft *res, const pgb_vec_znx_dft *a, const pgb_vmp_pmat *pmat, uint64_t limb_offset,
                   const pgb_batch *bt, uint32_t pm_div = 1);
int big_normalize_impl(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, int64_t res_offset, uint64_t res_col,
                       const pgb_vec_znx_big *a, uint64_t a_base2k, uint64_t a_col, int op, bool a_is_big, const pgb_batch *bt);
int big_add_small_impl(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col, const pgb_batch *bt);
// op: BIG_ADD_SMALL (res += a), BIG_SUB_SMALL (res -= a), BIG_SUB_SMALL_NEG (res = a - res, limbs of res beyond a.size negated)
int big_small_op_impl(pgb_module *m, int op, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col, const pgb_batch *bt);
int big_automorphism_impl(pgb_module *m, int64_t p, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx_big *a, uint64_t a_col,
                          const pgb_batch *bt);
int rsh_assign_impl(pgb_module *m, uint64_t base2k, uint64_t k, pgb_vec_znx *res, uint64_t res_col, const pgb_batch *bt);
