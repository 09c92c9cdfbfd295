// cmux.cu -- the CMux of poulpy-bin-fhe (glwe_sub, glwe_normalize_inplace, glwe_external_product_inplace, glwe_add_inplace,
// glwe_normalize_inplace), batched and device resident, with one prepared GGSW selector per ciphertext or one shared by the batch:
//
//     res = normalize( normalize(t - f) (x) s_b + f )
//
// t, f, res are GLWEs of rank k in base 2^base2k; s_b = s.data + b * ggsw_stride is a prepared GGSW (VmpPMat(dnum, k + 1, k + 1, size))
// in base 2^ggsw_base2k.  The difference kernel below writes normalize(t - f) in one pass; the external product and the final add +
// normalise run on the routes described at cmux_launch.  The blind rotation by GGSW bits (pgb_glwe_blind_rotate_ggsw_batched) chains one
// CMux per bit, acc <- cmux(X^(step 2^i) acc, acc, s_{b,i}), through the same routes; the CMux tree (pgb_glwe_cmux_tree_batched) runs one
// batched CMux per level, g_{i+1,j} = cmux(g_{i,2j+1}, g_{i,2j}, s_{b,i}); the BDD evaluator (pgb_glwe_bdd_eval_batched) runs one
// batched CMux per level of a circuit given as data, each node reading its children through a descriptor table.
#include "internal.h"
#include <vector>

// ---- d = normalize_assign(X^rot t - f) ------------------------------------------------------------------------------------------------
// One thread per (coefficient, column, ciphertext).  Limb j < size of d is t[j] - f[j] in wrapping i64 (a limb missing from an operand
// reads as 0), normalised from the last limb up with the carry in a register: the lsh = 0 steps of vec_znx_normalize_assign
// (reference/vec_znx/normalize.rs:403-425), whose first step keeps only the digit and whose last step drops the carry.  `fr`, when set,
// receives f (limbs >= f_size zeroed) in the same pass: the FFT64 fused route adds it inside its carry chain, and level 0 of the CMux tree
// hands every route this linear copy instead of the scattered leaves.
// DIFF_ROT reads t as X^rot t (rot = p mod 2n), the negacyclic index and sign of rotate_kernel (big.cu), so the blind rotation's rotated
// operand is never written.  DIFF_LEAF is level 0 of the CMux tree: grid item q = b * 2^lp + j reads t and f at item b's leaves 2j + 1
// and 2j (t_bs = f_bs = the table stride, t = f + the leaf stride, pair_bs = twice the leaf stride).  DIFF_GATHER is a level of a BDD:
// grid item q = b * P + j reads node j's descriptor, t and f at (src ? state : leaf) + off + b * bs with their own limb counts.  DIFF_PLAIN
// is the CMux's kernel.
enum { DIFF_PLAIN = 0, DIFF_ROT = 1, DIFF_LEAF = 2, DIFF_GATHER = 3 };
// an operand of every item of a chunk: item b's GLWE at (src ? state : leaf) + off + b * bs, `size` limbs (src 0: a leaf, relative to the
// chunk's leaf base; src 1: a node, relative to the scratch, where each level's block sits at the same place in every chunk)
struct GatherSrc { uint64_t off, bs; uint32_t src, size; };
struct GatherNode { GatherSrc t, f; };
struct CmuxDiffArgs {
    const char *t; uint64_t t_bs; // VecZnx(cols, t_size) per item, limb j at + j * words words
    const char *f; uint64_t f_bs; // VecZnx(cols, f_size)
    char *d;       uint64_t d_bs; // VecZnx(cols, size)
    char *fr;      uint64_t fr_bs; // VecZnx(cols, size) or null
    uint32_t words;               // n * cols: words per limb
    uint32_t n, rot;              // ring degree, and the rotation of t in [0, 2n) (DIFF_ROT only)
    int t_size, f_size, size, K;
    uint64_t pair_bs; uint32_t lp; // DIFF_LEAF only
    const GatherNode *desc; const char *leaf, *state; uint32_t P; // DIFF_GATHER only: the level's descriptors and its width
};
template <int MODE>
__global__ void __launch_bounds__(256) cmux_diff_kernel(CmuxDiffArgs p) {
    constexpr bool ROT = MODE == DIFF_ROT;
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x; // column * n + coefficient
    if (u >= p.words) return;
    const size_t b = blockIdx.y, ls = p.words;
    // operand offsets of grid item b: linear, or (DIFF_LEAF) its table and its leaf pair
    const size_t ob = MODE == DIFF_LEAF ? (b >> p.lp) : b, oj = MODE == DIFF_LEAF ? (b & ((1u << p.lp) - 1)) * p.pair_bs : 0;
    const char *tp = p.t + ob * p.t_bs + oj, *fp = p.f + ob * p.f_bs + oj;
    int t_size = p.t_size, f_size = p.f_size;
    if (MODE == DIFF_GATHER) {
        const uint32_t bi = (uint32_t)b / p.P, j = (uint32_t)b - bi * p.P;
        const GatherNode g = p.desc[j];
        tp = (g.t.src ? p.state : p.leaf) + g.t.off + bi * g.t.bs;
        fp = (g.f.src ? p.state : p.leaf) + g.f.off + bi * g.f.bs;
        t_size = (int)g.t.size;
        f_size = (int)g.f.size;
    }
    uint32_t tu = u;
    bool neg = false;
    if (ROT) { // (X^rot t)[i] = +-t[(i - rot) mod n], negated when exactly one of i < rot mod n, rot >= n holds
        const uint32_t i = u & (p.n - 1), r = p.rot & (p.n - 1);
        tu = u - i + (i >= r ? i - r : i + p.n - r);
        neg = (i < r) == (p.rot < p.n);
    }
    const long long *t = reinterpret_cast<const long long *>(tp) + tu;
    const long long *f = reinterpret_cast<const long long *>(fp) + u;
    long long *d = reinterpret_cast<long long *>(p.d + b * p.d_bs) + u;
    long long *fr = p.fr ? reinterpret_cast<long long *>(p.fr + b * p.fr_bs) + u : nullptr;
    const int sh = 64 - p.K;
    long long carry = 0;
    for (int j = p.size - 1; j >= 0; j--) {
        long long tv = j < t_size ? __ldg(t + (size_t)j * ls) : 0;
        if (ROT && neg) tv = (long long)(0ull - (unsigned long long)tv);
        const long long fv = j < f_size ? __ldg(f + (size_t)j * ls) : 0;
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

// level 0 of the CMux tree: CMux q = b * 2^lp + j reads t = leaf 2j + 1 and f = leaf 2j of item b, leaf l at a + b * a_bs + l * entry_stride
struct LeafPairs {
    const pgb_vec_znx *a;
    uint64_t a_bs, entry_stride;
    uint32_t lp;
};

// a level of a BDD: CMux q = b * P + j reads node j's operands through desc[j] (device memory)
struct NodeGather {
    const GatherNode *desc;
    const char *leaf, *state;
    uint32_t P;
    uint64_t f_size; // the level's f.size: res.size when an f child is a node, min(a.size, res.size) otherwise
    char *fr;        // the linear copy of f the difference kernel writes (B GLWEs of res.size limbs), off the FFT64 fused route
};

// the CMux operands: t (read as X^rot t) and f, item q at + q * t_bs / f_bs, or the leaf pairs of `lv`, or the nodes of `gv` (t and f
// then only give the column count)
struct CmuxIn {
    const pgb_vec_znx *t; uint64_t t_bs; uint32_t rot;
    const pgb_vec_znx *f; uint64_t f_bs;
    const LeafPairs *lv;
    const NodeGather *gv;
};

static int launch_diff(pgb_module *m, char *d, uint64_t d_bs, uint64_t size, const CmuxIn &in, char *fr, uint64_t fr_bs, uint64_t base2k,
                       uint64_t B) {
    const uint64_t words = m->n * in.t->cols;
    CmuxDiffArgs p = {(const char *)in.t->data, in.t_bs, (const char *)in.f->data, in.f_bs, d, d_bs, fr, fr_bs, (uint32_t)words,
                      (uint32_t)m->n, in.rot, (int)in.t->size, (int)in.f->size, (int)size, (int)base2k, 0, 0, nullptr, nullptr, nullptr, 0};
    if (in.lv) {
        p.t = (const char *)in.lv->a->data + in.lv->entry_stride;
        p.f = (const char *)in.lv->a->data;
        p.t_bs = p.f_bs = in.lv->a_bs;
        p.t_size = p.f_size = (int)in.lv->a->size;
        p.pair_bs = 2 * in.lv->entry_stride;
        p.lp = in.lv->lp;
    }
    if (in.gv) {
        p.desc = in.gv->desc;
        p.leaf = in.gv->leaf;
        p.state = in.gv->state;
        p.P = in.gv->P;
    }
    const dim3 grid((uint32_t)((words + 255) / 256), (uint32_t)B);
    { ProfScope _ps(m, PROF_NORMALIZE);
    if (in.lv) cmux_diff_kernel<DIFF_LEAF><<<grid, 256, 0, m->stream>>>(p);
    else if (in.gv) cmux_diff_kernel<DIFF_GATHER><<<grid, 256, 0, m->stream>>>(p);
    else if (in.rot) cmux_diff_kernel<DIFF_ROT><<<grid, 256, 0, m->stream>>>(p);
    else cmux_diff_kernel<DIFF_PLAIN><<<grid, 256, 0, m->stream>>>(p);
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
static int check_glwe(const char *who, const char *name, const pgb_module *m, const pgb_vec_znx *v, uint64_t cols, uint64_t stride, uint64_t count,
                      bool shared_ok) {
    PGB_REQUIRE(v->n == m->n, "%s: %s has ring degree %llu, the module %llu", who, name, (unsigned long long)v->n, (unsigned long long)m->n);
    PGB_REQUIRE(v->cols == cols, "%s: %s has %llu columns, the selector %llu", who, name, (unsigned long long)v->cols, (unsigned long long)cols);
    PGB_REQUIRE(v->size <= 65535, "%s: %s has %llu limbs", who, name, (unsigned long long)v->size);
    PGB_REQUIRE(v->data != nullptr && (uintptr_t)v->data % 16 == 0, "%s: %s data must be non-null and 16-byte aligned", who, name);
    const uint64_t item = v->n * v->cols * v->size * 8;
    PGB_REQUIRE(stride % 16 == 0 && (count == 1 || stride >= item || (shared_ok && stride == 0)),
                "%s: %s batch stride %llu must be a multiple of 16 and at least one item (%llu bytes)%s", who, name, (unsigned long long)stride,
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

// Steps 1-5 for B items after the caller's checks: t is read as X^rot t (rot in [0, 2n); 0 for the CMux), item b's selector at
// s->data + (b / sel_div) * ggsw_stride, and the buffers come from `scratch` (pgb_glwe_cmux_tmp_bytes of res.size limbs, plus one more
// GLWE batch of res.size limbs when in.lv is set).  Routes (all bit-exact with the five steps; DESIGN.md §3.5b):
//  * ggsw_stride == 0: d in scratch, then pgb_glwe_external_product_batched (with its single-kernel routes, gadget_fused in core.cu),
//    add f, normalise.
//  * per-item selectors, dsize == 1, ggsw_base2k == base2k, f.size <= min(res.size, s.size), fusion on:
//      NTT120 (n = 2^9 .. 2^13): d -> forward transform -> ntt120_fused_back with the per-item matrix stride and small = f on every column;
//      FFT64 (fft64_fused_back_supported): d and res = f -> forward transform -> vmp with the per-item matrix stride -> fft64_fused_back,
//      which adds res's own limbs inside its carry chain.
//    Both replace normalize(normalize(big) + f) by normalize(big + f): equal because f has no limb where the big integer is truncated.
//  * anything else: d -> (base conversion) -> the limb-wise external product with the per-item matrix stride -> add f, normalise.
// With leaf pairs (in.lv: level 0 of the CMux tree, f not affine in the item) the difference kernel also writes a linear copy of f, into
// res on the FFT64 fused route as always and into a scratch batch on the others, and steps 4-5 read that copy.  With node descriptors
// (in.gv: a level of a BDD) the same holds, the copy going to in.gv->fr off the FFT64 fused route, and f.size is the level's in.gv->f_size.
static int cmux_launch(pgb_module *m, pgb_vec_znx *res, uint64_t res_bs, const CmuxIn &in, uint64_t base2k, const pgb_vmp_pmat *s,
                       uint64_t ggsw_stride, uint32_t sel_div, uint64_t ggsw_base2k, uint64_t dsize, uint64_t B, void *scratch,
                       size_t scratch_len) {
    // ---- step 1 + 2 on every route: d = normalize(t - f), res.size limbs -----------------------------------------------------------------
    const uint64_t n = m->n, cols = s->cols_in, pb = prep_bytes(m);
    const uint64_t S = s->size, rs = res->size;
    const uint64_t d_bs = n * cols * rs * 8;
    const uint64_t f_size = in.gv ? in.gv->f_size : in.f->size;
    const bool fuse = ggsw_stride != 0 && dsize == 1 && ggsw_base2k == base2k && f_size <= umin64(rs, S) && !opt_on(m, PGB_OPT_NO_FUSION);
    const bool fuse_ntt = fuse && ntt120_fused_supported(m), fuse_fft = fuse && !fuse_ntt && fft64_fused_back_supported(m, (int)S);
    Arena ar = {(char *)scratch, scratch_len, 0};
    char *sp = (char *)ar.take(B * d_bs);
    pgb_vec_znx d = mk(sp, n, cols, rs);
    const pgb_vec_znx *f = in.f;
    uint64_t f_bs = in.f_bs;
    // the copy of f the difference kernel writes: into res on the FFT64 fused route; with leaf pairs into scratch on the other routes,
    // and steps 4-5 read f from it (limbs past res.size are never added)
    char *fr = fuse_fft ? (char *)res->data : in.lv ? (char *)ar.take(B * d_bs) : in.gv ? in.gv->fr : nullptr;
    const uint64_t fr_bs = fuse_fft ? res_bs : d_bs;
    pgb_vec_znx flin;
    if (in.lv) {
        PGB_REQUIRE(fr, "glwe_cmux_tree: scratch exhausted");
        flin = mk(fr, n, cols, umin64(in.f->size, rs));
    }
    if (in.gv) flin = mk(fr, n, cols, f_size);
    if (in.lv || in.gv) {
        f = &flin;
        f_bs = fr_bs;
    }
    PGB_TRY(launch_diff(m, sp, d_bs, rs, in, fr, fr ? fr_bs : 0, base2k, B));

    if (ggsw_stride == 0) { // one selector for the batch: the external product with every route it has
        pgb_batch bte = {B, res_bs, d_bs, 0};
        PGB_TRY(pgb_glwe_external_product_batched(m, res, base2k, &d, base2k, s, ggsw_base2k, dsize, &bte, ar.rest(), ar.rest_len()));
        return add_f_normalize(m, res, res_bs, f, f_bs, base2k, B);
    }

    const uint64_t R = umin64(s->rows * cols, cols * rs); // rows of the vector-matrix product (external_product/glwe.rs:231)
    const uint64_t a_dft_bs = n * cols * rs * pb, res_dft_bs = n * cols * S * pb;
    if (fuse_ntt) {
        char *a_dft = (char *)ar.take(B * a_dft_bs);
        LimbSet li = {sp, n * 8, d_bs}, lo = {a_dft, n * pb, a_dft_bs}; // polys (limb, column) are consecutive on both sides
        PGB_TRY(ntt120_forward(m, li, lo, (int)(rs * cols), (int)B));
        return ntt120_fused_back(m, a_dft, a_dft_bs, (const char *)s->data, (int)R, (int)(cols * S), (int)cols, (const char *)f->data, f_bs,
                                 cols * n * 8, (int)f->size, (char *)res->data, res_bs, cols * n * 8, (int)rs, (int)base2k, 0, (int)B,
                                 nullptr, 0, 0, nullptr, false, false, true, ggsw_stride, sel_div);
    }
    if (fuse_fft) {
        char *res_dft = (char *)ar.take(B * res_dft_bs), *a_dft = (char *)ar.take(B * a_dft_bs);
        LimbSet li = {sp, n * 8, d_bs}, lo = {a_dft, n * pb, a_dft_bs};
        PGB_TRY(fft64_forward(m, li, lo, (int)(rs * cols), (int)B));
        pgb_vec_znx_dft rd = {res_dft, n, cols, S, S}, ad = {a_dft, n, cols, rs, rs};
        pgb_batch btv = {B, res_dft_bs, a_dft_bs, ggsw_stride};
        PGB_TRY(vmp_apply_impl(m, &rd, &ad, s, 0, &btv, sel_div));
        return fft64_fused_back(m, res_dft, res_dft_bs, (int)cols, (int)S, (char *)res->data, res_bs, (int)rs, (int)base2k, (int)B);
    }

    // ---- limb-wise: the external product's HAL sequence with the per-item matrix stride -----------------------------------------------
    pgb_vec_znx_dft res_dft = mk(ar.take(B * res_dft_bs), n, cols, S);
    pgb_vec_znx ain; // the input in ggsw_base2k, as the external product does
    uint64_t ain_bs;
    PGB_TRY(glwe_to_base2k(m, ar, &d, d_bs, base2k, ggsw_base2k, B, &ain, &ain_bs));
    const uint64_t a_dft_max = div_ceil64(ain.size, dsize);
    pgb_vec_znx_dft a_dft = mk(ar.take(B * n * cols * a_dft_max * pb), n, cols, a_dft_max);
    void *tmp = dsize > 1 ? ar.take(B * res_dft_bs) : nullptr;
    PGB_REQUIRE(res_dft.data && ain.data && a_dft.data && (dsize == 1 || tmp), "glwe_cmux: scratch exhausted");
    PGB_TRY(external_product_limbwise(m, res, res_bs, base2k, &ain, ain_bs, s, ggsw_stride, sel_div, ggsw_base2k, dsize, B, &res_dft,
                                      &a_dft, tmp));
    return add_f_normalize(m, res, res_bs, f, f_bs, base2k, B);
}

// the checks the CMux and the blind rotation share: the batch, the selector's shape and ggsw_stride, res and the scratch pointer; returns
// the bytes of one prepared GGSW in *s_item
static int check_common(const char *who, pgb_module *m, const pgb_vec_znx *res, const pgb_vmp_pmat *s, uint64_t ggsw_stride, uint64_t base2k,
                        uint64_t ggsw_base2k, uint64_t dsize, const pgb_batch *bt, const void *scratch, uint64_t *s_item) {
    PGB_REQUIRE(bt && bt->count >= 1 && bt->count <= 65535, "%s: batch count must be in [1, 65535]", who);
    PGB_REQUIRE(res && s && s->data, "%s: null argument", who);
    PGB_REQUIRE(s->n == m->n, "%s: the selector has ring degree %llu, the module %llu", who, (unsigned long long)s->n, (unsigned long long)m->n);
    PGB_REQUIRE(s->cols_in == s->cols_out && s->cols_in >= 1 && s->rows >= 1 && s->size >= 1,
                "%s: the selector must be a non-empty VmpPMat(dnum, k + 1, k + 1, size)", who);
    PGB_TRY(check_glwe(who, "res", m, res, s->cols_in, bt->stride_res, bt->count, false));
    PGB_REQUIRE(res->size >= 1, "%s: res must have at least one limb", who);
    PGB_REQUIRE(dsize >= 1, "%s: dsize must be >= 1", who);
    PGB_REQUIRE(base2k >= 1 && base2k <= 63 && ggsw_base2k >= 1 && ggsw_base2k <= 63, "%s: base2k and ggsw_base2k must be in [1, 63]", who);
    *s_item = pgb_bytes_of_vmp_pmat(m, s->rows, s->cols_in, s->cols_in, s->size);
    PGB_REQUIRE((uintptr_t)s->data % 16 == 0 && (ggsw_stride == 0 || (ggsw_stride % 16 == 0 && ggsw_stride >= *s_item)),
                "%s: selector data must be 16-byte aligned and ggsw_stride 0 or a multiple of 16 of at least one prepared GGSW (%llu bytes)", who,
                (unsigned long long)*s_item);
    PGB_REQUIRE(scratch != nullptr && (uintptr_t)scratch % 256 == 0, "%s: scratch must be non-null and 256-byte aligned", who);
    return PGB_OK;
}

extern "C" int pgb_glwe_cmux_batched(pgb_module *m, pgb_vec_znx *res, const pgb_vec_znx *t, const pgb_vec_znx *f, uint64_t base2k,
                                     const pgb_vmp_pmat *s, uint64_t ggsw_stride, uint64_t ggsw_base2k, uint64_t dsize, const pgb_batch *bt,
                                     void *scratch, size_t scratch_len) {
    uint64_t s_item;
    PGB_REQUIRE(t && f, "glwe_cmux: null argument");
    PGB_TRY(check_common("glwe_cmux", m, res, s, ggsw_stride, base2k, ggsw_base2k, dsize, bt, scratch, &s_item));
    const uint64_t B = bt->count, n = m->n, cols = s->cols_in;
    PGB_TRY(check_glwe("glwe_cmux", "t", m, t, cols, bt->stride_a, B, true));
    PGB_TRY(check_glwe("glwe_cmux", "f", m, f, cols, bt->stride_b, B, true));
    const uint64_t need = pgb_glwe_cmux_tmp_bytes(m, res->size, t->size, f->size, base2k, s, ggsw_base2k, dsize, B);
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
    const CmuxIn in = {t, bt->stride_a, 0, f, bt->stride_b, nullptr};
    return cmux_launch(m, res, bt->stride_res, in, base2k, s, ggsw_stride, 1, ggsw_base2k, dsize, B, scratch, scratch_len);
}

// ---- blind rotation by GGSW bits: acc <- cmux(X^(step 2^i) acc, acc, s_{b,i}) for i < n_bits -------------------------------------------
extern "C" size_t pgb_glwe_blind_rotate_ggsw_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t base2k,
                                                       const pgb_vmp_pmat *s, uint64_t ggsw_base2k, uint64_t dsize, uint64_t n_bits,
                                                       uint64_t batch) {
    (void)a_size;
    // the ping-pong accumulator (res.size limbs; none for one bit) | the CMux's scratch for res.size-limb operands
    const uint64_t acc = n_bits > 1 ? align_up(batch * m->n * s->cols_in * res_size * 8) : 0;
    return acc + pgb_glwe_cmux_tmp_bytes(m, res_size, res_size, res_size, base2k, s, ggsw_base2k, dsize, batch);
}

// Bit i runs cmux_launch with t = X^(p_i) acc_i read in place by the difference kernel and f = acc_i, so each bit launches exactly what one
// CMux of that shape launches.  The accumulator alternates between res and one GLWE batch at the head of the scratch, with the parity that
// makes bit n_bits - 1 write res: no copy.
extern "C" int pgb_glwe_blind_rotate_ggsw_batched(pgb_module *m, pgb_vec_znx *res, const pgb_vec_znx *a, uint64_t base2k, int64_t step,
                                                  uint64_t n_bits, const pgb_vmp_pmat *s, uint64_t ggsw_stride, uint64_t bit_stride,
                                                  uint64_t ggsw_base2k, uint64_t dsize, const pgb_batch *bt, void *scratch, size_t scratch_len) {
    uint64_t s_item;
    PGB_REQUIRE(a, "glwe_blind_rotate_ggsw: null argument");
    PGB_TRY(check_common("glwe_blind_rotate_ggsw", m, res, s, ggsw_stride, base2k, ggsw_base2k, dsize, bt, scratch, &s_item));
    const uint64_t B = bt->count, n = m->n, cols = s->cols_in, rs = res->size;
    PGB_TRY(check_glwe("glwe_blind_rotate_ggsw", "a", m, a, cols, bt->stride_a, B, true));
    PGB_REQUIRE(bt->stride_b == 0, "glwe_blind_rotate_ggsw: stride_b must be 0");
    PGB_REQUIRE(n_bits >= 1 && n_bits <= 64, "glwe_blind_rotate_ggsw: n_bits must be in [1, 64]");
    PGB_REQUIRE(n_bits == 1 || (bit_stride % 16 == 0 && bit_stride >= s_item),
                "glwe_blind_rotate_ggsw: bit_stride %llu must be a multiple of 16 of at least one prepared GGSW (%llu bytes)",
                (unsigned long long)bit_stride, (unsigned long long)s_item);
    // every selector (b, i) lies in [s, s + s_ext): computed in 128 bits, so a stride that wraps the address space is rejected
    const unsigned __int128 s_ext128 = (unsigned __int128)(B - 1) * ggsw_stride + (unsigned __int128)(n_bits - 1) * bit_stride + s_item;
    PGB_REQUIRE(s_ext128 <= (unsigned __int128)(UINTPTR_MAX - (uintptr_t)s->data),
                "glwe_blind_rotate_ggsw: the selectors extend past the end of the address space");
    const uint64_t s_ext = (uint64_t)s_ext128;
    const uint64_t need = pgb_glwe_blind_rotate_ggsw_tmp_bytes(m, rs, a->size, base2k, s, ggsw_base2k, dsize, n_bits, B);
    if (scratch_len < need) {
        pgb_set_error("glwe_blind_rotate_ggsw: scratch of %zu bytes < required %llu", scratch_len, (unsigned long long)need);
        return PGB_ERR_SCRATCH;
    }
    const uint64_t res_ext = batch_extent(n * cols * rs * 8, bt->stride_res, B), a_ext = batch_extent(n * cols * a->size * 8, bt->stride_a, B);
    if (ranges_overlap(res->data, res_ext, a->data, a_ext) || ranges_overlap(res->data, res_ext, s->data, s_ext)) {
        pgb_set_error("glwe_blind_rotate_ggsw: res must not overlap a or a selector");
        return PGB_ERR_ALIAS;
    }
    if (ranges_overlap(scratch, scratch_len, res->data, res_ext) || ranges_overlap(scratch, scratch_len, a->data, a_ext) ||
        ranges_overlap(scratch, scratch_len, s->data, s_ext)) {
        pgb_set_error("glwe_blind_rotate_ggsw: scratch must not overlap res, a or a selector");
        return PGB_ERR_ALIAS;
    }

    const uint64_t acc_bs = n * cols * rs * 8, mask = 2 * n - 1;
    Arena ar = {(char *)scratch, scratch_len, 0};
    pgb_vec_znx acc[2] = {*res, mk(n_bits > 1 ? ar.take(B * acc_bs) : nullptr, n, cols, rs)};
    const uint64_t acc_stride[2] = {bt->stride_res, acc_bs};
    const pgb_vec_znx *cur = a;
    uint64_t cur_bs = bt->stride_a;
    for (uint64_t i = 0; i < n_bits; i++) {
        const int w = (int)((n_bits - 1 - i) & 1); // 0: res
        const uint32_t rot = (uint32_t)(((uint64_t)step << i) & mask);
        pgb_vmp_pmat si = *s;
        si.data = (char *)s->data + i * bit_stride;
        const CmuxIn in = {cur, cur_bs, rot, cur, cur_bs, nullptr};
        PGB_TRY(cmux_launch(m, &acc[w], acc_stride[w], in, base2k, &si, ggsw_stride, 1, ggsw_base2k, dsize, B, ar.rest(), ar.rest_len()));
        cur = &acc[w];
        cur_bs = acc_stride[w];
    }
    return PGB_OK;
}

// ---- CMux tree: g_{0,j} = leaf j, g_{i+1,j} = cmux(g_{i,2j+1}, g_{i,2j}, s_{b,i}) for i < n_bits, res = g_{n_bits,0} ----------------------
// Chunks of whole items run the whole tree; no level of a chunk of Bc items launches more than Bc 2^(n_bits-1) <= 65535 grid items.
static uint64_t tree_chunk_cap(uint64_t n_bits) { return 65535 >> (n_bits - 1); }

extern "C" size_t pgb_glwe_cmux_tree_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t base2k,
                                               const pgb_vmp_pmat *s, uint64_t ggsw_base2k, uint64_t dsize, uint64_t n_bits, uint64_t batch) {
    (void)a_size;
    if (n_bits < 1 || n_bits > 16) return 0;
    const uint64_t Bc = umin64(batch, tree_chunk_cap(n_bits)), g = m->n * s->cols_in * res_size * 8, P0 = Bc << (n_bits - 1);
    // the level-1 and level-2 outputs (the last level writes res) | level 0's CMux scratch and its linear copy of f (the later levels run
    // fewer CMuxes of the same shape in the same space)
    const uint64_t lv1 = n_bits > 1 ? align_up(P0 * g) : 0, lv2 = n_bits > 2 ? align_up((P0 >> 1) * g) : 0;
    return lv1 + lv2 + align_up(P0 * g) + pgb_glwe_cmux_tmp_bytes(m, res_size, res_size, res_size, base2k, s, ggsw_base2k, dsize, P0);
}

// Level i of a chunk is one cmux_launch over its Bc 2^(n_bits-1-i) CMuxes, q = b 2^lp + j (lp = n_bits - 1 - i): item b's outputs are
// consecutive, so the next level reads t = g_{i,2j+1} and f = g_{i,2j} at stride 2g from the buffer base + g and base, and the selector of
// CMux q is item q >> lp's (sel_div = 2^lp).  Level 0 reads the leaves through the difference kernel's DIFF_LEAF instance.
extern "C" int pgb_glwe_cmux_tree_batched(pgb_module *m, pgb_vec_znx *res, const pgb_vec_znx *a, uint64_t entry_stride, uint64_t base2k,
                                          uint64_t n_bits, const pgb_vmp_pmat *s, uint64_t ggsw_stride, uint64_t bit_stride,
                                          uint64_t ggsw_base2k, uint64_t dsize, const pgb_batch *bt, void *scratch, size_t scratch_len) {
    static const char *who = "glwe_cmux_tree";
    uint64_t s_item;
    PGB_REQUIRE(a, "%s: null argument", who);
    PGB_TRY(check_common(who, m, res, s, ggsw_stride, base2k, ggsw_base2k, dsize, bt, scratch, &s_item));
    const uint64_t B = bt->count, n = m->n, cols = s->cols_in, rs = res->size;
    PGB_TRY(check_glwe(who, "a", m, a, cols, bt->stride_a, B, true));
    PGB_REQUIRE(bt->stride_b == 0, "%s: stride_b must be 0", who);
    PGB_REQUIRE(n_bits >= 1 && n_bits <= 16, "%s: n_bits must be in [1, 16]", who);
    const uint64_t a_item = n * cols * a->size * 8;
    PGB_REQUIRE(entry_stride % 16 == 0 && entry_stride >= a_item,
                "%s: entry_stride %llu must be a multiple of 16 of at least one GLWE of a.size limbs (%llu bytes)", who,
                (unsigned long long)entry_stride, (unsigned long long)a_item);
    PGB_REQUIRE(n_bits == 1 || (bit_stride % 16 == 0 && bit_stride >= s_item),
                "%s: bit_stride %llu must be a multiple of 16 of at least one prepared GGSW (%llu bytes)", who, (unsigned long long)bit_stride,
                (unsigned long long)s_item);
    // every leaf (b, j) and selector (b, i) lies in [a, a + a_ext) and [s, s + s_ext): computed in 128 bits, so a stride that wraps the
    // address space is rejected
    const unsigned __int128 a_ext128 = (unsigned __int128)(B - 1) * bt->stride_a + (unsigned __int128)((1ull << n_bits) - 1) * entry_stride + a_item;
    const unsigned __int128 s_ext128 = (unsigned __int128)(B - 1) * ggsw_stride + (unsigned __int128)(n_bits - 1) * bit_stride + s_item;
    PGB_REQUIRE(a_ext128 <= (unsigned __int128)(UINTPTR_MAX - (uintptr_t)a->data), "%s: the table extends past the end of the address space",
                who);
    PGB_REQUIRE(s_ext128 <= (unsigned __int128)(UINTPTR_MAX - (uintptr_t)s->data),
                "%s: the selectors extend past the end of the address space", who);
    const uint64_t a_ext = (uint64_t)a_ext128, s_ext = (uint64_t)s_ext128;
    // the largest chunk of whole items whose scratch fits
    uint64_t lo = 1, hi = umin64(B, tree_chunk_cap(n_bits));
    if (scratch_len < pgb_glwe_cmux_tree_tmp_bytes(m, rs, a->size, base2k, s, ggsw_base2k, dsize, n_bits, 1)) {
        pgb_set_error("%s: scratch of %zu bytes < required %llu for one item", who, scratch_len,
                      (unsigned long long)pgb_glwe_cmux_tree_tmp_bytes(m, rs, a->size, base2k, s, ggsw_base2k, dsize, n_bits, 1));
        return PGB_ERR_SCRATCH;
    }
    while (lo < hi) {
        const uint64_t mid = (lo + hi + 1) / 2;
        if (pgb_glwe_cmux_tree_tmp_bytes(m, rs, a->size, base2k, s, ggsw_base2k, dsize, n_bits, mid) <= scratch_len) lo = mid;
        else hi = mid - 1;
    }
    const uint64_t Bc = lo;
    const uint64_t res_ext = batch_extent(n * cols * rs * 8, bt->stride_res, B);
    if (ranges_overlap(res->data, res_ext, a->data, a_ext) || ranges_overlap(res->data, res_ext, s->data, s_ext)) {
        pgb_set_error("%s: res must not overlap the table or a selector", who);
        return PGB_ERR_ALIAS;
    }
    if (ranges_overlap(scratch, scratch_len, res->data, res_ext) || ranges_overlap(scratch, scratch_len, a->data, a_ext) ||
        ranges_overlap(scratch, scratch_len, s->data, s_ext)) {
        pgb_set_error("%s: scratch must not overlap res, the table or a selector", who);
        return PGB_ERR_ALIAS;
    }

    const uint64_t g = n * cols * rs * 8, P0 = Bc << (n_bits - 1);
    Arena ar = {(char *)scratch, scratch_len, 0};
    pgb_vec_znx lvl[2] = {mk(n_bits > 1 ? ar.take(P0 * g) : nullptr, n, cols, rs), mk(n_bits > 2 ? ar.take((P0 >> 1) * g) : nullptr, n, cols, rs)};
    for (uint64_t b0 = 0; b0 < B; b0 += Bc) {
        const uint64_t nb = umin64(Bc, B - b0);
        pgb_vec_znx ab = *a, out_res = *res;
        ab.data = (char *)a->data + b0 * bt->stride_a;
        out_res.data = (char *)res->data + b0 * bt->stride_res;
        for (uint64_t i = 0; i < n_bits; i++) {
            const uint32_t lp = (uint32_t)(n_bits - 1 - i);
            pgb_vmp_pmat si = *s;
            si.data = (char *)s->data + b0 * ggsw_stride + i * bit_stride;
            const LeafPairs lv = {&ab, bt->stride_a, entry_stride, lp};
            pgb_vec_znx tin = lvl[(i + 1) & 1];  // g_i (i >= 1): level i's output buffer is lvl[i & 1], so g_i is in lvl[(i - 1) & 1]
            tin.data = (char *)tin.data + g;
            const CmuxIn in = i == 0 ? CmuxIn{&ab, 0, 0, &ab, 0, &lv} : CmuxIn{&tin, 2 * g, 0, &lvl[(i + 1) & 1], 2 * g, nullptr};
            pgb_vec_znx *out = i + 1 == n_bits ? &out_res : &lvl[i & 1];
            const uint64_t out_bs = i + 1 == n_bits ? bt->stride_res : g;
            PGB_TRY(cmux_launch(m, out, out_bs, in, base2k, &si, ggsw_stride, 1u << lp, ggsw_base2k, dsize, nb << lp, ar.rest(), ar.rest_len()));
        }
    }
    return PGB_OK;
}

// ---- binary decision diagram: state n_leaves + k = cmux(state[node_t[k]], state[node_f[k]], s_{b, level_bit[i]}) ----------------------
// One chunk of Bc items runs every level as one cmux_launch over its Bc * P_i CMuxes (q = b P_i + j, selector divisor P_i); node j of
// level L keeps its Bc outputs in level L's block at + (b P_L + j) * g, so every child is an affine pair (base + j g, per-item stride P_L g)
// or a leaf (a + b stride_a + j entry_stride).  The descriptors of all nodes and outputs form one table, uploaded once per call to the
// head of the scratch; a last launch per chunk copies the outputs.  Blocks are not reused between levels.
__global__ void __launch_bounds__(256) bdd_output_kernel(const GatherSrc *desc, const char *leaf, const char *state, char *res,
                                                         uint64_t res_bs, uint64_t out_stride, uint32_t words, uint32_t n_out, int size) {
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= words) return;
    const size_t b = blockIdx.y;
    for (uint32_t o = blockIdx.z; o < n_out; o += gridDim.z) {
        const GatherSrc g = desc[o];
        const long long *src = reinterpret_cast<const long long *>((g.src ? state : leaf) + g.off + b * g.bs) + u;
        long long *dst = reinterpret_cast<long long *>(res + b * res_bs + o * out_stride) + u;
        for (int j = 0; j < size; j++) dst[(size_t)j * words] = j < (int)g.size ? __ldg(src + (size_t)j * words) : 0;
    }
}

// the circuit's level widths: the total and the widest (1 without levels); false when a width is outside [1, 65535] or an array is null
static bool bdd_widths(const pgb_bdd_circuit *c, uint64_t *nodes, uint64_t *widest) {
    *nodes = 0;
    *widest = 1;
    if (!c || (c->n_levels && (!c->level_count || !c->level_bit))) return false;
    for (uint64_t i = 0; i < c->n_levels; i++) {
        const uint64_t w = c->level_count[i];
        if (w < 1 || w > 65535) return false;
        *nodes += w;
        *widest = w > *widest ? w : *widest;
    }
    return true;
}

static uint64_t bdd_table_bytes(uint64_t nodes, uint64_t n_out) { return nodes * sizeof(GatherNode) + n_out * sizeof(GatherSrc); }

extern "C" size_t pgb_glwe_bdd_eval_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t base2k,
                                              const pgb_vmp_pmat *s, uint64_t ggsw_base2k, uint64_t dsize, const pgb_bdd_circuit *c,
                                              uint64_t batch) {
    (void)a_size;
    uint64_t nodes, widest;
    if (!bdd_widths(c, &nodes, &widest)) return 0;
    const uint64_t Bc = umin64(batch, 65535 / widest), g = m->n * s->cols_in * res_size * 8;
    // the descriptor table | one block of Bc P_i GLWEs per level | the linear copy of f and one CMux's scratch, for the widest level
    uint64_t bytes = align_up(bdd_table_bytes(nodes, c->n_out));
    for (uint64_t i = 0; i < c->n_levels; i++) bytes += align_up(Bc * c->level_count[i] * g);
    if (c->n_levels)
        bytes += align_up(Bc * widest * g) + pgb_glwe_cmux_tmp_bytes(m, res_size, res_size, res_size, base2k, s, ggsw_base2k, dsize, Bc * widest);
    return bytes;
}

extern "C" int pgb_glwe_bdd_eval_batched(pgb_module *m, pgb_vec_znx *res, uint64_t out_stride, const pgb_vec_znx *a, uint64_t entry_stride,
                                         uint64_t base2k, uint64_t n_bits, const pgb_vmp_pmat *s, uint64_t ggsw_stride, uint64_t bit_stride,
                                         uint64_t ggsw_base2k, uint64_t dsize, const pgb_bdd_circuit *c, const pgb_batch *bt, void *scratch,
                                         size_t scratch_len) {
    static const char *who = "glwe_bdd_eval";
    uint64_t s_item;
    PGB_REQUIRE(a && c, "%s: null argument", who);
    PGB_TRY(check_common(who, m, res, s, ggsw_stride, base2k, ggsw_base2k, dsize, bt, scratch, &s_item));
    const uint64_t B = bt->count, n = m->n, cols = s->cols_in, rs = res->size;
    PGB_TRY(check_glwe(who, "a", m, a, cols, bt->stride_a, B, true));
    PGB_REQUIRE(bt->stride_b == 0, "%s: stride_b must be 0", who);
    PGB_REQUIRE(n_bits >= 1 && n_bits <= 64, "%s: n_bits must be in [1, 64]", who);
    // ---- the circuit, from the host arrays ----
    uint64_t nodes, widest;
    PGB_REQUIRE(bdd_widths(c, &nodes, &widest), "%s: every level needs a width in [1, 65535] (and non-null level arrays)", who);
    PGB_REQUIRE(nodes == 0 || (c->node_t && c->node_f), "%s: null node arrays", who);
    PGB_REQUIRE(c->n_out >= 1 && c->outputs, "%s: the circuit needs at least one output", who);
    const uint64_t states = c->n_leaves + nodes;
    uint64_t max_bit = 0;
    for (uint64_t i = 0, k = 0; i < c->n_levels; i++) {
        PGB_REQUIRE(c->level_bit[i] < n_bits, "%s: level %llu selects with bit %u, not below n_bits = %llu", who, (unsigned long long)i,
                    c->level_bit[i], (unsigned long long)n_bits);
        max_bit = c->level_bit[i] > max_bit ? c->level_bit[i] : max_bit;
        const uint64_t first = c->n_leaves + k; // children must be states below the level's first node
        for (uint64_t e = k + c->level_count[i]; k < e; k++)
            PGB_REQUIRE(c->node_t[k] < first && c->node_f[k] < first,
                        "%s: node %llu of level %llu has a child that is not a leaf or a node of an earlier level", who, (unsigned long long)k,
                        (unsigned long long)i);
    }
    for (uint64_t o = 0; o < c->n_out; o++)
        PGB_REQUIRE(c->outputs[o] < states, "%s: output %llu names state %u of %llu", who, (unsigned long long)o, c->outputs[o],
                    (unsigned long long)states);
    // ---- strides and extents ----
    const uint64_t a_item = n * cols * a->size * 8, g = n * cols * rs * 8;
    PGB_REQUIRE(entry_stride % 16 == 0 && entry_stride >= a_item,
                "%s: entry_stride %llu must be a multiple of 16 of at least one GLWE of a.size limbs (%llu bytes)", who,
                (unsigned long long)entry_stride, (unsigned long long)a_item);
    PGB_REQUIRE(n_bits == 1 || (bit_stride % 16 == 0 && bit_stride >= s_item),
                "%s: bit_stride %llu must be a multiple of 16 of at least one prepared GGSW (%llu bytes)", who, (unsigned long long)bit_stride,
                (unsigned long long)s_item);
    PGB_REQUIRE(c->n_out == 1 || (out_stride % 16 == 0 && out_stride >= g),
                "%s: out_stride %llu must be a multiple of 16 of at least one GLWE of res.size limbs (%llu bytes)", who,
                (unsigned long long)out_stride, (unsigned long long)g);
    const unsigned __int128 item_ext128 = (unsigned __int128)(c->n_out - 1) * out_stride + g; // one item's outputs
    PGB_REQUIRE(B == 1 || bt->stride_res >= item_ext128, "%s: stride_res %llu must cover the n_out outputs of an item (%llu bytes)", who,
                (unsigned long long)bt->stride_res, (unsigned long long)item_ext128);
    // every leaf (b, j), selector (b, i) and output (b, o) lies in [a, a + a_ext), [s, s + s_ext), [res, res + res_ext): computed in 128
    // bits, so a stride that wraps the address space is rejected
    const unsigned __int128 a_ext128 = (unsigned __int128)(B - 1) * bt->stride_a +
                                       (unsigned __int128)(c->n_leaves ? c->n_leaves - 1 : 0) * entry_stride + a_item;
    const unsigned __int128 s_ext128 = (unsigned __int128)(B - 1) * ggsw_stride + (unsigned __int128)max_bit * bit_stride + s_item;
    const unsigned __int128 res_ext128 = (unsigned __int128)(B - 1) * bt->stride_res + item_ext128;
    PGB_REQUIRE(a_ext128 <= (unsigned __int128)(UINTPTR_MAX - (uintptr_t)a->data), "%s: the leaves extend past the end of the address space",
                who);
    PGB_REQUIRE(s_ext128 <= (unsigned __int128)(UINTPTR_MAX - (uintptr_t)s->data),
                "%s: the selectors extend past the end of the address space", who);
    PGB_REQUIRE(res_ext128 <= (unsigned __int128)(UINTPTR_MAX - (uintptr_t)res->data),
                "%s: the outputs extend past the end of the address space", who);
    const uint64_t a_ext = (uint64_t)a_ext128, s_ext = (uint64_t)s_ext128, res_ext = (uint64_t)res_ext128;
    // ---- the largest chunk of whole items whose scratch fits ----
    const uint64_t need1 = pgb_glwe_bdd_eval_tmp_bytes(m, rs, a->size, base2k, s, ggsw_base2k, dsize, c, 1);
    if (scratch_len < need1) {
        pgb_set_error("%s: scratch of %zu bytes < required %llu for one item", who, scratch_len, (unsigned long long)need1);
        return PGB_ERR_SCRATCH;
    }
    uint64_t lo = 1, hi = umin64(B, 65535 / widest);
    while (lo < hi) {
        const uint64_t mid = (lo + hi + 1) / 2;
        if (pgb_glwe_bdd_eval_tmp_bytes(m, rs, a->size, base2k, s, ggsw_base2k, dsize, c, mid) <= scratch_len) lo = mid;
        else hi = mid - 1;
    }
    const uint64_t Bc = lo;
    if (ranges_overlap(res->data, res_ext, a->data, a_ext) || ranges_overlap(res->data, res_ext, s->data, s_ext)) {
        pgb_set_error("%s: res must not overlap the leaves or a selector", who);
        return PGB_ERR_ALIAS;
    }
    if (ranges_overlap(scratch, scratch_len, res->data, res_ext) || ranges_overlap(scratch, scratch_len, a->data, a_ext) ||
        ranges_overlap(scratch, scratch_len, s->data, s_ext)) {
        pgb_set_error("%s: scratch must not overlap res, the leaves or a selector", who);
        return PGB_ERR_ALIAS;
    }

    // ---- scratch layout and the descriptor table (offsets of nodes relative to the scratch, of leaves to the chunk's leaf base) ----
    Arena ar = {(char *)scratch, scratch_len, 0};
    char *table = (char *)ar.take(bdd_table_bytes(nodes, c->n_out));
    std::vector<uint64_t> block(c->n_levels);
    std::vector<uint64_t> level_of(nodes); // node k -> its level
    for (uint64_t i = 0, k = 0; i < c->n_levels; i++) {
        block[i] = (uint64_t)((char *)ar.take(Bc * c->level_count[i] * g) - (char *)scratch);
        for (uint64_t e = k + c->level_count[i]; k < e; k++) level_of[k] = i;
    }
    std::vector<uint64_t> first(c->n_levels); // state index of each level's first node
    for (uint64_t i = 0, k = c->n_leaves; i < c->n_levels; i++) {
        first[i] = k;
        k += c->level_count[i];
    }
    auto src_of = [&](uint32_t st) -> GatherSrc {
        if (st < c->n_leaves) return GatherSrc{st * entry_stride, bt->stride_a, 0, (uint32_t)a->size};
        const uint64_t L = level_of[st - c->n_leaves];
        return GatherSrc{block[L] + (st - first[L]) * g, c->level_count[L] * g, 1, (uint32_t)rs};
    };
    std::vector<char> host(bdd_table_bytes(nodes, c->n_out));
    GatherNode *hn = reinterpret_cast<GatherNode *>(host.data());
    GatherSrc *ho = reinterpret_cast<GatherSrc *>(host.data() + nodes * sizeof(GatherNode));
    for (uint64_t k = 0; k < nodes; k++) hn[k] = GatherNode{src_of(c->node_t[k]), src_of(c->node_f[k])};
    for (uint64_t o = 0; o < c->n_out; o++) ho[o] = src_of(c->outputs[o]);
    char *fr = c->n_levels ? (char *)ar.take(Bc * widest * g) : nullptr;
    PGB_REQUIRE(table && (c->n_levels == 0 || fr), "%s: scratch exhausted", who);
    PGB_CHECK_CUDA(cudaMemcpyAsync(table, host.data(), host.size(), cudaMemcpyHostToDevice, m->stream));

    const GatherNode *desc = reinterpret_cast<const GatherNode *>(table);
    for (uint64_t b0 = 0; b0 < B; b0 += Bc) {
        const uint64_t nb = umin64(Bc, B - b0);
        const char *leaf = (const char *)a->data + b0 * bt->stride_a;
        for (uint64_t i = 0, k = 0; i < c->n_levels; k += c->level_count[i], i++) {
            const uint32_t P = c->level_count[i];
            bool f_node = false;
            for (uint64_t e = k; e < k + P; e++) f_node |= c->node_f[e] >= c->n_leaves;
            const NodeGather gv = {desc + k, leaf, (const char *)scratch, P, f_node ? rs : umin64(a->size, rs), fr};
            pgb_vmp_pmat si = *s;
            si.data = (char *)s->data + b0 * ggsw_stride + c->level_bit[i] * bit_stride;
            pgb_vec_znx out = mk((char *)scratch + block[i], n, cols, rs);
            const CmuxIn in = {a, 0, 0, a, 0, nullptr, &gv};
            PGB_TRY(cmux_launch(m, &out, g, in, base2k, &si, ggsw_stride, P, ggsw_base2k, dsize, nb * P, ar.rest(), ar.rest_len()));
        }
        const uint32_t words = (uint32_t)(n * cols);
        const dim3 grid((words + 255) / 256, (uint32_t)nb, (uint32_t)umin64(c->n_out, 65535));
        { ProfScope _ps(m, PROF_ELEMENTWISE);
        bdd_output_kernel<<<grid, 256, 0, m->stream>>>(reinterpret_cast<const GatherSrc *>(table + nodes * sizeof(GatherNode)), leaf,
                                                       (const char *)scratch, (char *)res->data + b0 * bt->stride_res, bt->stride_res,
                                                       out_stride, words, (uint32_t)c->n_out, (int)rs);
        }
        PGB_CHECK_CUDA(cudaGetLastError());
    }
    return PGB_OK;
}
