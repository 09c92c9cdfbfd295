// pack.cu -- glwe_pack (poulpy-core/src/glwe_packing.rs:15-170) batched on the device: n_in GLWEs per item become one GLWE whose
// coefficient index[j] carries the constant coefficient of input j.  Round i < log_n - log_gap_out (t = n >> (i + 1)) folds key j + t onto
// key j for every j < t, through one of three cases of pack_internal (glwe_packing.rs:15-96):
//
//     both:    x = normalize(rsh1(X^-t lo - hi)),  y = rsh1(X^-t lo + hi),  z = glwe_automorphism(x),  out = X^t normalize(y - z)
//     lo only: x = rsh1(lo),                       out = glwe_automorphism_add(x)         (op 0: aut(ks(x)) + x)
//     hi only: x = rsh1(X^t hi),                   out = glwe_automorphism_sub_negate(x)  (op 2: x - aut(ks(x)))
//
// then the single state goes through glwe_trace(skip = log_n - log_gap_out) into res.  The host turns `index` into a plan (every state a
// compact slot per round) and a descriptor table uploaded once per call to the head of the scratch.  A round of a chunk is one prep kernel
// over (item, slot), at most three automorphism launches (one per case, each over its case's contiguous block under the round's shared key
// keys[i], through the batched entries the composition calls), and one combine kernel when `both` is present.
#include "internal.h"
#include "znx.cuh"
#include <algorithm>
#include <vector>

enum { PACK_BOTH = 0, PACK_LO = 1, PACK_HI = 2 };
// an operand of every item of a chunk: item b's GLWE at (src ? scratch : the chunk's inputs) + off + b * bs
struct PackSrc { uint64_t off, bs; uint32_t src, pad; };
// slot w of a round: its case, its operands, and where the prep kernel writes x (item b at scratch + x_off + b * x_bs) and, for `both`,
// y (scratch + y_off + b * x_bs)
struct PackSlot { PackSrc lo, hi; uint64_t x_off, x_bs, y_off; uint32_t kind, pad; };

struct PackPrepArgs {
    const PackSlot *desc;  // the round's W slots
    const char *in, *scratch;
    uint32_t words, n, W, t; // words = cols * n per limb; t = n >> (i + 1)
    int size, K;
};

// One thread per (column, coefficient) of slot w = q mod W of item q / W.  The sum is staged in the thread's own words of x (and y), then
// shifted and normalised in place by the same thread with the device code of vec_znx_rsh_assign and vec_znx_normalize_assign; the rotated
// operand is read through rotate_kernel's index and sign and never written.
__global__ void __launch_bounds__(256) pack_prep_kernel(PackPrepArgs p) {
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= p.words) return;
    const uint32_t q = blockIdx.y, b = q / p.W, w = q - b * p.W;
    const PackSlot s = p.desc[w];
    const size_t ls = p.words;
    const uint32_t i = u & (p.n - 1), col0 = u - i;
    long long *x = reinterpret_cast<long long *>(const_cast<char *>(p.scratch) + s.x_off + (size_t)b * s.x_bs) + u;
    auto X = [&](int j) -> long long & { return x[(size_t)j * ls]; };
    auto at = [&](const PackSrc &g) { return reinterpret_cast<const long long *>((g.src ? p.scratch : p.in) + g.off + (size_t)b * g.bs); };
    if (s.kind == PACK_LO) {
        const long long *lo = at(s.lo) + u;
        for (int j = 0; j < p.size; j++) X(j) = __ldg(lo + (size_t)j * ls);
        rsh_assign_coeff(X, p.size, p.K, 1);
    } else if (s.kind == PACK_HI) {
        bool neg;
        const long long *hi = at(s.hi) + col0 + rotate_src(i, (long long)p.t, p.n, &neg);
        for (int j = 0; j < p.size; j++) {
            const long long v = __ldg(hi + (size_t)j * ls);
            X(j) = neg ? (long long)(0ull - (unsigned long long)v) : v;
        }
        rsh_assign_coeff(X, p.size, p.K, 1);
    } else {
        bool neg;
        const long long *lo = at(s.lo) + col0 + rotate_src(i, -(long long)p.t, p.n, &neg), *hi = at(s.hi) + u;
        long long *y = reinterpret_cast<long long *>(const_cast<char *>(p.scratch) + s.y_off + (size_t)b * s.x_bs) + u;
        auto Y = [&](int j) -> long long & { return y[(size_t)j * ls]; };
        for (int j = 0; j < p.size; j++) {
            const long long lv = __ldg(lo + (size_t)j * ls), hv = __ldg(hi + (size_t)j * ls);
            const unsigned long long l = neg ? 0ull - (unsigned long long)lv : (unsigned long long)lv;
            X(j) = (long long)(l - (unsigned long long)hv);
            Y(j) = (long long)(l + (unsigned long long)hv);
        }
        rsh_assign_coeff(X, p.size, p.K, 1);
        normalize_coeff(X, [&](int j, long long v) { X(j) = v; }, p.size, p.K);
        rsh_assign_coeff(Y, p.size, p.K, 1);
    }
}

// out = X^t normalize(y - z) for `both` slot q (item-major, q = b * nb + s): one thread per destination (column, coefficient), which
// runs the carry chain of its source coefficient and writes each limb with the rotation's sign
struct PackCombineArgs {
    const char *y, *z; uint64_t g; // y and z of pair q at + q * g
    char *out; uint64_t out_bs;    // out of pair q at + q * out_bs
    uint32_t words, n, t;
    int size, K;
};
__global__ void __launch_bounds__(256) pack_combine_kernel(PackCombineArgs p) {
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= p.words) return;
    const size_t q = blockIdx.y, ls = p.words;
    const uint32_t i = u & (p.n - 1);
    bool neg;
    const uint32_t su = u - i + rotate_src(i, (long long)p.t, p.n, &neg);
    const long long *y = reinterpret_cast<const long long *>(p.y + q * p.g) + su, *z = reinterpret_cast<const long long *>(p.z + q * p.g) + su;
    long long *out = reinterpret_cast<long long *>(p.out + q * p.out_bs) + u;
    normalize_coeff([&](int j) { return (long long)((unsigned long long)__ldg(y + (size_t)j * ls) - (unsigned long long)__ldg(z + (size_t)j * ls)); },
                    [&](int j, long long v) { out[(size_t)j * ls] = neg ? (long long)(0ull - (unsigned long long)v) : v; }, p.size, p.K);
}

// the state of a packing without rounds (log_gap_out = log_n, one input at index 0) copied into res with 16-byte words, for inputs whose
// item stride is below one GLWE (0: shared by the batch)
__global__ void __launch_bounds__(256) pack_copy_kernel(const char *a, uint64_t a_bs, char *res, uint64_t res_bs, uint32_t words) {
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= words) return;
    const size_t b = blockIdx.y;
    reinterpret_cast<uint4 *>(res + b * res_bs)[u] = __ldg(reinterpret_cast<const uint4 *>(a + b * a_bs) + u);
}

// ---- the plan --------------------------------------------------------------------------------------------------------------------------
// Round i's slots in the order both, lo only, hi only (slot w = case_off[case] + s); a state is an input (round -1, slot j) or slot w of
// round i.  Slot w's x, and its output when round i is not the last, sit in blocks of Bc W_i GLWEs laid out per case: case c's block at
// case_off[c] * Bc GLWEs, item b's slot s at + b * n_c + s, so each case is one contiguous batch of nb * n_c GLWEs for the automorphism.
struct PackRef { int64_t round; uint32_t w; };
struct PackRound { uint32_t nb = 0, nl = 0, nh = 0; std::vector<PackRef> lo, hi; uint32_t width() const { return nb + nl + nh; } };
struct PackPlan {
    std::vector<PackRound> rounds;
    uint32_t widest = 1, max_nb = 0, max_op = 0; // widest round (1 without rounds), most `both` / lo-or-hi slots of a round
    uint64_t slots = 0;
};

// false when an index is out of range, repeated, or not a multiple of 2^log_gap_out (such an input cannot reach coefficient index[j])
static bool pack_plan(uint64_t n, int log_n, const uint32_t *index, uint64_t n_in, uint64_t log_gap_out, PackPlan *plan) {
    std::vector<PackRef> cur(n, PackRef{-2, 0}); // key -> state (round -2: none)
    for (uint64_t j = 0; j < n_in; j++) {
        const uint64_t k = index[j];
        if (k >= n || cur[k].round != -2 || (k & ((1ull << log_gap_out) - 1))) return false;
        cur[k] = PackRef{-1, (uint32_t)j};
    }
    const uint64_t R = (uint64_t)log_n - log_gap_out;
    plan->rounds.assign(R, PackRound());
    for (uint64_t i = 0; i < R; i++) {
        const uint64_t t = n >> (i + 1);
        PackRound &r = plan->rounds[i];
        std::vector<uint64_t> kb, kl, kh; // the keys of each case, in key order
        for (uint64_t j = 0; j < t; j++) {
            const bool l = cur[j].round != -2, h = cur[j + t].round != -2;
            if (l && h) kb.push_back(j);
            else if (l) kl.push_back(j);
            else if (h) kh.push_back(j);
        }
        r.nb = (uint32_t)kb.size();
        r.nl = (uint32_t)kl.size();
        r.nh = (uint32_t)kh.size();
        std::vector<PackRef> next(t, PackRef{-2, 0});
        uint32_t w = 0;
        for (uint64_t j : kb) { r.lo.push_back(cur[j]); r.hi.push_back(cur[j + t]); next[j] = PackRef{(int64_t)i, w++}; }
        for (uint64_t j : kl) { r.lo.push_back(cur[j]); r.hi.push_back(PackRef{-2, 0}); next[j] = PackRef{(int64_t)i, w++}; }
        for (uint64_t j : kh) { r.lo.push_back(PackRef{-2, 0}); r.hi.push_back(cur[j + t]); next[j] = PackRef{(int64_t)i, w++}; }
        cur.assign(n, PackRef{-2, 0});
        for (uint64_t j = 0; j < t; j++) cur[j] = next[j];
        plan->widest = i == 0 ? r.width() : plan->widest;
        plan->max_nb = r.nb > plan->max_nb ? r.nb : plan->max_nb;
        plan->max_op = r.nl > plan->max_op ? r.nl : plan->max_op;
        plan->max_op = r.nh > plan->max_op ? r.nh : plan->max_op;
        plan->slots += r.width();
    }
    return true;
}

// the scratch of a chunk of Bc items: the descriptor table | two ping-pong state blocks of Bc * widest GLWEs (round i writes its outputs
// to block i & 1 and its z to block (i + 1) & 1, whose states the prep kernel has consumed) | x (Bc * widest GLWEs) | y (Bc * max_nb GLWEs)
// | the scratch of the automorphism and trace calls.  Offsets from the scratch base in *lay when lay is set.
struct PackLayout { uint64_t table, blk[2], x, y, rest; };
static uint64_t pack_bytes(const pgb_module *m, uint64_t size, uint64_t base2k, const pgb_vmp_pmat *key, uint64_t dsize, uint64_t log_gap_out,
                           const PackPlan &plan, uint64_t Bc, PackLayout *lay) {
    const uint64_t g = m->n * key->cols_out * size * 8, R = plan.rounds.size();
    PackLayout l = {};
    uint64_t off = align_up(plan.slots * sizeof(PackSlot));
    if (R) {
        l.blk[0] = off;
        off += align_up(Bc * plan.widest * g);
        l.blk[1] = off;
        off += align_up(Bc * plan.widest * g);
        l.x = off;
        off += align_up(Bc * plan.widest * g);
        l.y = off;
        off += align_up(Bc * plan.max_nb * g);
    }
    l.rest = off;
    uint64_t rest = 0;
    if (plan.max_nb) rest = pgb_glwe_automorphism_tmp_bytes(m, size, size, base2k, key, base2k, dsize, Bc * plan.max_nb);
    if (plan.max_op) rest = std::max<uint64_t>(rest, pgb_glwe_automorphism_add_assign_tmp_bytes(m, size, base2k, key, base2k, dsize, Bc * plan.max_op));
    if (log_gap_out) rest = std::max<uint64_t>(rest, pgb_glwe_trace_assign_tmp_bytes(m, size, base2k, key, base2k, dsize, Bc));
    if (lay) *lay = l;
    return off + rest;
}

static uint64_t pack_chunk_cap(const PackPlan &plan) { return 65535 / plan.widest; }

extern "C" size_t pgb_glwe_pack_tmp_bytes(const pgb_module *m, uint64_t size, uint64_t base2k, const pgb_vmp_pmat *key, uint64_t dsize,
                                          const uint32_t *index, uint64_t n_in, uint64_t log_gap_out, uint64_t batch) {
    PackPlan plan;
    if (!m || !key || !index || n_in < 1 || n_in > m->n || log_gap_out > (uint64_t)m->log_n || batch < 1) return 0;
    if (!pack_plan(m->n, m->log_n, index, n_in, log_gap_out, &plan)) return 0;
    return pack_bytes(m, size, base2k, key, dsize, log_gap_out, plan, umin64(batch, pack_chunk_cap(plan)), nullptr);
}

extern "C" int pgb_glwe_pack_batched(pgb_module *m, pgb_vec_znx *res, const pgb_vec_znx *a, uint64_t entry_stride, const uint32_t *index,
                                     uint64_t n_in, uint64_t log_gap_out, uint64_t base2k, const pgb_vmp_pmat *keys, uint64_t nkeys,
                                     uint64_t dsize, const pgb_batch *bt, void *scratch, size_t scratch_len) {
    static const char *who = "glwe_pack";
    PGB_REQUIRE(m && res && a && index && keys && bt, "%s: null argument", who);
    PGB_REQUIRE(bt->count >= 1 && bt->count <= 65535, "%s: batch count must be in [1, 65535]", who);
    const uint64_t n = m->n, log_n = (uint64_t)m->log_n, B = bt->count;
    PGB_REQUIRE(n_in >= 1 && n_in <= n, "%s: n_in must be in [1, n]", who);
    PGB_REQUIRE(log_gap_out <= log_n, "%s: log_gap_out %llu > log_n", who, (unsigned long long)log_gap_out);
    PGB_REQUIRE(nkeys >= log_n, "%s: needs log_n automorphism keys", who);
    PGB_REQUIRE(base2k >= 1 && base2k <= 63, "%s: base2k must be in [1, 63]", who);
    PGB_REQUIRE(dsize >= 1, "%s: dsize must be >= 1", who);
    // ---- the GLWEs: one layout on both sides ----
    const uint64_t cols = res->cols, size = res->size;
    PGB_REQUIRE(res->n == n && a->n == n, "%s: ring degree mismatch", who);
    PGB_REQUIRE(cols >= 2 && a->cols == cols, "%s: res and a must have the same rank + 1 >= 2 columns", who);
    PGB_REQUIRE(size >= 1 && size <= 65535 && a->size == size, "%s: res and a must have the same size in [1, 65535]", who);
    PGB_REQUIRE(res->data && a->data && (uintptr_t)res->data % 16 == 0 && (uintptr_t)a->data % 16 == 0,
                "%s: res and a data must be non-null and 16-byte aligned", who);
    const uint64_t g = n * cols * size * 8;
    PGB_REQUIRE(bt->stride_res % 16 == 0 && (B == 1 || bt->stride_res >= g),
                "%s: stride_res %llu must be a multiple of 16 and at least one GLWE (%llu bytes)", who, (unsigned long long)bt->stride_res,
                (unsigned long long)g);
    PGB_REQUIRE(bt->stride_a % 16 == 0, "%s: stride_a %llu must be a multiple of 16 (0 shares the inputs)", who, (unsigned long long)bt->stride_a);
    PGB_REQUIRE(bt->stride_b == 0, "%s: stride_b must be 0", who);
    PGB_REQUIRE(entry_stride % 16 == 0 && (n_in == 1 || entry_stride >= g),
                "%s: entry_stride %llu must be a multiple of 16 of at least one GLWE (%llu bytes)", who, (unsigned long long)entry_stride,
                (unsigned long long)g);
    // ---- the keys: log_n of one shape, cols_in = cols - 1, cols_out = cols ----
    const uint64_t key_bytes = pgb_bytes_of_vmp_pmat(m, keys[0].rows, keys[0].cols_in, keys[0].cols_out, keys[0].size);
    for (uint64_t i = 0; i < log_n; i++) {
        const pgb_vmp_pmat &k = keys[i];
        PGB_REQUIRE(k.data && (uintptr_t)k.data % 16 == 0, "%s: key %llu data must be non-null and 16-byte aligned", who, (unsigned long long)i);
        PGB_REQUIRE(k.n == n && k.cols_in == cols - 1 && k.cols_out == cols && k.rows >= 1 && k.size >= 1 && k.rows == keys[0].rows &&
                        k.size == keys[0].size,
                    "%s: key %llu must be a VmpPMat(dnum, rank, rank + 1, size) of the ring and of key 0's shape", who, (unsigned long long)i);
    }
    // ---- the index map ----
    PackPlan plan;
    PGB_REQUIRE(pack_plan(n, m->log_n, index, n_in, log_gap_out, &plan),
                "%s: the indices must be distinct, below n and multiples of 2^log_gap_out", who);
    // ---- extents in 128 bits, aliasing, scratch ----
    const unsigned __int128 a_ext128 = (unsigned __int128)(B - 1) * bt->stride_a + (unsigned __int128)(n_in - 1) * entry_stride + g;
    const unsigned __int128 res_ext128 = (unsigned __int128)(B - 1) * bt->stride_res + g;
    PGB_REQUIRE(a_ext128 <= (unsigned __int128)(UINTPTR_MAX - (uintptr_t)a->data), "%s: the inputs extend past the end of the address space",
                who);
    PGB_REQUIRE(res_ext128 <= (unsigned __int128)(UINTPTR_MAX - (uintptr_t)res->data),
                "%s: res extends past the end of the address space", who);
    const uint64_t a_ext = (uint64_t)a_ext128, res_ext = (uint64_t)res_ext128;
    PGB_REQUIRE(scratch != nullptr && (uintptr_t)scratch % 256 == 0, "%s: scratch must be non-null and 256-byte aligned", who);
    bool key_alias = false, key_scratch = false;
    for (uint64_t i = 0; i < log_n; i++) {
        key_alias |= ranges_overlap(res->data, res_ext, keys[i].data, key_bytes);
        key_scratch |= ranges_overlap(scratch, scratch_len, keys[i].data, key_bytes);
    }
    if (ranges_overlap(res->data, res_ext, a->data, a_ext) || key_alias) {
        pgb_set_error("%s: res must not overlap the inputs or a key", who);
        return PGB_ERR_ALIAS;
    }
    if (ranges_overlap(scratch, scratch_len, res->data, res_ext) || ranges_overlap(scratch, scratch_len, a->data, a_ext) || key_scratch) {
        pgb_set_error("%s: scratch must not overlap res, the inputs or a key", who);
        return PGB_ERR_ALIAS;
    }
    // the largest chunk of whole items whose scratch fits
    const uint64_t need1 = pack_bytes(m, size, base2k, &keys[0], dsize, log_gap_out, plan, 1, nullptr);
    if (scratch_len < need1) {
        pgb_set_error("%s: scratch of %zu bytes < required %llu for one item", who, scratch_len, (unsigned long long)need1);
        return PGB_ERR_SCRATCH;
    }
    uint64_t lo = 1, hi = umin64(B, pack_chunk_cap(plan));
    while (lo < hi) {
        const uint64_t mid = (lo + hi + 1) / 2;
        if (pack_bytes(m, size, base2k, &keys[0], dsize, log_gap_out, plan, mid, nullptr) <= scratch_len) lo = mid;
        else hi = mid - 1;
    }
    const uint64_t Bc = lo;
    PackLayout L;
    pack_bytes(m, size, base2k, &keys[0], dsize, log_gap_out, plan, Bc, &L);

    // ---- the descriptor table (offsets of states relative to the scratch, of inputs to the chunk's input base) ----
    const uint64_t R = plan.rounds.size();
    std::vector<PackSlot> host(plan.slots);
    std::vector<uint64_t> round_first(R);
    auto state_src = [&](const PackRef &r) -> PackSrc {
        if (r.round == -1) return PackSrc{r.w * entry_stride, bt->stride_a, 0, 0};
        const PackRound &pr = plan.rounds[r.round];
        const uint32_t c_off = r.w < pr.nb ? 0 : r.w < pr.nb + pr.nl ? pr.nb : pr.nb + pr.nl;
        const uint32_t n_c = r.w < pr.nb ? pr.nb : r.w < pr.nb + pr.nl ? pr.nl : pr.nh;
        return PackSrc{L.blk[r.round & 1] + (c_off * Bc + (r.w - c_off)) * g, n_c * g, 1, 0};
    };
    for (uint64_t i = 0, e = 0; i < R; i++) {
        const PackRound &pr = plan.rounds[i];
        round_first[i] = e;
        for (uint32_t w = 0; w < pr.width(); w++, e++) {
            PackSlot &s = host[e];
            s = PackSlot{};
            s.kind = w < pr.nb ? PACK_BOTH : w < pr.nb + pr.nl ? PACK_LO : PACK_HI;
            if (s.kind != PACK_HI) s.lo = state_src(pr.lo[w]);
            if (s.kind != PACK_LO) s.hi = state_src(pr.hi[w]);
            const uint32_t c_off = s.kind == PACK_BOTH ? 0 : s.kind == PACK_LO ? pr.nb : pr.nb + pr.nl;
            const uint32_t n_c = s.kind == PACK_BOTH ? pr.nb : s.kind == PACK_LO ? pr.nl : pr.nh;
            s.x_off = L.x + (c_off * Bc + (w - c_off)) * g;
            s.x_bs = n_c * g;
            s.y_off = L.y + w * g; // `both` slots only (w < nb)
        }
    }
    char *sc = (char *)scratch;
    if (R) PGB_CHECK_CUDA(cudaMemcpyAsync(sc, host.data(), host.size() * sizeof(PackSlot), cudaMemcpyHostToDevice, m->stream));

    const uint32_t words = (uint32_t)(n * cols);
    const uint64_t skip = log_n - log_gap_out;
    for (uint64_t b0 = 0; b0 < B; b0 += Bc) {
        const uint64_t nb = umin64(Bc, B - b0);
        const char *in = (const char *)a->data + b0 * bt->stride_a;
        pgb_vec_znx rc = *res;
        rc.data = (char *)res->data + b0 * bt->stride_res;
        for (uint64_t i = 0; i < R; i++) {
            const PackRound &pr = plan.rounds[i];
            const bool last = i + 1 == R;
            const uint32_t t = (uint32_t)(n >> (i + 1));
            const int64_t p = pgb_trace_galois_element(m, i);
            {
                PackPrepArgs pa = {reinterpret_cast<const PackSlot *>(sc) + round_first[i], in, sc, words, (uint32_t)n, pr.width(), t, (int)size,
                                   (int)base2k};
                ProfScope _ps(m, PROF_NORMALIZE);
                pack_prep_kernel<<<dim3((words + 255) / 256, (uint32_t)(nb * pr.width())), 256, 0, m->stream>>>(pa);
            }
            PGB_CHECK_CUDA(cudaGetLastError());
            // round i's outputs: block i & 1 per case (res in the last round, whose single slot is item-major already)
            auto out_of = [&](uint32_t c_off, pgb_vec_znx *o, uint64_t *o_bs) {
                *o = last ? rc : mk(sc + L.blk[i & 1] + c_off * Bc * g, n, cols, size);
                *o_bs = last ? bt->stride_res : g;
            };
            pgb_vec_znx z = mk(sc + L.blk[(i + 1) & 1], n, cols, size);
            if (pr.nb) {
                const pgb_vec_znx xb = mk(sc + L.x, n, cols, size);
                pgb_batch bta = {nb * pr.nb, g, g, 0};
                PGB_TRY(pgb_glwe_automorphism_batched(m, &z, base2k, &xb, base2k, &keys[i], base2k, p, dsize, &bta,
                                                      sc + L.rest, scratch_len - L.rest));
            }
            for (int kind = PACK_LO; kind <= PACK_HI; kind++) {
                const uint32_t c_off = kind == PACK_LO ? pr.nb : pr.nb + pr.nl, n_c = kind == PACK_LO ? pr.nl : pr.nh;
                if (!n_c) continue;
                pgb_vec_znx o;
                uint64_t o_bs;
                out_of(c_off, &o, &o_bs);
                const pgb_vec_znx xc = mk(sc + L.x + c_off * Bc * g, n, cols, size);
                pgb_batch bto = {nb * n_c, o_bs, g, 0};
                PGB_TRY(pgb_glwe_automorphism_op_batched(m, kind == PACK_LO ? 0 : 2, &o, base2k, &xc, &keys[i], base2k, p, dsize, &bto,
                                                         sc + L.rest, scratch_len - L.rest));
            }
            if (pr.nb) {
                pgb_vec_znx o;
                uint64_t o_bs;
                out_of(0, &o, &o_bs);
                PackCombineArgs ca = {sc + L.y, (const char *)z.data, g, (char *)o.data, o_bs, words, (uint32_t)n, t, (int)size, (int)base2k};
                { ProfScope _ps(m, PROF_NORMALIZE);
                pack_combine_kernel<<<dim3((words + 255) / 256, (uint32_t)(nb * pr.nb)), 256, 0, m->stream>>>(ca);
                }
                PGB_CHECK_CUDA(cudaGetLastError());
            }
        }
        if (!R && bt->stride_a >= g) { // no rounds: input 0 is the state, copied as the composition's glwe_copy does
            PGB_CHECK_CUDA(cudaMemcpy2DAsync(rc.data, bt->stride_res, in, bt->stride_a, g, nb, cudaMemcpyDeviceToDevice, m->stream));
        } else if (!R) { // the same with inputs shared by the batch, or items closer than one GLWE (a pitch the 2D copy does not take)
            { ProfScope _ps(m, PROF_ELEMENTWISE);
            pack_copy_kernel<<<dim3((uint32_t)((g / 16 + 255) / 256), (uint32_t)nb), 256, 0, m->stream>>>(in, bt->stride_a, (char *)rc.data,
                                                                                                          bt->stride_res, (uint32_t)(g / 16));
            }
            PGB_CHECK_CUDA(cudaGetLastError());
        }
        if (skip < log_n) {
            pgb_batch btt = {nb, bt->stride_res, 0, 0};
            PGB_TRY(pgb_glwe_trace_assign_batched(m, &rc, base2k, skip, keys, nkeys, base2k, dsize, &btt, sc + L.rest, scratch_len - L.rest));
        }
    }
    return PGB_OK;
}
