// api.cu -- the C ABI (include/poulpy_b200.h): module / memory management and the HalImpl-shaped entry points.
// Shape rules (min sizes, zero tails, limb_offset, step/offset gathers) restate the reference HAL semantics cited in
// the header; all arithmetic is in the kernels of ntt120_dft.cu, ntt120_ops.cu, fft64.cu and big.cu.
#include <stdarg.h>

#include "common.cuh"
#include "internal.h"

static thread_local char g_err[512] = "";
void pgb_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}
extern "C" const char *pgb_last_error(void) { return g_err; }

extern "C" int pgb_device_count(void) {
    int c = 0;
    if (cudaGetDeviceCount(&c) != cudaSuccess) return 0;
    return c;
}

// ---- profiler: CUDA events on the launching stream around every kernel, accumulated per category --------------
#include <vector>
struct ProfState {
    std::vector<cudaEvent_t> pool;            // start/stop pairs
    std::vector<int> cat;                     // category of pair i
    size_t used = 0;
    double ms[PROF_NCAT] = {0};
    uint64_t count[PROF_NCAT] = {0};
};
void prof_begin(pgb_module *m, int cat) {
    ProfState *p = m->prof;
    if (p->used * 2 + 2 > p->pool.size()) {
        cudaEvent_t a, b;
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        p->pool.push_back(a);
        p->pool.push_back(b);
        p->cat.push_back(cat);
    }
    p->cat[p->used] = cat;
    cudaEventRecord(p->pool[2 * p->used], m->stream);
}
void prof_end(pgb_module *m) {
    ProfState *p = m->prof;
    cudaEventRecord(p->pool[2 * p->used + 1], m->stream);
    p->used++;
}
static int prof_collect(pgb_module *m) {
    ProfState *p = m->prof;
    if (!p) return PGB_OK;
    PGB_CHECK_CUDA(cudaStreamSynchronize(m->stream));
    for (size_t i = 0; i < p->used; i++) {
        float ms = 0.f;
        PGB_CHECK_CUDA(cudaEventElapsedTime(&ms, p->pool[2 * i], p->pool[2 * i + 1]));
        p->ms[p->cat[i]] += ms;
        p->count[p->cat[i]]++;
    }
    p->used = 0;
    return PGB_OK;
}
extern "C" int pgb_profile_enable(pgb_module *m, int on) {
    if (on && !m->prof) m->prof = new ProfState();
    if (!on) PGB_TRY(prof_collect(m));
    m->prof_on = on != 0;
    return PGB_OK;
}
extern "C" int pgb_profile_read(pgb_module *m, double *ms, uint64_t *launches, int reset) {
    PGB_REQUIRE(m->prof != nullptr, "pgb_profile_read: profiling was never enabled");
    PGB_TRY(prof_collect(m));
    for (int c = 0; c < PROF_NCAT; c++) {
        ms[c] = m->prof->ms[c];
        launches[c] = m->prof->count[c];
        if (reset) {
            m->prof->ms[c] = 0;
            m->prof->count[c] = 0;
        }
    }
    return PGB_OK;
}
extern "C" const char *pgb_profile_category_name(int c) {
    static const char *names[PROF_NCAT] = {"dft_forward", "dft_inverse", "vmp_apply", "normalize", "elementwise", "other", "gadget_fused"};
    return (c >= 0 && c < PROF_NCAT) ? names[c] : "?";
}

// ---- module -------------------------------------------------------------------------------------------
extern "C" int pgb_module_new(uint64_t n, int flavour, int device, pgb_module **out) {
    PGB_REQUIRE(out != nullptr, "pgb_module_new: out is null");
    *out = nullptr;
    PGB_REQUIRE(n >= 16 && n <= (1u << 16) && (n & (n - 1)) == 0, "pgb_module_new: n must be a power of two in [16, 2^16], got %llu",
                (unsigned long long)n);
    PGB_REQUIRE(flavour == PGB_NTT120 || flavour == PGB_FFT64, "pgb_module_new: unknown flavour %d", flavour);
    int cnt = 0;
    cudaError_t e = cudaGetDeviceCount(&cnt);
    if (e != cudaSuccess || cnt == 0) {
        pgb_set_error("pgb_module_new: no CUDA device available (%s); this backend has no CPU fallback",
                      e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        return PGB_ERR_CUDA;
    }
    PGB_REQUIRE(device >= 0 && device < cnt, "pgb_module_new: device %d out of range [0, %d)", device, cnt);
    PGB_CHECK_CUDA(cudaSetDevice(device));
    pgb_module *m = (pgb_module *)calloc(1, sizeof(pgb_module));
    m->n = n;
    m->log_n = ilog2_u64(n);
    m->flavour = flavour;
    m->device = device;
    {   // the environment seeds the knobs once per module (pgb_module_set_option changes them later)
        static const struct { int opt; const char *env; int64_t dflt; bool flag; } seeds[] = {
            {PGB_OPT_NO_FUSION, "PGB_NO_FUSION", 0, true},   {PGB_OPT_NO_GADGET, "PGB_NO_GADGET", 0, true},
            {PGB_OPT_NO_COLLAPSE, "PGB_NO_COLLAPSE", 0, true}, {PGB_OPT_CGGI_VARIANT, "PGB_CGGI_VARIANT", 0, false},
            {PGB_OPT_CGGI_BLOCK_BT1, "PGB_CGGI_BLOCK_BT1", 0, true}, {PGB_OPT_VMP_NO_BT, "PGB_VMP_NO_BT", 0, true},
            {PGB_OPT_VMP_CT, "PGB_VMP_CT", 0, false},       {PGB_OPT_GADGET_MB, "PGB_GADGET_MB", 3, false},
            {PGB_OPT_HOST_CHUNK_MB, "PGB_HOST_CHUNK_MB", 32, false}, {PGB_OPT_CGGI_NTT_PRIMES, "PGB_CGGI_NTT_PRIMES", 0, false},
            {PGB_OPT_GADGET_PRIMES, "PGB_GADGET_PRIMES", 0, false}, {PGB_OPT_CGGI_CLUSTER, "PGB_CGGI_CLUSTER", 0, false}};
        for (const auto &sd : seeds) {
            const char *e = getenv(sd.env);
            m->opt[sd.opt] = e ? (sd.flag ? 1 : (int64_t)atoll(e)) : sd.dflt;
        }
    }
    PGB_CHECK_CUDA(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking));
    m->own_stream = true;
    for (int i = 0; i < 2; i++) PGB_CHECK_CUDA(cudaStreamCreateWithFlags(&m->aux_stream[i], cudaStreamNonBlocking));
    for (int i = 0; i < 8; i++) PGB_CHECK_CUDA(cudaEventCreateWithFlags(&m->ev[i], cudaEventDisableTiming));
    int s = flavour == PGB_NTT120 ? ntt120_module_init(m) : fft64_module_init(m);
    if (s != PGB_OK) {
        pgb_module_destroy(m);
        return s;
    }
    *out = m;
    return PGB_OK;
}

extern "C" void pgb_module_destroy(pgb_module *m) {
    if (!m) return;
    cudaSetDevice(m->device);
    cudaDeviceSynchronize();
    cudaFree(m->ntt_fwd);
    cudaFree(m->ntt_inv);
    cudaFree(m->ntt_last16_f);
    cudaFree(m->ntt_last16_i);
    cudaFree(m->fft_fwd);
    cudaFree(m->fft_inv);
    cudaFree(m->fft_last_f);
    cudaFree(m->fft_last_i);
    cudaFree(m->ws);
    cudaFree(m->carry_ws);
    cudaFree(m->aux_ws);
    key_cache_destroy(m);
    if (m->prof) {
        for (cudaEvent_t e : m->prof->pool) cudaEventDestroy(e);
        delete m->prof;
    }
    for (int i = 0; i < 4; i++)
        if (m->pinned[i]) cudaFreeHost(m->pinned[i]);
    if (m->own_stream && m->stream) cudaStreamDestroy(m->stream);
    for (int i = 0; i < 2; i++)
        if (m->aux_stream[i]) cudaStreamDestroy(m->aux_stream[i]);
    for (int i = 0; i < 8; i++)
        if (m->ev[i]) cudaEventDestroy(m->ev[i]);
    free(m);
}
extern "C" int pgb_module_set_option(pgb_module *m, int option, int64_t value) {
    PGB_REQUIRE(m && option >= 0 && option < PGB_OPT_COUNT, "pgb_module_set_option: unknown option %d", option);
    m->opt[option] = value;
    return PGB_OK;
}
extern "C" int64_t pgb_module_get_option(const pgb_module *m, int option) {
    return (m && option >= 0 && option < PGB_OPT_COUNT) ? m->opt[option] : -1;
}
extern "C" uint64_t pgb_module_n(const pgb_module *m) { return m->n; }
extern "C" int pgb_module_flavour(const pgb_module *m) { return m->flavour; }
extern "C" uint64_t pgb_module_launch_count(const pgb_module *m) { return m->launches; }
extern "C" int pgb_module_set_stream(pgb_module *m, void *cuda_stream) {
    PGB_CHECK_CUDA(cudaStreamSynchronize(m->stream));
    if (m->own_stream && m->stream) cudaStreamDestroy(m->stream);
    if (cuda_stream == nullptr) {
        PGB_CHECK_CUDA(cudaStreamCreateWithFlags(&m->stream, cudaStreamNonBlocking));
        m->own_stream = true;
    } else {
        m->stream = (cudaStream_t)cuda_stream;
        m->own_stream = false;
    }
    return PGB_OK;
}
extern "C" int pgb_module_sync(pgb_module *m) {
    PGB_CHECK_CUDA(cudaStreamSynchronize(m->stream));
    return PGB_OK;
}

// ---- memory ---------------------------------------------------------------------------------------------
extern "C" void *pgb_alloc_bytes(size_t len) {
    void *p = nullptr;
    if (cudaMallocManaged(&p, len ? len : 1) != cudaSuccess) return nullptr;
    cudaMemset(p, 0, len);
    cudaDeviceSynchronize();
    return p;
}
extern "C" void *pgb_alloc_device_bytes(size_t len) {
    void *p = nullptr;
    if (cudaMalloc(&p, len ? len : 1) != cudaSuccess) return nullptr;
    // the memset runs on the legacy stream, the modules' streams are non-blocking: without the synchronisation a kernel launched right
    // after the allocation could be overtaken by the zero fill
    cudaMemset(p, 0, len);
    cudaStreamSynchronize(0);
    return p;
}
extern "C" void *pgb_alloc_pinned_bytes(size_t len) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, len ? len : 1, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
extern "C" void pgb_free(void *p) { cudaFree(p); }
extern "C" void pgb_free_pinned(void *p) { cudaFreeHost(p); }
// Setup / test helpers, not on the hot path.  They run on the legacy stream while the modules' streams are non-blocking, and a pageable
// host-to-device cudaMemcpy may return before its last DMA chunk has landed: a full device synchronisation on both sides makes them
// ordered against every module stream.
extern "C" int pgb_memcpy_h2d(void *dst, const void *src, size_t len) {
    PGB_CHECK_CUDA(cudaDeviceSynchronize());
    PGB_CHECK_CUDA(cudaMemcpy(dst, src, len, cudaMemcpyHostToDevice));
    PGB_CHECK_CUDA(cudaDeviceSynchronize());
    return PGB_OK;
}
extern "C" int pgb_memcpy_d2h(void *dst, const void *src, size_t len) {
    PGB_CHECK_CUDA(cudaDeviceSynchronize());
    PGB_CHECK_CUDA(cudaMemcpy(dst, src, len, cudaMemcpyDeviceToHost));
    return PGB_OK;
}
extern "C" int pgb_memcpy_d2d(void *dst, const void *src, size_t len) {
    PGB_CHECK_CUDA(cudaDeviceSynchronize());
    PGB_CHECK_CUDA(cudaMemcpy(dst, src, len, cudaMemcpyDeviceToDevice));
    PGB_CHECK_CUDA(cudaDeviceSynchronize());
    return PGB_OK;
}
extern "C" int pgb_memset(void *dst, int byte, size_t len) {
    PGB_CHECK_CUDA(cudaMemset(dst, byte, len));
    return PGB_OK;
}
// Zero fill of a block that is being recycled by a host-side pool: ordered against every module stream on both sides (work that still
// uses the block's previous life finishes first; nothing launched afterwards can overtake the fill).
extern "C" int pgb_set_device(int device) {
    PGB_CHECK_CUDA(cudaSetDevice(device));
    return PGB_OK;
}
extern "C" int pgb_module_device(const pgb_module *m) { return m ? m->device : -1; }
extern "C" int pgb_current_device(void) {
    int d = -1;
    return cudaGetDevice(&d) == cudaSuccess ? d : -1;
}
extern "C" int pgb_recycle_device_bytes(void *p, size_t len) {
    PGB_CHECK_CUDA(cudaDeviceSynchronize());
    PGB_CHECK_CUDA(cudaMemset(p, 0, len));
    PGB_CHECK_CUDA(cudaStreamSynchronize(0));
    return PGB_OK;
}

extern "C" size_t pgb_size_of_scalar_prep(const pgb_module *m) { return prep_bytes(m); }
extern "C" size_t pgb_size_of_scalar_big(const pgb_module *m) { return big_bytes(m); }
extern "C" size_t pgb_bytes_of_vec_znx(const pgb_module *m, uint64_t cols, uint64_t size) { return m->n * cols * size * 8; }
extern "C" size_t pgb_bytes_of_vec_znx_dft(const pgb_module *m, uint64_t cols, uint64_t size) { return m->n * cols * size * prep_bytes(m); }
extern "C" size_t pgb_bytes_of_vec_znx_big(const pgb_module *m, uint64_t cols, uint64_t size) { return m->n * cols * size * big_bytes(m); }
extern "C" size_t pgb_bytes_of_svp_ppol(const pgb_module *m, uint64_t cols) { return m->n * cols * prep_bytes(m); }
extern "C" size_t pgb_bytes_of_vmp_pmat(const pgb_module *m, uint64_t rows, uint64_t cols_in, uint64_t cols_out, uint64_t size) {
    return m->n * rows * cols_in * cols_out * size * prep_bytes(m);
}

// ---- helpers ----------------------------------------------------------------------------------------------
static const pgb_batch ONE = {1, 0, 0, 0};
#define CHECK_BATCH(bt)                                                                          \
    PGB_REQUIRE((bt) != nullptr && (bt)->count <= 65535, "batch count must be <= 65535 per call (got %llu)", \
                (unsigned long long)((bt) ? (bt)->count : 0))
#define CHECK_N(v, what) PGB_REQUIRE((v)->n == m->n, what ": n = %llu does not match the module (%llu)", (unsigned long long)(v)->n, (unsigned long long)m->n)
#define CHECK_COL(v, col, what) PGB_REQUIRE((col) < (v)->cols, what ": column %llu out of range (cols = %llu)", (unsigned long long)(col), (unsigned long long)(v)->cols)

static int sync_if(pgb_module *m, bool sync) {
    if (sync) PGB_CHECK_CUDA(cudaStreamSynchronize(m->stream));
    return PGB_OK;
}

// ---- vec_znx_dft_apply -------------------------------------------------------------------------------------
static int dft_apply_impl(pgb_module *m, uint64_t step, uint64_t offset, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx *a,
                          uint64_t a_col, const pgb_batch *bt) {
    CHECK_BATCH(bt);
    CHECK_N(res, "vec_znx_dft_apply(res)");
    CHECK_N(a, "vec_znx_dft_apply(a)");
    CHECK_COL(res, res_col, "vec_znx_dft_apply(res)");
    CHECK_COL(a, a_col, "vec_znx_dft_apply(a)");
    PGB_REQUIRE(step > 0, "vec_znx_dft_apply: step must be > 0");
    const uint64_t n = m->n, pb = prep_bytes(m);
    const uint64_t steps = div_ceil64(a->size, step);
    const uint64_t min_steps = umin64(res->size, steps);
    // limbs j < nvalid have a source limb offset + j*step < a.size
    uint64_t nvalid = offset < a->size ? umin64(min_steps, div_ceil64(a->size - offset, step)) : 0;
    LimbSet in = {(char *)a->data + limb_off(n, a->cols, a_col, offset, 8), step * a->cols * n * 8, bt->stride_a};
    LimbSet out = {(char *)res->data + limb_off(n, res->cols, res_col, 0, pb), res->cols * n * pb, bt->stride_res};
    if (m->flavour == PGB_NTT120) {
        PGB_TRY(ntt120_forward(m, in, out, (int)nvalid, (int)bt->count));
        // ntt120/vec_znx_dft.rs:201-214: every other limb of the column is zeroed
        LimbSet z = out;
        z.base += nvalid * out.limb_stride;
        PGB_TRY(raw_limbs(m, true, z, z, n * pb, (uint32_t)(res->size - nvalid), (uint32_t)bt->count));
    } else {
        PGB_TRY(fft64_forward(m, in, out, (int)nvalid, (int)bt->count));
        // fft64/vec_znx_dft.rs:189-199: only limbs >= min_steps are zeroed; limbs in [nvalid, min_steps) stay untouched
        LimbSet z = out;
        z.base += min_steps * out.limb_stride;
        PGB_TRY(raw_limbs(m, true, z, z, n * pb, (uint32_t)(res->size - min_steps), (uint32_t)bt->count));
    }
    return PGB_OK;
}
extern "C" int pgb_vec_znx_dft_apply(pgb_module *m, uint64_t step, uint64_t offset, pgb_vec_znx_dft *res, uint64_t res_col,
                                     const pgb_vec_znx *a, uint64_t a_col) {
    PGB_TRY(dft_apply_impl(m, step, offset, res, res_col, a, a_col, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_dft_apply_batched(pgb_module *m, uint64_t step, uint64_t offset, pgb_vec_znx_dft *res, uint64_t res_col,
                                             const pgb_vec_znx *a, uint64_t a_col, const pgb_batch *bt) {
    return dft_apply_impl(m, step, offset, res, res_col, a, a_col, bt);
}

// ---- vec_znx_idft_apply ------------------------------------------------------------------------------------
extern "C" size_t pgb_vec_znx_idft_apply_tmp_bytes(const pgb_module *) { return 0; }

static int idft_apply_impl(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx_dft *a, uint64_t a_col,
                           const pgb_batch *bt) {
    CHECK_BATCH(bt);
    CHECK_N(res, "vec_znx_idft_apply(res)");
    CHECK_N(a, "vec_znx_idft_apply(a)");
    CHECK_COL(res, res_col, "vec_znx_idft_apply(res)");
    CHECK_COL(a, a_col, "vec_znx_idft_apply(a)");
    const uint64_t n = m->n, pb = prep_bytes(m), bb = big_bytes(m);
    const uint64_t min_size = umin64(res->size, a->size);
    LimbSet in = {(char *)a->data + limb_off(n, a->cols, a_col, 0, pb), a->cols * n * pb, bt->stride_a};
    LimbSet out = {(char *)res->data + limb_off(n, res->cols, res_col, 0, bb), res->cols * n * bb, bt->stride_res};
    if (m->flavour == PGB_NTT120) PGB_TRY(ntt120_inverse_big(m, in, out, (int)min_size, (int)bt->count));
    else PGB_TRY(fft64_inverse_big(m, in, out, (int)min_size, (int)bt->count));
    LimbSet z = out;
    z.base += min_size * out.limb_stride;
    return raw_limbs(m, true, z, z, n * bb, (uint32_t)(res->size - min_size), (uint32_t)bt->count);
}
extern "C" int pgb_vec_znx_idft_apply(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx_dft *a, uint64_t a_col) {
    PGB_TRY(idft_apply_impl(m, res, res_col, a, a_col, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_idft_apply_batched(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx_dft *a,
                                              uint64_t a_col, const pgb_batch *bt) {
    return idft_apply_impl(m, res, res_col, a, a_col, bt);
}
extern "C" int pgb_vec_znx_idft_apply_tmpa(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, pgb_vec_znx_dft *a, uint64_t a_col) {
    // `a` may be clobbered by the reference; this backend leaves it intact (allowed: tmpa only permits, never requires, it)
    return pgb_vec_znx_idft_apply(m, res, res_col, a, a_col);
}
static int idft_consume_impl(pgb_module *m, pgb_vec_znx_dft *a, const pgb_batch *bt) {
    CHECK_BATCH(bt);
    CHECK_N(a, "vec_znx_idft_apply_consume(a)");
    const uint64_t n = m->n, pb = prep_bytes(m), bb = big_bytes(m);
    PGB_REQUIRE(bb <= pb, "vec_znx_idft_apply_consume: ScalarBig larger than ScalarPrep");
    // flat limb k: DFT limb at k*n*pb, big limb at k*n*bb (vec_znx_dft.rs:327-409); pb == bb for both flavours here
    LimbSet in = {(char *)a->data, n * pb, bt->stride_res};
    LimbSet out = {(char *)a->data, n * bb, bt->stride_res};
    const int jobs = (int)(a->cols * a->size);
    if (m->flavour == PGB_NTT120) return ntt120_inverse_big(m, in, out, jobs, (int)bt->count);
    return fft64_inverse_big(m, in, out, jobs, (int)bt->count);
}
extern "C" int pgb_vec_znx_idft_apply_consume(pgb_module *m, pgb_vec_znx_dft *a) {
    PGB_TRY(idft_consume_impl(m, a, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_idft_apply_consume_batched(pgb_module *m, pgb_vec_znx_dft *a, const pgb_batch *bt) {
    return idft_consume_impl(m, a, bt);
}

// ---- DFT-domain add / sub / copy / zero ----------------------------------------------------------------------
static LimbSet dft_col(const pgb_module *m, const pgb_vec_znx_dft *v, uint64_t col, uint64_t first_limb, uint64_t bstride) {
    const uint64_t pb = prep_bytes(m);
    LimbSet s = {(char *)v->data + limb_off(m->n, v->cols, col, first_limb, pb), v->cols * m->n * pb, bstride};
    return s;
}
static int dft_ew(pgb_module *m, int op, LimbSet dst, LimbSet a, LimbSet b, uint64_t jobs, uint64_t batch) {
    if (op == EW_COPY || op == EW_ZERO) return raw_limbs(m, op == EW_ZERO, dst, a, m->n * prep_bytes(m), (uint32_t)jobs, (uint32_t)batch);
    if (m->flavour == PGB_NTT120) return ntt120_ew(m, op, dst, a, b, (uint32_t)jobs, (uint32_t)batch);
    return fft64_ew(m, op, dst, a, b, (uint32_t)jobs, (uint32_t)batch);
}
static LimbSet shift(LimbSet s, uint64_t limbs) {
    s.base += limbs * s.limb_stride;
    return s;
}

// add_into / sub share the size rules of vec_znx_dft.rs:418-470 / :522-580
static int dft_addsub_into(pgb_module *m, bool sub, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a, uint64_t a_col,
                           const pgb_vec_znx_dft *b, uint64_t b_col) {
    CHECK_N(res, "vec_znx_dft_add/sub(res)");
    CHECK_N(a, "vec_znx_dft_add/sub(a)");
    CHECK_N(b, "vec_znx_dft_add/sub(b)");
    CHECK_COL(res, res_col, "vec_znx_dft_add/sub(res)");
    CHECK_COL(a, a_col, "vec_znx_dft_add/sub(a)");
    CHECK_COL(b, b_col, "vec_znx_dft_add/sub(b)");
    LimbSet R = dft_col(m, res, res_col, 0, 0), A = dft_col(m, a, a_col, 0, 0), B = dft_col(m, b, b_col, 0, 0);
    const uint64_t rs = res->size;
    const bool a_small = a->size <= b->size;
    const uint64_t sum = umin64(a_small ? a->size : b->size, rs), cpy = umin64(a_small ? b->size : a->size, rs);
    PGB_TRY(dft_ew(m, sub ? EW_SUB : EW_ADD, R, A, B, sum, 1));
    if (a_small) PGB_TRY(dft_ew(m, sub ? EW_NEG : EW_COPY, shift(R, sum), shift(B, sum), shift(B, sum), cpy - sum, 1));
    else PGB_TRY(dft_ew(m, EW_COPY, shift(R, sum), shift(A, sum), shift(A, sum), cpy - sum, 1));
    PGB_TRY(dft_ew(m, EW_ZERO, shift(R, cpy), shift(R, cpy), shift(R, cpy), rs - cpy, 1));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_dft_add_into(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a, uint64_t a_col,
                                        const pgb_vec_znx_dft *b, uint64_t b_col) {
    return dft_addsub_into(m, false, res, res_col, a, a_col, b, b_col);
}
extern "C" int pgb_vec_znx_dft_sub(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a, uint64_t a_col,
                                   const pgb_vec_znx_dft *b, uint64_t b_col) {
    return dft_addsub_into(m, true, res, res_col, a, a_col, b, b_col);
}
static int dft_assign_impl(pgb_module *m, int op, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a, uint64_t a_col,
                           uint64_t res_first, uint64_t a_first, uint64_t count, const pgb_batch *bt) {
    CHECK_BATCH(bt);
    CHECK_N(res, "vec_znx_dft_*_assign(res)");
    CHECK_N(a, "vec_znx_dft_*_assign(a)");
    CHECK_COL(res, res_col, "vec_znx_dft_*_assign(res)");
    CHECK_COL(a, a_col, "vec_znx_dft_*_assign(a)");
    LimbSet R = dft_col(m, res, res_col, res_first, bt->stride_res), A = dft_col(m, a, a_col, a_first, bt->stride_a);
    return dft_ew(m, op, R, R, A, count, bt->count); // R = R op A
}
extern "C" int pgb_vec_znx_dft_add_assign(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a, uint64_t a_col) {
    PGB_TRY(dft_assign_impl(m, EW_ADD, res, res_col, a, a_col, 0, 0, umin64(res->size, a->size), &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_dft_add_assign_batched(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a,
                                                  uint64_t a_col, const pgb_batch *bt) {
    return dft_assign_impl(m, EW_ADD, res, res_col, a, a_col, 0, 0, umin64(res->size, a->size), bt);
}
extern "C" int pgb_vec_znx_dft_sub_assign(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a, uint64_t a_col) {
    PGB_TRY(dft_assign_impl(m, EW_SUB, res, res_col, a, a_col, 0, 0, umin64(res->size, a->size), &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_dft_sub_assign_batched(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a,
                                                  uint64_t a_col, const pgb_batch *bt) {
    return dft_assign_impl(m, EW_SUB, res, res_col, a, a_col, 0, 0, umin64(res->size, a->size), bt);
}
// vec_znx_dft.rs:488-520
extern "C" int pgb_vec_znx_dft_add_scaled_assign(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a,
                                                 uint64_t a_col, int64_t a_scale) {
    const uint64_t rs = res->size, as = a->size;
    if (a_scale > 0) {
        const uint64_t sh = umin64((uint64_t)a_scale, as), mn = umin64(as, rs);
        PGB_TRY(dft_assign_impl(m, EW_ADD, res, res_col, a, a_col, 0, sh, mn > sh ? mn - sh : 0, &ONE));
    } else if (a_scale < 0) {
        const uint64_t sh = umin64((uint64_t)(-a_scale), rs);
        PGB_TRY(dft_assign_impl(m, EW_ADD, res, res_col, a, a_col, sh, 0, umin64(as, rs - sh), &ONE));
    } else {
        PGB_TRY(dft_assign_impl(m, EW_ADD, res, res_col, a, a_col, 0, 0, umin64(as, rs), &ONE));
    }
    return sync_if(m, true);
}
// vec_znx_dft.rs:598-616: res = a - res over min sizes, res = -res on the remaining limbs
extern "C" int pgb_vec_znx_dft_sub_negate_assign(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a,
                                                 uint64_t a_col) {
    CHECK_N(res, "vec_znx_dft_sub_negate_assign(res)");
    CHECK_N(a, "vec_znx_dft_sub_negate_assign(a)");
    CHECK_COL(res, res_col, "vec_znx_dft_sub_negate_assign(res)");
    CHECK_COL(a, a_col, "vec_znx_dft_sub_negate_assign(a)");
    const uint64_t rs = res->size, sum = umin64(rs, a->size);
    LimbSet R = dft_col(m, res, res_col, 0, 0), A = dft_col(m, a, a_col, 0, 0);
    PGB_TRY(dft_ew(m, EW_SUB, R, A, R, sum, 1));
    PGB_TRY(dft_ew(m, EW_NEG, shift(R, sum), shift(R, sum), shift(R, sum), rs - sum, 1));
    return sync_if(m, true);
}
static int dft_copy_impl(pgb_module *m, uint64_t step, uint64_t offset, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a,
                         uint64_t a_col, const pgb_batch *bt) {
    CHECK_BATCH(bt);
    CHECK_N(res, "vec_znx_dft_copy(res)");
    CHECK_N(a, "vec_znx_dft_copy(a)");
    CHECK_COL(res, res_col, "vec_znx_dft_copy(res)");
    CHECK_COL(a, a_col, "vec_znx_dft_copy(a)");
    PGB_REQUIRE(step > 0, "vec_znx_dft_copy: step must be > 0");
    const uint64_t steps = div_ceil64(a->size, step), min_steps = umin64(res->size, steps);
    const uint64_t nvalid = offset < a->size ? umin64(min_steps, div_ceil64(a->size - offset, step)) : 0;
    LimbSet R = dft_col(m, res, res_col, 0, bt->stride_res);
    LimbSet A = dft_col(m, a, a_col, offset, bt->stride_a);
    A.limb_stride *= step;
    PGB_TRY(dft_ew(m, EW_COPY, R, A, A, nvalid, bt->count));
    return dft_ew(m, EW_ZERO, shift(R, nvalid), shift(R, nvalid), shift(R, nvalid), res->size - nvalid, bt->count);
}
extern "C" int pgb_vec_znx_dft_copy(pgb_module *m, uint64_t step, uint64_t offset, pgb_vec_znx_dft *res, uint64_t res_col,
                                    const pgb_vec_znx_dft *a, uint64_t a_col) {
    PGB_TRY(dft_copy_impl(m, step, offset, res, res_col, a, a_col, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_dft_copy_batched(pgb_module *m, uint64_t step, uint64_t offset, pgb_vec_znx_dft *res, uint64_t res_col,
                                            const pgb_vec_znx_dft *a, uint64_t a_col, const pgb_batch *bt) {
    return dft_copy_impl(m, step, offset, res, res_col, a, a_col, bt);
}
static int dft_zero_impl(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_batch *bt) {
    CHECK_BATCH(bt);
    CHECK_N(res, "vec_znx_dft_zero(res)");
    CHECK_COL(res, res_col, "vec_znx_dft_zero(res)");
    LimbSet R = dft_col(m, res, res_col, 0, bt->stride_res);
    return dft_ew(m, EW_ZERO, R, R, R, res->size, bt->count);
}
extern "C" int pgb_vec_znx_dft_zero(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col) {
    PGB_TRY(dft_zero_impl(m, res, res_col, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_dft_zero_batched(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_batch *bt) {
    return dft_zero_impl(m, res, res_col, bt);
}

// ---- svp ------------------------------------------------------------------------------------------------------
extern "C" int pgb_svp_prepare(pgb_module *m, pgb_svp_ppol *res, uint64_t res_col, const pgb_scalar_znx *a, uint64_t a_col) {
    CHECK_N(res, "svp_prepare(res)");
    CHECK_N(a, "svp_prepare(a)");
    CHECK_COL(res, res_col, "svp_prepare(res)");
    CHECK_COL(a, a_col, "svp_prepare(a)");
    const uint64_t n = m->n, pb = prep_bytes(m);
    LimbSet in = {(char *)a->data + a_col * n * 8, 0, 0};
    LimbSet out = {(char *)res->data + res_col * n * pb, 0, 0};
    if (m->flavour == PGB_NTT120) PGB_TRY(ntt120_forward(m, in, out, 1, 1));
    else PGB_TRY(fft64_forward(m, in, out, 1, 1));
    return sync_if(m, true);
}
static int svp_apply_impl(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_svp_ppol *a, uint64_t a_col,
                          const pgb_vec_znx_dft *b, uint64_t b_col, const pgb_batch *bt) {
    CHECK_BATCH(bt);
    CHECK_N(res, "svp_apply_dft_to_dft(res)");
    CHECK_N(a, "svp_apply_dft_to_dft(a)");
    CHECK_N(b, "svp_apply_dft_to_dft(b)");
    CHECK_COL(res, res_col, "svp_apply_dft_to_dft(res)");
    CHECK_COL(a, a_col, "svp_apply_dft_to_dft(a)");
    CHECK_COL(b, b_col, "svp_apply_dft_to_dft(b)");
    const uint64_t pb = prep_bytes(m);
    const uint64_t min_size = umin64(res->size, b->size);
    LimbSet R = dft_col(m, res, res_col, 0, bt->stride_res), B = dft_col(m, b, b_col, 0, bt->stride_b);
    LimbSet P = {(char *)a->data + a_col * m->n * pb, 0, bt->stride_a}; // same ppol for every limb
    PGB_TRY(dft_ew(m, EW_MUL, R, P, B, min_size, bt->count));
    return dft_ew(m, EW_ZERO, shift(R, min_size), shift(R, min_size), shift(R, min_size), res->size - min_size, bt->count);
}
extern "C" int pgb_svp_apply_dft_to_dft(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_svp_ppol *a, uint64_t a_col,
                                        const pgb_vec_znx_dft *b, uint64_t b_col) {
    PGB_TRY(svp_apply_impl(m, res, res_col, a, a_col, b, b_col, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_svp_apply_dft_to_dft_batched(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_svp_ppol *a,
                                                uint64_t a_col, const pgb_vec_znx_dft *b, uint64_t b_col, const pgb_batch *bt) {
    return svp_apply_impl(m, res, res_col, a, a_col, b, b_col, bt);
}
// HalImpl::svp_apply_dft (hal_impl.rs:600): res[res_col] = ppol[a_col] * DFT(b[b_col]) for min(res.size, b.size) limbs, zero the rest
// (fft64/svp.rs:21-55; NTT120: hal_defaults/svp_ppol.rs:93-107 = vec_znx_dft_apply into a temporary + svp_apply_dft_to_dft).  The
// forward transforms land directly in res, then the product is taken in place: same values, no temporary.
extern "C" int pgb_svp_apply_dft(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_svp_ppol *a, uint64_t a_col,
                                 const pgb_vec_znx *b, uint64_t b_col) {
    CHECK_N(res, "svp_apply_dft(res)");
    CHECK_N(a, "svp_apply_dft(a)");
    CHECK_N(b, "svp_apply_dft(b)");
    CHECK_COL(res, res_col, "svp_apply_dft(res)");
    CHECK_COL(a, a_col, "svp_apply_dft(a)");
    CHECK_COL(b, b_col, "svp_apply_dft(b)");
    const uint64_t n = m->n, pb = prep_bytes(m), min_size = umin64(res->size, b->size);
    LimbSet in = {(char *)b->data + limb_off(n, b->cols, b_col, 0, 8), b->cols * n * 8, 0};
    LimbSet R = dft_col(m, res, res_col, 0, 0);
    if (m->flavour == PGB_NTT120) PGB_TRY(ntt120_forward(m, in, R, (int)min_size, 1));
    else PGB_TRY(fft64_forward(m, in, R, (int)min_size, 1));
    LimbSet P = {(char *)a->data + a_col * n * pb, 0, 0};
    PGB_TRY(dft_ew(m, EW_MUL, R, P, R, min_size, 1));
    PGB_TRY(dft_ew(m, EW_ZERO, shift(R, min_size), shift(R, min_size), shift(R, min_size), res->size - min_size, 1));
    return sync_if(m, true);
}
extern "C" int pgb_svp_apply_dft_to_dft_assign(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_svp_ppol *a,
                                               uint64_t a_col) {
    CHECK_N(res, "svp_apply_dft_to_dft_assign(res)");
    CHECK_N(a, "svp_apply_dft_to_dft_assign(a)");
    CHECK_COL(res, res_col, "svp_apply_dft_to_dft_assign(res)");
    CHECK_COL(a, a_col, "svp_apply_dft_to_dft_assign(a)");
    LimbSet R = dft_col(m, res, res_col, 0, 0);
    LimbSet P = {(char *)a->data + a_col * m->n * prep_bytes(m), 0, 0};
    PGB_TRY(dft_ew(m, EW_MUL, R, P, R, res->size, 1));
    return sync_if(m, true);
}

// ---- vmp --------------------------------------------------------------------------------------------------------
extern "C" size_t pgb_vmp_prepare_tmp_bytes(const pgb_module *, uint64_t, uint64_t, uint64_t, uint64_t) { return 0; }
extern "C" size_t pgb_vmp_apply_dft_to_dft_tmp_bytes(const pgb_module *, uint64_t, uint64_t, uint64_t, uint64_t, uint64_t, uint64_t) { return 0; }

extern "C" int pgb_vmp_prepare(pgb_module *m, pgb_vmp_pmat *res, const pgb_mat_znx *a) {
    CHECK_N(res, "vmp_prepare(res)");
    CHECK_N(a, "vmp_prepare(a)");
    PGB_REQUIRE(res->rows == a->rows && res->cols_in == a->cols_in && res->cols_out == a->cols_out && res->size == a->size,
                "vmp_prepare: shape mismatch between VmpPMat and MatZnx");
    // MatZnx poly (row_i, col_i) at n*(row_i*ncols + col_i) i64 (mat_znx.rs:161-176) -> pmat poly (row_i*ncols + col_i): one
    // forward transform per polynomial, written straight into the [row][col] layout.
    const uint64_t n = m->n, pb = prep_bytes(m);
    const uint64_t polys = a->rows * a->cols_in * a->cols_out * a->size;
    key_cache_invalidate(m, res->data, polys * n * pb); // a pinned key that is prepared again loses its cached gadget forms
    LimbSet in = {(char *)a->data, n * 8, 0};
    LimbSet out = {(char *)res->data, n * pb, 0};
    if (m->flavour == PGB_NTT120) PGB_TRY(ntt120_forward(m, in, out, (int)polys, 1));
    else PGB_TRY(fft64_forward(m, in, out, (int)polys, 1));
    return sync_if(m, true);
}
// count MatZnx (a.data + b * stride_a) -> count VmpPMat (res.data + b * stride_res): the same per-polynomial forward transform as
// pgb_vmp_prepare, as ONE launch over count * polys polynomials (the batch stride of the LimbSets).  Asynchronous like every batched entry.
extern "C" int pgb_vmp_prepare_batched(pgb_module *m, pgb_vmp_pmat *res, const pgb_mat_znx *a, const pgb_batch *bt) {
    PGB_REQUIRE(bt && bt->count >= 1 && bt->count <= 65535, "vmp_prepare_batched: batch count must be in [1, 65535]");
    CHECK_N(res, "vmp_prepare_batched(res)");
    CHECK_N(a, "vmp_prepare_batched(a)");
    PGB_REQUIRE(res->rows == a->rows && res->cols_in == a->cols_in && res->cols_out == a->cols_out && res->size == a->size,
                "vmp_prepare_batched: shape mismatch between VmpPMat and MatZnx");
    const uint64_t n = m->n, pb = prep_bytes(m), B = bt->count;
    const uint64_t polys = a->rows * a->cols_in * a->cols_out * a->size;
    const uint64_t res_item = polys * n * pb, a_item = polys * n * 8;
    PGB_REQUIRE(polys >= 1 && polys * B <= 0x7fffffffull, "vmp_prepare_batched: %llu polynomials per call (must be in [1, 2^31))",
                (unsigned long long)(polys * B));
    PGB_REQUIRE(res->data && (uintptr_t)res->data % 16 == 0 && bt->stride_res % 16 == 0 && (B == 1 || bt->stride_res >= res_item),
                "vmp_prepare_batched: VmpPMat data and stride must be multiples of 16 bytes, the stride at least one matrix (%llu bytes)",
                (unsigned long long)res_item);
    PGB_REQUIRE(a->data && (uintptr_t)a->data % 8 == 0 && bt->stride_a % 8 == 0 && (B == 1 || bt->stride_a >= a_item),
                "vmp_prepare_batched: MatZnx data and stride must be multiples of 8 bytes, the stride at least one matrix (%llu bytes)",
                (unsigned long long)a_item);
    const uint64_t res_ext = batch_extent(res_item, bt->stride_res, B);
    if (ranges_overlap(res->data, res_ext, a->data, batch_extent(a_item, bt->stride_a, B))) {
        pgb_set_error("vmp_prepare_batched: res and a must not overlap");
        return PGB_ERR_ALIAS;
    }
    key_cache_invalidate(m, res->data, res_ext); // every pinned key inside the written extent loses its cached gadget forms
    LimbSet in = {(char *)a->data, n * 8, bt->stride_a};
    LimbSet out = {(char *)res->data, n * pb, bt->stride_res};
    if (m->flavour == PGB_NTT120) return ntt120_forward(m, in, out, (int)polys, (int)B);
    return fft64_forward(m, in, out, (int)polys, (int)B);
}

int vmp_apply_impl(pgb_module *m, pgb_vec_znx_dft *res, const pgb_vec_znx_dft *a, const pgb_vmp_pmat *pmat, uint64_t limb_offset,
                   const pgb_batch *bt, uint32_t pm_div) {
    CHECK_BATCH(bt);
    CHECK_N(res, "vmp_apply_dft_to_dft(res)");
    CHECK_N(a, "vmp_apply_dft_to_dft(a)");
    CHECK_N(pmat, "vmp_apply_dft_to_dft(pmat)");
    const uint64_t n = m->n, pb = prep_bytes(m), poly = n * pb;
    const uint64_t nrows = pmat->cols_in * pmat->rows, ncols = pmat->cols_out * pmat->size;
    const uint64_t a_polys = a->cols * a->size, res_polys = res->cols * res->size;
    const uint64_t off = limb_offset * pmat->cols_out; // ntt120/vmp.rs:335, fft64/vmp.rs:177
    const uint64_t row_max = umin64(nrows, a_polys);
    LimbSet R = {(char *)res->data, poly, bt->stride_res};
    if (m->flavour == PGB_NTT120) {
        const uint64_t col_max = umin64(ncols, res_polys + off); // ntt120/vmp.rs:189-190
        if (off >= col_max) return raw_limbs(m, true, R, R, poly, (uint32_t)res_polys, (uint32_t)bt->count);
        const uint64_t active = col_max - off;
        // an odd col_max short of the matrix: the reference reads the last poly's column pair with the single-column stride (:262-273);
        // reproduced verbatim by ntt120_vmp_odd_last (the columns before it are the plain product)
        const bool quirk = (col_max & 1) && col_max < ncols;
        PGB_TRY(ntt120_vmp(m, (const char *)a->data, bt->stride_a, (char *)res->data, bt->stride_res, (const char *)pmat->data,
                           bt->stride_b, (uint32_t)row_max, (uint32_t)ncols, (uint32_t)off, (uint32_t)(active - (quirk ? 1 : 0)),
                           (uint32_t)bt->count, pm_div));
        if (quirk)
            PGB_TRY(ntt120_vmp_odd_last(m, (const char *)a->data, bt->stride_a, (char *)res->data + (active - 1) * poly, bt->stride_res,
                                        (const char *)pmat->data, bt->stride_b, (uint32_t)row_max, (uint32_t)ncols, (uint32_t)(col_max - 1),
                                        (uint32_t)bt->count, pm_div));
        return raw_limbs(m, true, shift(R, active), shift(R, active), poly, (uint32_t)(res_polys - active), (uint32_t)bt->count); // :282-287
    } else {
        const uint64_t col_max = umin64(ncols, res_polys); // fft64/vmp.rs:214-215
        if (off >= col_max) return raw_limbs(m, true, R, R, poly, (uint32_t)res_polys, (uint32_t)bt->count);
        const uint64_t active = col_max - off;
        PGB_TRY(fft64_vmp(m, (const char *)a->data, bt->stride_a, (char *)res->data, bt->stride_res, (const char *)pmat->data,
                          bt->stride_b, (uint32_t)row_max, (uint32_t)ncols, (uint32_t)off, (uint32_t)active, (uint32_t)bt->count, pm_div));
        // fft64/vmp.rs:263 zeroes res[col_max..] only; polys in [col_max - off, col_max) keep their previous content
        return raw_limbs(m, true, shift(R, col_max), shift(R, col_max), poly, (uint32_t)(res_polys - col_max), (uint32_t)bt->count);
    }
}
extern "C" int pgb_vmp_apply_dft_to_dft(pgb_module *m, pgb_vec_znx_dft *res, const pgb_vec_znx_dft *a, const pgb_vmp_pmat *pmat,
                                        uint64_t limb_offset) {
    PGB_TRY(vmp_apply_impl(m, res, a, pmat, limb_offset, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vmp_apply_dft_to_dft_batched(pgb_module *m, pgb_vec_znx_dft *res, const pgb_vec_znx_dft *a, const pgb_vmp_pmat *pmat,
                                                uint64_t limb_offset, const pgb_batch *bt) {
    return vmp_apply_impl(m, res, a, pmat, limb_offset, bt);
}
// HalImpl::vmp_apply_dft_tmp_bytes / vmp_apply_dft (hal_impl.rs:626-640; poulpy-cpu-ref/src/hal_impl/family_common.rs:3-58): forward
// transform of the last min(a.cols, cols_in) columns of `a` into a scratch VecZnxDft(cols_in, min(a.size, rows)) whose leading
// columns are zero, then vmp_apply_dft_to_dft with limb_offset 0.
extern "C" size_t pgb_vmp_apply_dft_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t b_rows, uint64_t b_cols_in,
                                              uint64_t b_cols_out, uint64_t b_size) {
    (void)res_size; (void)b_cols_out; (void)b_size;
    return m->n * b_cols_in * umin64(a_size, b_rows) * prep_bytes(m) + 256;
}
extern "C" int pgb_vmp_apply_dft(pgb_module *m, pgb_vec_znx_dft *res, const pgb_vec_znx *a, const pgb_vmp_pmat *pmat, void *scratch,
                                 size_t scratch_len) {
    CHECK_N(res, "vmp_apply_dft(res)");
    CHECK_N(a, "vmp_apply_dft(a)");
    CHECK_N(pmat, "vmp_apply_dft(pmat)");
    const uint64_t n = m->n, pb = prep_bytes(m);
    const uint64_t cols_to_copy = umin64(a->cols, pmat->cols_in), a_start_col = a->cols - cols_to_copy;
    const uint64_t a_dft_size = umin64(a->size, pmat->rows), offset = pmat->cols_in - cols_to_copy;
    const size_t need = pgb_vmp_apply_dft_tmp_bytes(m, res->size, a->size, pmat->rows, pmat->cols_in, pmat->cols_out, pmat->size);
    if (scratch_len < need) {
        pgb_set_error("vmp_apply_dft: scratch of %zu bytes < required %zu", scratch_len, need);
        return PGB_ERR_SCRATCH;
    }
    char *sp = (char *)(((uintptr_t)scratch + 255) & ~(uintptr_t)255);
    pgb_vec_znx_dft a_dft = {sp, n, pmat->cols_in, a_dft_size, a_dft_size};
    if (a_dft_size) {
        for (uint64_t j = 0; j < offset; j++) PGB_TRY(dft_zero_impl(m, &a_dft, j, &ONE));
        for (uint64_t j = 0; j < cols_to_copy; j++) PGB_TRY(dft_apply_impl(m, 1, 0, &a_dft, offset + j, a, a_start_col + j, &ONE));
    }
    (void)pb;
    PGB_TRY(vmp_apply_impl(m, res, &a_dft, pmat, 0, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vmp_zero(pgb_module *m, pgb_vmp_pmat *res) {
    CHECK_N(res, "vmp_zero(res)");
    key_cache_invalidate(m, res->data, pgb_bytes_of_vmp_pmat(m, res->rows, res->cols_in, res->cols_out, res->size));
    PGB_CHECK_CUDA(cudaMemsetAsync(res->data, 0, pgb_bytes_of_vmp_pmat(m, res->rows, res->cols_in, res->cols_out, res->size), m->stream));
    return sync_if(m, true);
}

// ---- vec_znx_big --------------------------------------------------------------------------------------------------
extern "C" size_t pgb_vec_znx_big_normalize_tmp_bytes(const pgb_module *) { return 0; }

int big_normalize_impl(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, int64_t res_offset, uint64_t res_col,
                       const pgb_vec_znx_big *a, uint64_t a_base2k, uint64_t a_col, int op, bool a_is_big, const pgb_batch *bt) {
    CHECK_BATCH(bt);
    CHECK_N(res, "normalize(res)");
    CHECK_N(a, "normalize(a)");
    CHECK_COL(res, res_col, "normalize(res)");
    CHECK_COL(a, a_col, "normalize(a)");
    const uint64_t n = m->n;
    const bool i128big = a_is_big && m->flavour == PGB_NTT120;
    const uint64_t ab = i128big ? 16 : 8;
    PGB_REQUIRE(op == 0 || i128big, "normalize_{add,sub}_assign exists only for the NTT120 big type in the reference");
    LimbSet R = {(char *)res->data + limb_off(n, res->cols, res_col, 0, 8), res->cols * n * 8, bt->stride_res};
    LimbSet A = {(char *)a->data + limb_off(n, a->cols, a_col, 0, ab), a->cols * n * ab, bt->stride_a};
    return big_normalize(m, i128big, R, (int)res->size, (int)res_base2k, res_offset, A, (int)a->size, (int)a_base2k, op,
                         (uint32_t)bt->count);
}
extern "C" int pgb_vec_znx_big_normalize(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, int64_t res_offset, uint64_t res_col,
                                         const pgb_vec_znx_big *a, uint64_t a_base2k, uint64_t a_col) {
    PGB_TRY(big_normalize_impl(m, res, res_base2k, res_offset, res_col, a, a_base2k, a_col, 0, true, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_big_normalize_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, int64_t res_offset,
                                                 uint64_t res_col, const pgb_vec_znx_big *a, uint64_t a_base2k, uint64_t a_col,
                                                 const pgb_batch *bt) {
    return big_normalize_impl(m, res, res_base2k, res_offset, res_col, a, a_base2k, a_col, 0, true, bt);
}
extern "C" int pgb_vec_znx_big_normalize_add_assign(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, int64_t res_offset,
                                                    uint64_t res_col, const pgb_vec_znx_big *a, uint64_t a_base2k, uint64_t a_col) {
    PGB_TRY(big_normalize_impl(m, res, res_base2k, res_offset, res_col, a, a_base2k, a_col, +1, true, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_big_normalize_sub_assign(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, int64_t res_offset,
                                                    uint64_t res_col, const pgb_vec_znx_big *a, uint64_t a_base2k, uint64_t a_col) {
    PGB_TRY(big_normalize_impl(m, res, res_base2k, res_offset, res_col, a, a_base2k, a_col, -1, true, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_normalize(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, int64_t res_offset, uint64_t res_col,
                                     const pgb_vec_znx *a, uint64_t a_base2k, uint64_t a_col) {
    PGB_TRY(big_normalize_impl(m, res, res_base2k, res_offset, res_col, a, a_base2k, a_col, 0, false, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_normalize_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, int64_t res_offset, uint64_t res_col,
                                             const pgb_vec_znx *a, uint64_t a_base2k, uint64_t a_col, const pgb_batch *bt) {
    return big_normalize_impl(m, res, res_base2k, res_offset, res_col, a, a_base2k, a_col, 0, false, bt);
}

int big_add_small_impl(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col, const pgb_batch *bt) {
    CHECK_BATCH(bt);
    CHECK_N(res, "vec_znx_big_add_small_assign(res)");
    CHECK_N(a, "vec_znx_big_add_small_assign(a)");
    CHECK_COL(res, res_col, "vec_znx_big_add_small_assign(res)");
    CHECK_COL(a, a_col, "vec_znx_big_add_small_assign(a)");
    const uint64_t n = m->n, bb = big_bytes(m);
    LimbSet R = {(char *)res->data + limb_off(n, res->cols, res_col, 0, bb), res->cols * n * bb, bt->stride_res};
    LimbSet A = {(char *)a->data + limb_off(n, a->cols, a_col, 0, 8), a->cols * n * 8, bt->stride_a};
    return big_ew(m, m->flavour == PGB_NTT120, BIG_ADD_SMALL, R, A, (uint32_t)umin64(res->size, a->size), (uint32_t)bt->count);
}
// vec_znx_big_sub_small_assign / _sub_small_negate_assign (ntt120/vec_znx_big.rs:1285-1318 and the FFT64 twins): res -= a ; res = a - res
int big_small_op_impl(pgb_module *m, int op, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col, const pgb_batch *bt) {
    if (op == BIG_ADD_SMALL) return big_add_small_impl(m, res, res_col, a, a_col, bt);
    CHECK_BATCH(bt);
    CHECK_N(res, "vec_znx_big_sub_small(res)");
    CHECK_N(a, "vec_znx_big_sub_small(a)");
    CHECK_COL(res, res_col, "vec_znx_big_sub_small(res)");
    CHECK_COL(a, a_col, "vec_znx_big_sub_small(a)");
    const uint64_t n = m->n, bb = big_bytes(m), mn = umin64(res->size, a->size);
    LimbSet R = {(char *)res->data + limb_off(n, res->cols, res_col, 0, bb), res->cols * n * bb, bt->stride_res};
    LimbSet A = {(char *)a->data + limb_off(n, a->cols, a_col, 0, 8), a->cols * n * 8, bt->stride_a};
    PGB_TRY(big_ew(m, m->flavour == PGB_NTT120, op, R, A, (uint32_t)mn, (uint32_t)bt->count));
    if (op == BIG_SUB_SMALL_NEG && res->size > a->size) // (:1315-1317) the remaining limbs of res are negated
        PGB_TRY(big_ew(m, m->flavour == PGB_NTT120, BIG_NEG, shift(R, a->size), shift(R, a->size), (uint32_t)(res->size - a->size), (uint32_t)bt->count));
    return PGB_OK;
}
extern "C" int pgb_vec_znx_big_sub_small_assign(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col) {
    PGB_TRY(big_small_op_impl(m, BIG_SUB_SMALL, res, res_col, a, a_col, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_big_sub_small_negate_assign(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col) {
    PGB_TRY(big_small_op_impl(m, BIG_SUB_SMALL_NEG, res, res_col, a, a_col, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_big_add_small_assign(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col) {
    PGB_TRY(big_add_small_impl(m, res, res_col, a, a_col, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_big_add_small_assign_batched(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx *a,
                                                        uint64_t a_col, const pgb_batch *bt) {
    return big_add_small_impl(m, res, res_col, a, a_col, bt);
}
extern "C" int pgb_vec_znx_big_from_small(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col) {
    CHECK_N(res, "vec_znx_big_from_small(res)");
    CHECK_N(a, "vec_znx_big_from_small(a)");
    CHECK_COL(res, res_col, "vec_znx_big_from_small(res)");
    CHECK_COL(a, a_col, "vec_znx_big_from_small(a)");
    const uint64_t n = m->n, bb = big_bytes(m);
    LimbSet R = {(char *)res->data + limb_off(n, res->cols, res_col, 0, bb), res->cols * n * bb, 0};
    LimbSet A = {(char *)a->data + limb_off(n, a->cols, a_col, 0, 8), a->cols * n * 8, 0};
    const uint64_t mn = umin64(res->size, a->size);
    PGB_TRY(big_ew(m, m->flavour == PGB_NTT120, BIG_FROM_SMALL, R, A, (uint32_t)mn, 1));
    PGB_TRY(big_ew(m, m->flavour == PGB_NTT120, BIG_ZERO, shift(R, mn), shift(R, mn), (uint32_t)(res->size - mn), 1));
    return sync_if(m, true);
}

// batched twin of pgb_vec_znx_rotate (stream-ordered; one p for the whole batch)
extern "C" int pgb_vec_znx_rotate_batched(pgb_module *m, int64_t p, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col,
                                          const pgb_batch *bt) {
    CHECK_BATCH(bt);
    CHECK_N(res, "vec_znx_rotate(res)");
    CHECK_N(a, "vec_znx_rotate(a)");
    CHECK_COL(res, res_col, "vec_znx_rotate(res)");
    CHECK_COL(a, a_col, "vec_znx_rotate(a)");
    PGB_REQUIRE_DISJOINT(res, bt->stride_res, a, bt->stride_a, bt->count, 8, "vec_znx_rotate");
    const uint64_t n = m->n;
    LimbSet R = {(char *)res->data + limb_off(n, res->cols, res_col, 0, 8), res->cols * n * 8, bt->stride_res};
    LimbSet A = {(char *)a->data + limb_off(n, a->cols, a_col, 0, 8), a->cols * n * 8, bt->stride_a};
    const uint64_t mn = umin64(res->size, a->size);
    PGB_TRY(znx_rotate(m, R, A, p, nullptr, 0, (uint32_t)mn, (uint32_t)bt->count));
    return raw_limbs(m, true, shift(R, mn), shift(R, mn), n * 8, (uint32_t)(res->size - mn), (uint32_t)bt->count);
}
// strided device-to-device copy on the module's stream: `count` rows of `width` bytes (glwe_copy between containers of different strides)
extern "C" int pgb_memcpy_d2d_strided(pgb_module *m, void *dst, uint64_t dst_stride, const void *src, uint64_t src_stride, uint64_t width,
                                      uint64_t count) {
    PGB_CHECK_CUDA(cudaMemcpy2DAsync(dst, dst_stride, src, src_stride, width, count, cudaMemcpyDeviceToDevice, m->stream));
    return PGB_OK;
}
extern "C" int pgb_vec_znx_rotate(pgb_module *m, int64_t p, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col) {
    CHECK_N(res, "vec_znx_rotate(res)");
    CHECK_N(a, "vec_znx_rotate(a)");
    CHECK_COL(res, res_col, "vec_znx_rotate(res)");
    CHECK_COL(a, a_col, "vec_znx_rotate(a)");
    PGB_REQUIRE_DISJOINT(res, 0, a, 0, 1, 8, "vec_znx_rotate");
    const uint64_t n = m->n;
    LimbSet R = {(char *)res->data + limb_off(n, res->cols, res_col, 0, 8), res->cols * n * 8, 0};
    LimbSet A = {(char *)a->data + limb_off(n, a->cols, a_col, 0, 8), a->cols * n * 8, 0};
    const uint64_t mn = umin64(res->size, a->size);
    PGB_TRY(znx_rotate(m, R, A, p, nullptr, 0, (uint32_t)mn, 1));
    PGB_TRY(raw_limbs(m, true, shift(R, mn), shift(R, mn), n * 8, (uint32_t)(res->size - mn), 1));
    return sync_if(m, true);
}

// ---- coefficient-domain helpers used by execute_standard (SURVEY 8f N1) --------------------------------------------------------
// vec_znx_add_assign / vec_znx_sub_assign (reference/vec_znx/add.rs:60-82, sub.rs:60-82): the first min(res.size, a.size) limbs
static int znx_assign_impl(pgb_module *m, int op, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col, const pgb_batch *bt) {
    CHECK_BATCH(bt);
    CHECK_N(res, "vec_znx_add/sub_assign(res)");
    CHECK_N(a, "vec_znx_add/sub_assign(a)");
    CHECK_COL(res, res_col, "vec_znx_add/sub_assign(res)");
    CHECK_COL(a, a_col, "vec_znx_add/sub_assign(a)");
    const uint64_t n = m->n;
    LimbSet R = {(char *)res->data + limb_off(n, res->cols, res_col, 0, 8), res->cols * n * 8, bt->stride_res};
    LimbSet A = {(char *)a->data + limb_off(n, a->cols, a_col, 0, 8), a->cols * n * 8, bt->stride_a};
    return znx_ew(m, op, R, A, 0, nullptr, 0, (uint32_t)umin64(res->size, a->size), (uint32_t)bt->count);
}
extern "C" int pgb_vec_znx_add_assign(pgb_module *m, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col) {
    PGB_TRY(znx_assign_impl(m, 0, res, res_col, a, a_col, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_add_assign_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col,
                                              const pgb_batch *bt) {
    return znx_assign_impl(m, 0, res, res_col, a, a_col, bt);
}
extern "C" int pgb_vec_znx_sub_assign(pgb_module *m, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col) {
    PGB_TRY(znx_assign_impl(m, 1, res, res_col, a, a_col, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_sub_assign_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col,
                                              const pgb_batch *bt) {
    return znx_assign_impl(m, 1, res, res_col, a, a_col, bt);
}
// vec_znx_mul_xp_minus_one (reference/vec_znx/mul_xp_minus_one.rs:13-22): res = rotate(p, a) - a on the common limbs, zero the rest
// (rotate zero-fills, sub_assign only touches the common limbs).  res and a must not alias.
extern "C" int pgb_vec_znx_mul_xp_minus_one(pgb_module *m, int64_t p, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col) {
    CHECK_N(res, "vec_znx_mul_xp_minus_one(res)");
    CHECK_N(a, "vec_znx_mul_xp_minus_one(a)");
    CHECK_COL(res, res_col, "vec_znx_mul_xp_minus_one(res)");
    CHECK_COL(a, a_col, "vec_znx_mul_xp_minus_one(a)");
    PGB_REQUIRE_DISJOINT(res, 0, a, 0, 1, 8, "vec_znx_mul_xp_minus_one");
    const uint64_t n = m->n, mn = umin64(res->size, a->size);
    LimbSet R = {(char *)res->data + limb_off(n, res->cols, res_col, 0, 8), res->cols * n * 8, 0};
    LimbSet A = {(char *)a->data + limb_off(n, a->cols, a_col, 0, 8), a->cols * n * 8, 0};
    PGB_TRY(znx_ew(m, 2, R, A, p, nullptr, 0, (uint32_t)mn, 1));
    PGB_TRY(raw_limbs(m, true, shift(R, mn), shift(R, mn), n * 8, (uint32_t)(res->size - mn), 1));
    return sync_if(m, true);
}
// vec_znx_normalize_assign (reference/vec_znx/normalize.rs:403-425): in place, equal base2k, offset 0
extern "C" int pgb_vec_znx_normalize_assign(pgb_module *m, uint64_t base2k, pgb_vec_znx *res, uint64_t res_col) {
    PGB_TRY(big_normalize_impl(m, res, base2k, 0, res_col, res, base2k, res_col, 0, false, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_normalize_assign_batched(pgb_module *m, uint64_t base2k, pgb_vec_znx *res, uint64_t res_col, const pgb_batch *bt) {
    pgb_batch b2 = {bt->count, bt->stride_res, bt->stride_res, 0};
    return big_normalize_impl(m, res, base2k, 0, res_col, res, base2k, res_col, 0, false, &b2);
}

// ---- bivariate convolution (HalImpl::cnv_*, hal_impl.rs:670-754; kernels in cnv.cu) --------------------------------------------
extern "C" size_t pgb_bytes_of_cnv_pvec_left(const pgb_module *m, uint64_t cols, uint64_t size) { return m->n * cols * size * prep_bytes(m); }
extern "C" size_t pgb_bytes_of_cnv_pvec_right(const pgb_module *m, uint64_t cols, uint64_t size) { return m->n * cols * size * prep_bytes(m); }
extern "C" size_t pgb_cnv_prepare_left_tmp_bytes(const pgb_module *, uint64_t, uint64_t) { return 0; }
extern "C" size_t pgb_cnv_prepare_right_tmp_bytes(const pgb_module *, uint64_t, uint64_t) { return 0; }
extern "C" size_t pgb_cnv_prepare_self_tmp_bytes(const pgb_module *, uint64_t, uint64_t) { return 0; }
extern "C" size_t pgb_cnv_apply_dft_tmp_bytes(const pgb_module *, uint64_t, uint64_t, uint64_t, uint64_t) { return 0; }
extern "C" size_t pgb_cnv_pairwise_apply_dft_tmp_bytes(const pgb_module *, uint64_t, uint64_t, uint64_t, uint64_t) { return 0; }
extern "C" size_t pgb_cnv_by_const_apply_tmp_bytes(const pgb_module *, uint64_t, uint64_t, uint64_t, uint64_t) { return 0; }

// cnv_prepare_left / right (ntt120/convolution.rs:66-157, fft64/convolution.rs:13-73): every column of res; limbs [0, min(res.size,
// a.size)) transformed, the last active one ANDed with `mask` first, the remaining limbs zero
int cnv_prepare_impl(pgb_module *m, pgb_vec_znx_dft *res, const pgb_vec_znx *a, int64_t mask, const pgb_batch *bt) {
    CHECK_BATCH(bt);
    CHECK_N(res, "cnv_prepare(res)");
    CHECK_N(a, "cnv_prepare(a)");
    PGB_REQUIRE(a->cols >= res->cols, "cnv_prepare: a has %llu columns, res %llu", (unsigned long long)a->cols, (unsigned long long)res->cols);
    const uint64_t n = m->n, pb = prep_bytes(m), min_size = umin64(res->size, a->size);
    for (uint64_t col = 0; col < res->cols; col++) {
        LimbSet in = {(char *)a->data + limb_off(n, a->cols, col, 0, 8), a->cols * n * 8, bt->stride_a};
        LimbSet out = dft_col(m, res, col, 0, bt->stride_res);
        if (min_size > 1) {
            if (m->flavour == PGB_NTT120) PGB_TRY(ntt120_forward(m, in, out, (int)(min_size - 1), (int)bt->count));
            else PGB_TRY(fft64_forward(m, in, out, (int)(min_size - 1), (int)bt->count));
        }
        if (min_size > 0) {
            LimbSet il = in, ol = out;
            il.base += (min_size - 1) * in.limb_stride;
            ol.base += (min_size - 1) * out.limb_stride;
            if (m->flavour == PGB_NTT120) PGB_TRY(ntt120_forward(m, il, ol, 1, (int)bt->count, mask));
            else PGB_TRY(fft64_forward(m, il, ol, 1, (int)bt->count, mask));
        }
        PGB_TRY(raw_limbs(m, true, shift(out, min_size), shift(out, min_size), n * pb, (uint32_t)(res->size - min_size), (uint32_t)bt->count));
    }
    return PGB_OK;
}
extern "C" int pgb_cnv_prepare_left(pgb_module *m, pgb_vec_znx_dft *res, const pgb_vec_znx *a, int64_t mask) {
    PGB_TRY(cnv_prepare_impl(m, res, a, mask, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_cnv_prepare_right(pgb_module *m, pgb_vec_znx_dft *res, const pgb_vec_znx *a, int64_t mask) {
    PGB_TRY(cnv_prepare_impl(m, res, a, mask, &ONE));
    return sync_if(m, true);
}
// cnv_prepare_self (ntt120/convolution.rs:177-236): both operands from one input; here both layouts coincide
extern "C" int pgb_cnv_prepare_self(pgb_module *m, pgb_vec_znx_dft *left, pgb_vec_znx_dft *right, const pgb_vec_znx *a, int64_t mask) {
    PGB_REQUIRE(left->cols == right->cols && left->size == right->size, "cnv_prepare_self: left and right must have the same shape");
    PGB_TRY(cnv_prepare_impl(m, left, a, mask, &ONE));
    PGB_CHECK_CUDA(cudaMemcpyAsync(right->data, left->data, m->n * left->cols * left->size * prep_bytes(m), cudaMemcpyDeviceToDevice, m->stream));
    return sync_if(m, true);
}
static int cnv_apply_impl(pgb_module *m, uint64_t cnv_offset, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a, uint64_t a_i,
                          uint64_t a_j, const pgb_vec_znx_dft *b, uint64_t b_i, uint64_t b_j, const pgb_batch *bt) {
    CHECK_BATCH(bt);
    CHECK_N(res, "cnv_apply_dft(res)");
    CHECK_N(a, "cnv_apply_dft(a)");
    CHECK_N(b, "cnv_apply_dft(b)");
    CHECK_COL(res, res_col, "cnv_apply_dft(res)");
    CHECK_COL(a, a_i, "cnv_apply_dft(a)");
    CHECK_COL(a, a_j, "cnv_apply_dft(a)");
    CHECK_COL(b, b_i, "cnv_apply_dft(b)");
    CHECK_COL(b, b_j, "cnv_apply_dft(b)");
    LimbSet none = {nullptr, 0, 0};
    const bool pair = a_i != a_j;
    return cnv_apply(m, dft_col(m, res, res_col, 0, bt->stride_res), (int)res->size, dft_col(m, a, a_i, 0, bt->stride_a),
                     pair ? dft_col(m, a, a_j, 0, bt->stride_a) : none, (int)a->size, dft_col(m, b, b_i, 0, bt->stride_b),
                     pair ? dft_col(m, b, b_j, 0, bt->stride_b) : none, (int)b->size, cnv_offset, (uint32_t)bt->count);
}
extern "C" int pgb_cnv_apply_dft(pgb_module *m, uint64_t cnv_offset, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a,
                                 uint64_t a_col, const pgb_vec_znx_dft *b, uint64_t b_col) {
    PGB_TRY(cnv_apply_impl(m, cnv_offset, res, res_col, a, a_col, a_col, b, b_col, b_col, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_cnv_apply_dft_batched(pgb_module *m, uint64_t cnv_offset, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a,
                                         uint64_t a_col, const pgb_vec_znx_dft *b, uint64_t b_col, const pgb_batch *bt) {
    return cnv_apply_impl(m, cnv_offset, res, res_col, a, a_col, a_col, b, b_col, b_col, bt);
}
// cnv_pairwise_apply_dft (ntt120/convolution.rs:441-557): (a[:, i] + a[:, j]) x (b[:, i] + b[:, j]); i == j is the plain product
extern "C" int pgb_cnv_pairwise_apply_dft(pgb_module *m, uint64_t cnv_offset, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a,
                                          const pgb_vec_znx_dft *b, uint64_t col_i, uint64_t col_j) {
    PGB_TRY(cnv_apply_impl(m, cnv_offset, res, res_col, a, col_i, col_j, b, col_i, col_j, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_cnv_pairwise_apply_dft_batched(pgb_module *m, uint64_t cnv_offset, pgb_vec_znx_dft *res, uint64_t res_col,
                                                  const pgb_vec_znx_dft *a, const pgb_vec_znx_dft *b, uint64_t col_i, uint64_t col_j,
                                                  const pgb_batch *bt) {
    return cnv_apply_impl(m, cnv_offset, res, res_col, a, col_i, col_j, b, col_i, col_j, bt);
}
// cnv_by_const_apply (ntt120/convolution.rs:361-410, fft64/convolution.rs:144-191): `b` is a HOST array of b_size limb constants
extern "C" int pgb_cnv_by_const_apply(pgb_module *m, uint64_t cnv_offset, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx *a,
                                      uint64_t a_col, const int64_t *b, uint64_t b_size) {
    CHECK_N(res, "cnv_by_const_apply(res)");
    CHECK_N(a, "cnv_by_const_apply(a)");
    CHECK_COL(res, res_col, "cnv_by_const_apply(res)");
    CHECK_COL(a, a_col, "cnv_by_const_apply(a)");
    PGB_REQUIRE(b_size <= 4096, "cnv_by_const_apply: b_size too large");
    const uint64_t n = m->n, bb = big_bytes(m);
    long long *b_dev = nullptr;
    if (b_size) {
        PGB_CHECK_CUDA(cudaMallocAsync(&b_dev, b_size * 8, m->stream));
        PGB_CHECK_CUDA(cudaMemcpyAsync(b_dev, b, b_size * 8, cudaMemcpyHostToDevice, m->stream));
    }
    LimbSet R = {(char *)res->data + limb_off(n, res->cols, res_col, 0, bb), res->cols * n * bb, 0};
    LimbSet A = {(char *)a->data + limb_off(n, a->cols, a_col, 0, 8), a->cols * n * 8, 0};
    int s = cnv_by_const(m, R, (int)res->size, A, (int)a->size, b_dev, (int)b_size, cnv_offset, 1);
    if (b_dev) cudaFreeAsync(b_dev, m->stream);
    PGB_TRY(s);
    return sync_if(m, true);
}

// ---- vec_znx_automorphism (reference/vec_znx/automorphism.rs:9-38; SURVEY 8f N4) ---------------------------------------------------
static int automorphism_impl(pgb_module *m, int64_t p, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col, const pgb_batch *bt) {
    CHECK_BATCH(bt);
    CHECK_N(res, "vec_znx_automorphism(res)");
    CHECK_N(a, "vec_znx_automorphism(a)");
    CHECK_COL(res, res_col, "vec_znx_automorphism(res)");
    CHECK_COL(a, a_col, "vec_znx_automorphism(a)");
    PGB_REQUIRE_DISJOINT(res, bt->stride_res, a, bt->stride_a, bt->count, 8, "vec_znx_automorphism");
    PGB_REQUIRE((p & 1) != 0, "vec_znx_automorphism: the Galois element must be odd");
    const uint64_t n = m->n, mn = umin64(res->size, a->size);
    LimbSet R = {(char *)res->data + limb_off(n, res->cols, res_col, 0, 8), res->cols * n * 8, bt->stride_res};
    LimbSet A = {(char *)a->data + limb_off(n, a->cols, a_col, 0, 8), a->cols * n * 8, bt->stride_a};
    PGB_TRY(znx_automorphism(m, R, A, p, (uint32_t)mn, (uint32_t)bt->count));
    return raw_limbs(m, true, shift(R, mn), shift(R, mn), n * 8, (uint32_t)(res->size - mn), (uint32_t)bt->count);
}
// vec_znx_big_automorphism (ntt120/vec_znx_big.rs:1462-1497, fft64/vec_znx_big.rs:144-170): out of place, limbs of res beyond a.size zeroed
int big_automorphism_impl(pgb_module *m, int64_t p, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx_big *a, uint64_t a_col,
                          const pgb_batch *bt) {
    CHECK_BATCH(bt);
    CHECK_N(res, "vec_znx_big_automorphism(res)");
    CHECK_N(a, "vec_znx_big_automorphism(a)");
    CHECK_COL(res, res_col, "vec_znx_big_automorphism(res)");
    CHECK_COL(a, a_col, "vec_znx_big_automorphism(a)");
    PGB_REQUIRE_DISJOINT(res, bt->stride_res, a, bt->stride_a, bt->count, big_bytes(m), "vec_znx_big_automorphism");
    PGB_REQUIRE((p & 1) != 0, "vec_znx_big_automorphism: the Galois element must be odd");
    const uint64_t n = m->n, bb = big_bytes(m), mn = umin64(res->size, a->size);
    LimbSet R = {(char *)res->data + limb_off(n, res->cols, res_col, 0, bb), res->cols * n * bb, bt->stride_res};
    LimbSet A = {(char *)a->data + limb_off(n, a->cols, a_col, 0, bb), a->cols * n * bb, bt->stride_a};
    PGB_TRY(znx_automorphism(m, R, A, p, (uint32_t)mn, (uint32_t)bt->count, m->flavour == PGB_NTT120));
    return raw_limbs(m, true, shift(R, mn), shift(R, mn), n * bb, (uint32_t)(res->size - mn), (uint32_t)bt->count);
}
extern "C" int pgb_vec_znx_big_automorphism(pgb_module *m, int64_t p, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx_big *a,
                                            uint64_t a_col) {
    PGB_TRY(big_automorphism_impl(m, p, res, res_col, a, a_col, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_big_automorphism_batched(pgb_module *m, int64_t p, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx_big *a,
                                                    uint64_t a_col, const pgb_batch *bt) {
    return big_automorphism_impl(m, p, res, res_col, a, a_col, bt);
}
// vec_znx_big_automorphism_assign (ntt120/vec_znx_big.rs:1499-1529): the reference permutes through an n-element tmp; here the column is
// staged in a stream-ordered temporary and permuted back
extern "C" size_t pgb_vec_znx_big_automorphism_assign_tmp_bytes(const pgb_module *m) { return m->n * big_bytes(m); }
extern "C" int pgb_vec_znx_big_automorphism_assign(pgb_module *m, int64_t p, pgb_vec_znx_big *res, uint64_t res_col) {
    CHECK_N(res, "vec_znx_big_automorphism_assign(res)");
    CHECK_COL(res, res_col, "vec_znx_big_automorphism_assign(res)");
    PGB_REQUIRE((p & 1) != 0, "vec_znx_big_automorphism_assign: the Galois element must be odd");
    const uint64_t n = m->n, bb = big_bytes(m);
    if (res->size == 0) return PGB_OK;
    char *tmp = nullptr;
    PGB_CHECK_CUDA(cudaMallocAsync(&tmp, res->size * n * bb, m->stream));
    LimbSet R = {(char *)res->data + limb_off(n, res->cols, res_col, 0, bb), res->cols * n * bb, 0};
    LimbSet Tm = {tmp, n * bb, 0};
    int s = raw_limbs(m, false, Tm, R, n * bb, (uint32_t)res->size, 1);
    if (s == PGB_OK) s = znx_automorphism(m, R, Tm, p, (uint32_t)res->size, 1, m->flavour == PGB_NTT120);
    cudaFreeAsync(tmp, m->stream);
    PGB_TRY(s);
    return sync_if(m, true);
}

// vec_znx_rsh_assign (reference/vec_znx/shift.rs:186-243)
int rsh_assign_impl(pgb_module *m, uint64_t base2k, uint64_t k, pgb_vec_znx *res, uint64_t res_col, const pgb_batch *bt) {
    CHECK_BATCH(bt);
    CHECK_N(res, "vec_znx_rsh_assign(res)");
    CHECK_COL(res, res_col, "vec_znx_rsh_assign(res)");
    PGB_REQUIRE(base2k >= 1 && base2k <= 63, "vec_znx_rsh_assign: base2k must be in [1, 63]");
    PGB_REQUIRE(div_ceil64(k, base2k) <= res->size, "vec_znx_rsh_assign: shift of %llu bits exceeds the %llu limbs of res (the reference panics)",
                (unsigned long long)k, (unsigned long long)res->size);
    const uint64_t n = m->n;
    LimbSet R = {(char *)res->data + limb_off(n, res->cols, res_col, 0, 8), res->cols * n * 8, bt->stride_res};
    return znx_rsh_assign(m, R, (int)res->size, (int)base2k, (int)k, (uint32_t)bt->count);
}
extern "C" int pgb_vec_znx_rsh_assign(pgb_module *m, uint64_t base2k, uint64_t k, pgb_vec_znx *res, uint64_t res_col) {
    PGB_TRY(rsh_assign_impl(m, base2k, k, res, res_col, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_rsh_assign_batched(pgb_module *m, uint64_t base2k, uint64_t k, pgb_vec_znx *res, uint64_t res_col, const pgb_batch *bt) {
    return rsh_assign_impl(m, base2k, k, res, res_col, bt);
}

extern "C" int pgb_vec_znx_automorphism(pgb_module *m, int64_t p, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col) {
    PGB_TRY(automorphism_impl(m, p, res, res_col, a, a_col, &ONE));
    return sync_if(m, true);
}
extern "C" int pgb_vec_znx_automorphism_batched(pgb_module *m, int64_t p, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col,
                                                const pgb_batch *bt) {
    return automorphism_impl(m, p, res, res_col, a, a_col, bt);
}
