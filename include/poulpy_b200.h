/*
 * poulpy_b200.h -- C ABI of the B200-native poulpy-hal backend (libpoulpy_b200.so).
 *
 * This is the drop-in boundary for the hot path of phantomzone-org/poulpy v0.5.0: one
 * `extern "C"` symbol per hot `unsafe trait HalImpl<BE>` method
 * (poulpy-hal/src/oep/hal_impl.rs:25-755), taking plain pointers and sizes.  A Rust backend
 * crate `poulpy-gpu-b200` binds these one-to-one (see INTEGRATION.md for the `extern "C"` block
 * and the `unsafe impl HalImpl<B200Ntt120> for B200Ntt120` stubs).  All paths below are relative
 * to the reference root; "R#" / "F#" / "C#" are the SURVEY.md section 8(a) rows.
 *
 * Conventions
 *  - Every function returns 0 on success, a negative pgb_status otherwise; pgb_last_error()
 *    returns the message (thread-local).  The Rust shim turns non-zero into panic!, matching the
 *    reference's assert!/panic! error model (hal_defaults/scratch.rs:79, ntt.rs:223-227).
 *  - Layout descriptors mirror the reference's #[repr(C)] structs field for field; `data` must be
 *    device-accessible (pgb_alloc_bytes = CUDA managed memory, host-dereferenceable as the
 *    reference's `DataRef: AsRef<[u8]>` requires; pgb_alloc_device_bytes = plain device memory).
 *    Limb j of column i starts at scalar offset n*(j*cols+i) (layouts/znx_base.rs:57-84).
 *  - The non-batched entry points are logically synchronous (complete before returning:
 *    poulpy-hal/docs/backend_safety_contract.md "Synchronization").  The *_batched twins run the
 *    same operation on `count` independent operands laid out `stride` bytes apart, enqueue on the
 *    module's stream and return immediately; call pgb_module_sync() before touching results.
 *  - The backend owns the byte layout of the prepared types (Backend::ScalarPrep / ScalarBig are
 *    backend-chosen, layouts/module.rs:28-70):
 *      NTT120 flavour: ScalarPrep = 16 B  (4 x u32 canonical residues mod Q[k]; a DFT limb is
 *                      four planes [k][n] of u32 in the reference's bit-reversed frequency order),
 *                      ScalarBig  = 16 B  (little-endian i128), VmpPMat = [row][col][k][n] u32.
 *      FFT64  flavour: ScalarPrep = 8 B (f64, limb = [re(m) | im(m)], reference frequency order),
 *                      ScalarBig  = 8 B (i64), VmpPMat = [row][col][re(m) | im(m)].
 *  - No CPU fallback exists: without a CUDA device pgb_module_new fails.
 */
#ifndef POULPY_B200_H
#define POULPY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum { PGB_NTT120 = 0, PGB_FFT64 = 1 } pgb_flavour;

typedef enum {
    PGB_OK = 0,
    PGB_ERR_SHAPE = -1,   /* shape / argument violation (reference: assert!/debug_assert!) */
    PGB_ERR_CUDA = -2,    /* CUDA runtime error */
    PGB_ERR_ALIAS = -3,   /* forbidden aliasing (backend_safety_contract.md "Aliasing") */
    PGB_ERR_SCRATCH = -4, /* scratch too small (reference: assert!(scratch.available() >= ...)) */
    PGB_ERR_UNSUPPORTED = -5
} pgb_status;

/* Opaque module handle = `Module<B>`'s `Handle` (layouts/module.rs:84-104, oep/hal_impl.rs:320). */
typedef struct pgb_module pgb_module;

/* layouts/vec_znx.rs:33-41, vec_znx_dft.rs:25-34, vec_znx_big.rs:25-33 (same five fields). */
typedef struct { void *data; uint64_t n, cols, size, max_size; } pgb_vec_znx;
typedef pgb_vec_znx pgb_vec_znx_dft;
typedef pgb_vec_znx pgb_vec_znx_big;
/* layouts/svp_ppol.rs:23-28 and layouts/scalar_znx.rs (data, n, cols). */
typedef struct { void *data; uint64_t n, cols; } pgb_svp_ppol;
typedef pgb_svp_ppol pgb_scalar_znx;
/* layouts/vmp_pmat.rs:25-33 (data, n, size, rows, cols_in, cols_out) and layouts/mat_znx.rs:28-36. */
typedef struct { void *data; uint64_t n, size, rows, cols_in, cols_out; } pgb_vmp_pmat;
typedef pgb_vmp_pmat pgb_mat_znx;

/* Batch descriptor of the *_batched twins: operand x of item b lives at x.data + b*stride_x bytes.
 * A stride of 0 shares the operand across the batch (e.g. one prepared key for all ciphertexts). */
typedef struct { uint64_t count; uint64_t stride_res, stride_a, stride_b; } pgb_batch;

const char *pgb_last_error(void);
int pgb_device_count(void);

/* ---- module (HalImpl::new, oep/hal_impl.rs:320; Backend::destroy, layouts/module.rs:260-266) ---- */
int pgb_module_new(uint64_t n, int flavour, int device, pgb_module **out);
void pgb_module_destroy(pgb_module *m);
uint64_t pgb_module_n(const pgb_module *m);
int pgb_module_flavour(const pgb_module *m);
/* Use an externally owned CUDA stream (e.g. torch's current stream) for all launches; 0 = own stream. */
int pgb_module_set_stream(pgb_module *m, void *cuda_stream);
int pgb_module_sync(pgb_module *m);
/* Route / tuning knobs of one module (test and profiling aids; the defaults are the product paths).  Each knob is seeded ONCE, when the
 * module is created, from the environment variable named below, and can be changed afterwards with pgb_module_set_option; no entry
 * point reads the environment. */
typedef enum {
    PGB_OPT_NO_FUSION = 0,      /* PGB_NO_FUSION: limb-wise HAL sequences instead of the fused single-kernel routes */
    PGB_OPT_NO_GADGET = 1,      /* PGB_NO_GADGET: disable the single-kernel gadget products only */
    PGB_OPT_NO_COLLAPSE = 2,    /* PGB_NO_COLLAPSE: per-limb inverse transforms in ntt120_fused_back */
    PGB_OPT_CGGI_VARIANT = 3,   /* PGB_CGGI_VARIANT: 0 = newest fused CGGI kernel, 1 / 2 / 3 = older generations (FFT64) */
    PGB_OPT_CGGI_BLOCK_BT1 = 4, /* PGB_CGGI_BLOCK_BT1: one ciphertext per thread in the FFT64 block kernel */
    PGB_OPT_VMP_NO_BT = 5,      /* PGB_VMP_NO_BT: no batch tiling in the NTT120 vmp */
    PGB_OPT_VMP_CT = 6,         /* PGB_VMP_CT: output polys per thread of the vmp kernels: 0 = chosen per launch (default), 2 / 4 (/ 8 NTT120) forced */
    PGB_OPT_GADGET_MB = 7,      /* PGB_GADGET_MB: resident clusters per SM the NTT120 gadget kernel is compiled for (3 or 4) */
    PGB_OPT_HOST_CHUNK_MB = 8,  /* PGB_HOST_CHUNK_MB: staging bytes per slot of the *_host pipelines (default 32) */
    PGB_OPT_CGGI_NTT_PRIMES = 9, /* PGB_CGGI_NTT_PRIMES: 0 = adaptive prime count in the NTT120 whole-rotation kernel, 2 / 3 / 4 = forced */
    PGB_OPT_GADGET_PRIMES = 10, /* PGB_GADGET_PRIMES: 0 = the NTT120 gadget kernel works on three primes when a pinned key's bound allows it, 4 = always four */
    PGB_OPT_LAST_GADGET_PRIMES = 11, /* read-only diagnostic: primes the last NTT120 gadget-kernel launch worked on (3 or 4; 0 = none yet) */
    PGB_OPT_CGGI_CLUSTER = 12,  /* PGB_CGGI_CLUSTER: 2 = the FFT64 whole-rotation kernel runs in clusters of two CTAs that share every key tile by TMA multicast */
    PGB_OPT_COUNT = 16
} pgb_option;
int pgb_module_set_option(pgb_module *m, int option, int64_t value);
int64_t pgb_module_get_option(const pgb_module *m, int option);
/* number of kernels launched by this module since creation (bench.py's gpu_launches) */
uint64_t pgb_module_launch_count(const pgb_module *m);

/* Optional per-kernel timing: when enabled every kernel launch is bracketed by CUDA events on the module's stream and the
 * elapsed device time is accumulated per category (0 dft_forward, 1 dft_inverse, 2 vmp_apply, 3 normalize, 4 elementwise,
 * 5 other, 6 gadget_fused = the single-kernel key-switch / external product).  pgb_profile_read synchronises the stream and
 * fills ms[PGB_PROFILE_NCAT] / launches[PGB_PROFILE_NCAT]. */
#define PGB_PROFILE_NCAT 7
int pgb_profile_enable(pgb_module *m, int on);
int pgb_profile_read(pgb_module *m, double *ms, uint64_t *launches, int reset);
const char *pgb_profile_category_name(int category);

/* ---- memory (Backend::alloc_bytes / from_bytes, layouts/module.rs:36-39; lib.rs:146 alignment) ---- */
void *pgb_alloc_bytes(size_t len);        /* CUDA managed, host-dereferenceable, zero-filled */
void *pgb_alloc_device_bytes(size_t len); /* device only, zero-filled */
void *pgb_alloc_pinned_bytes(size_t len); /* page-locked host memory for staging */
void pgb_free(void *p);
void pgb_free_pinned(void *p);
int pgb_memcpy_h2d(void *dst, const void *src, size_t len);
int pgb_memcpy_d2h(void *dst, const void *src, size_t len);
int pgb_memcpy_d2d(void *dst, const void *src, size_t len);
int pgb_memset(void *dst, int byte, size_t len);
/* zero fill of a block a host-side pool hands out again (device-wide synchronisation on both sides) */
int pgb_recycle_device_bytes(void *p, size_t len);
int pgb_current_device(void); /* the device pgb_alloc_device_bytes allocates on (-1 on error) */
/* The allocation / copy helpers above act on the CURRENT device (as cudaMalloc does); a caller that drives modules on several devices from
 * one thread selects the device first.  Entry points that take a module make the module's device current themselves before any launch. */
int pgb_set_device(int device);
int pgb_module_device(const pgb_module *m);

/* Backend::bytes_of_* (layouts/module.rs:44-70) */
size_t pgb_size_of_scalar_prep(const pgb_module *m);
size_t pgb_size_of_scalar_big(const pgb_module *m);
size_t pgb_bytes_of_vec_znx(const pgb_module *m, uint64_t cols, uint64_t size);
size_t pgb_bytes_of_vec_znx_dft(const pgb_module *m, uint64_t cols, uint64_t size);
size_t pgb_bytes_of_vec_znx_big(const pgb_module *m, uint64_t cols, uint64_t size);
size_t pgb_bytes_of_svp_ppol(const pgb_module *m, uint64_t cols);
size_t pgb_bytes_of_vmp_pmat(const pgb_module *m, uint64_t rows, uint64_t cols_in, uint64_t cols_out, uint64_t size);

/* ---- vec_znx_dft (oep/hal_impl.rs:529-593; R6/R7/R12, F4) -------------------------------------- */
/* HalImpl::vec_znx_dft_apply :529  (reference/ntt120/vec_znx_dft.rs:177-215, fft64/vec_znx_dft.rs:160-200) */
int pgb_vec_znx_dft_apply(pgb_module *m, uint64_t step, uint64_t offset, pgb_vec_znx_dft *res, uint64_t res_col,
                          const pgb_vec_znx *a, uint64_t a_col);
int pgb_vec_znx_dft_apply_batched(pgb_module *m, uint64_t step, uint64_t offset, pgb_vec_znx_dft *res, uint64_t res_col,
                                  const pgb_vec_znx *a, uint64_t a_col, const pgb_batch *bt);
/* HalImpl::vec_znx_idft_apply_tmp_bytes :534 -- the GPU path needs no scratch (returns 0). */
size_t pgb_vec_znx_idft_apply_tmp_bytes(const pgb_module *m);
/* HalImpl::vec_znx_idft_apply :536 (ntt120/vec_znx_dft.rs:236-268, fft64/vec_znx_dft.rs:202-232) */
int pgb_vec_znx_idft_apply(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx_dft *a, uint64_t a_col);
int pgb_vec_znx_idft_apply_batched(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx_dft *a,
                                   uint64_t a_col, const pgb_batch *bt);
/* HalImpl::vec_znx_idft_apply_tmpa :541 (a may be clobbered) */
int pgb_vec_znx_idft_apply_tmpa(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, pgb_vec_znx_dft *a, uint64_t a_col);
/* HalImpl::vec_znx_idft_apply_consume :546 -- in place; afterwards a->data is a VecZnxBig(n, cols, size)
 * (ntt120/vec_znx_dft.rs:327-409: big limb k at byte offset 16*n*k; fft64/vec_znx_dft.rs:264-288). */
int pgb_vec_znx_idft_apply_consume(pgb_module *m, pgb_vec_znx_dft *a);
int pgb_vec_znx_idft_apply_consume_batched(pgb_module *m, pgb_vec_znx_dft *a, const pgb_batch *bt);
/* HalImpl::vec_znx_dft_add_into :553, add_scaled_assign :559, add_assign :564, sub :569, sub_assign :575,
 * sub_negate_assign :580, copy :585, zero :590 (ntt120/vec_znx_dft.rs:418-652, fft64/vec_znx_dft.rs:13-157,290-405) */
int pgb_vec_znx_dft_add_into(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a, uint64_t a_col,
                             const pgb_vec_znx_dft *b, uint64_t b_col);
int pgb_vec_znx_dft_add_scaled_assign(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a,
                                      uint64_t a_col, int64_t a_scale);
int pgb_vec_znx_dft_add_assign(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a, uint64_t a_col);
int pgb_vec_znx_dft_sub(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a, uint64_t a_col,
                        const pgb_vec_znx_dft *b, uint64_t b_col);
int pgb_vec_znx_dft_sub_assign(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a, uint64_t a_col);
int pgb_vec_znx_dft_sub_negate_assign(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a,
                                      uint64_t a_col);
int pgb_vec_znx_dft_copy(pgb_module *m, uint64_t step, uint64_t offset, pgb_vec_znx_dft *res, uint64_t res_col,
                         const pgb_vec_znx_dft *a, uint64_t a_col);
int pgb_vec_znx_dft_zero(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col);
int pgb_vec_znx_dft_add_assign_batched(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a,
                                       uint64_t a_col, const pgb_batch *bt);
int pgb_vec_znx_dft_sub_assign_batched(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_vec_znx_dft *a,
                                       uint64_t a_col, const pgb_batch *bt);
int pgb_vec_znx_dft_copy_batched(pgb_module *m, uint64_t step, uint64_t offset, pgb_vec_znx_dft *res, uint64_t res_col,
                                 const pgb_vec_znx_dft *a, uint64_t a_col, const pgb_batch *bt);
int pgb_vec_znx_dft_zero_batched(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_batch *bt);

/* ---- svp (oep/hal_impl.rs:595-616; R11, F6) ------------------------------------------------------ */
/* HalImpl::svp_prepare :595 (ntt120/svp.rs:52-70, fft64/svp.rs:9-20) */
int pgb_svp_prepare(pgb_module *m, pgb_svp_ppol *res, uint64_t res_col, const pgb_scalar_znx *a, uint64_t a_col);
/* HalImpl::svp_apply_dft :600 (fft64/svp.rs:21-55; NTT120 default poulpy-cpu-ref/src/hal_defaults/svp_ppol.rs:93-107): b is a VecZnx */
int pgb_svp_apply_dft(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_svp_ppol *a, uint64_t a_col,
                      const pgb_vec_znx *b, uint64_t b_col);
/* HalImpl::svp_apply_dft_to_dft :606 (ntt120/svp.rs:87-133, fft64/svp.rs:57-79) */
int pgb_svp_apply_dft_to_dft(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_svp_ppol *a, uint64_t a_col,
                             const pgb_vec_znx_dft *b, uint64_t b_col);
/* bt->stride_a strides the SvpPPol (0 = shared), bt->stride_b strides b. */
int pgb_svp_apply_dft_to_dft_batched(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_svp_ppol *a,
                                     uint64_t a_col, const pgb_vec_znx_dft *b, uint64_t b_col, const pgb_batch *bt);
/* HalImpl::svp_apply_dft_to_dft_assign :612 (ntt120/svp.rs:148-180, fft64/svp.rs:81-94) */
int pgb_svp_apply_dft_to_dft_assign(pgb_module *m, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_svp_ppol *a,
                                    uint64_t a_col);

/* ---- vmp (oep/hal_impl.rs:618-668; R9/R10, F5) ---------------------------------------------------- */
/* HalImpl::vmp_prepare_tmp_bytes :618 / vmp_apply_dft_to_dft_tmp_bytes :643 -- no scratch needed (0). */
size_t pgb_vmp_prepare_tmp_bytes(const pgb_module *m, uint64_t rows, uint64_t cols_in, uint64_t cols_out, uint64_t size);
size_t pgb_vmp_apply_dft_to_dft_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t rows,
                                          uint64_t cols_in, uint64_t cols_out, uint64_t size);
/* HalImpl::vmp_apply_dft_tmp_bytes :626 / vmp_apply_dft :636 (poulpy-cpu-ref/src/hal_impl/family_common.rs:3-58): `a` is a VecZnx; the
 * library transforms its last min(a.cols, cols_in) columns into `scratch` (device memory) and applies the matrix. */
size_t pgb_vmp_apply_dft_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t rows, uint64_t cols_in,
                                   uint64_t cols_out, uint64_t size);
int pgb_vmp_apply_dft(pgb_module *m, pgb_vec_znx_dft *res, const pgb_vec_znx *a, const pgb_vmp_pmat *pmat, void *scratch,
                      size_t scratch_len);
/* HalImpl::vmp_prepare :620 (ntt120/vmp.rs:64-119, fft64/vmp.rs:52-93); `a` is a MatZnx of i64. */
int pgb_vmp_prepare(pgb_module *m, pgb_vmp_pmat *res, const pgb_mat_znx *a);
/* count MatZnx -> count VmpPMat in one forward-transform launch: item b reads a->data + b*stride_a and writes res->data + b*stride_res
 * (VmpPMat data and stride multiples of 16 bytes, MatZnx multiples of 8, strides at least one matrix; count in [1, 65535]).  res and a
 * must not overlap (PGB_ERR_ALIAS).  Like pgb_vmp_prepare it drops the cached gadget forms of every pinned key inside the written extent.
 * Asynchronous (call pgb_module_sync before reading). */
int pgb_vmp_prepare_batched(pgb_module *m, pgb_vmp_pmat *res, const pgb_mat_znx *a, const pgb_batch *bt);
/* HalImpl::vmp_apply_dft_to_dft :653 (ntt120/vmp.rs:301-341 + core :169-288; fft64/vmp.rs:144-264).
 * Overwrites res; limb_offset is in limbs and is scaled by cols_out exactly as ntt120/vmp.rs:335. */
int pgb_vmp_apply_dft_to_dft(pgb_module *m, pgb_vec_znx_dft *res, const pgb_vec_znx_dft *a, const pgb_vmp_pmat *pmat,
                             uint64_t limb_offset);
/* bt->stride_a strides a, bt->stride_b strides pmat (0 = one matrix shared by the whole batch). */
int pgb_vmp_apply_dft_to_dft_batched(pgb_module *m, pgb_vec_znx_dft *res, const pgb_vec_znx_dft *a,
                                     const pgb_vmp_pmat *pmat, uint64_t limb_offset, const pgb_batch *bt);
/* HalImpl::vmp_zero :665 */
int pgb_vmp_zero(pgb_module *m, pgb_vmp_pmat *res);

/* ---- vec_znx_big (oep/hal_impl.rs:323-527; R13/R14, F7) -------------------------------------------- */
/* HalImpl::vec_znx_big_normalize_tmp_bytes :428 -- carries live in registers (0). */
size_t pgb_vec_znx_big_normalize_tmp_bytes(const pgb_module *m);
/* HalImpl::vec_znx_big_normalize :431 (ntt120/vec_znx_big.rs:1383-1402 -> :367-446 / :453-597;
 * fft64/vec_znx_big.rs:241-278 -> reference/vec_znx/normalize.rs:18-426) */
int pgb_vec_znx_big_normalize(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, int64_t res_offset, uint64_t res_col,
                              const pgb_vec_znx_big *a, uint64_t a_base2k, uint64_t a_col);
int pgb_vec_znx_big_normalize_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, int64_t res_offset,
                                      uint64_t res_col, const pgb_vec_znx_big *a, uint64_t a_base2k, uint64_t a_col,
                                      const pgb_batch *bt);
/* HalImpl::vec_znx_big_normalize_add_assign :478 / _sub_assign :498 (ntt120/vec_znx_big.rs:600-803,1405-1461) */
int pgb_vec_znx_big_normalize_add_assign(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, int64_t res_offset,
                                         uint64_t res_col, const pgb_vec_znx_big *a, uint64_t a_base2k, uint64_t a_col);
int pgb_vec_znx_big_normalize_sub_assign(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, int64_t res_offset,
                                         uint64_t res_col, const pgb_vec_znx_big *a, uint64_t a_base2k, uint64_t a_col);
/* HalImpl::vec_znx_big_add_small_assign :362 (ntt120/vec_znx_big.rs:1128-1140) */
int pgb_vec_znx_big_add_small_assign(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col);
int pgb_vec_znx_big_add_small_assign_batched(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx *a,
                                             uint64_t a_col, const pgb_batch *bt);
/* HalImpl::vec_znx_big_from_small :323 */
int pgb_vec_znx_big_from_small(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col);

/* ---- coefficient-domain helpers used by the compositions (oep/hal_impl.rs:41-53, :225-228) ---------- */
/* HalImpl::vec_znx_normalize :41 (reference/vec_znx/normalize.rs:18-50) */
int pgb_vec_znx_normalize(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, int64_t res_offset, uint64_t res_col,
                          const pgb_vec_znx *a, uint64_t a_base2k, uint64_t a_col);
int pgb_vec_znx_normalize_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, int64_t res_offset,
                                  uint64_t res_col, const pgb_vec_znx *a, uint64_t a_base2k, uint64_t a_col,
                                  const pgb_batch *bt);
/* HalImpl::vec_znx_rotate :225 (reference/vec_znx/rotate.rs:9-38) */
int pgb_vec_znx_rotate(pgb_module *m, int64_t p, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col);
int pgb_vec_znx_rotate_batched(pgb_module *m, int64_t p, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col,
                               const pgb_batch *bt);
/* strided device-to-device copy on the module's stream (glwe_copy between containers of different batch strides) */
int pgb_memcpy_d2d_strided(pgb_module *m, void *dst, uint64_t dst_stride, const void *src, uint64_t src_stride, uint64_t width, uint64_t count);

/* ---- CoreImpl tier: fused, device-resident, batched pipelines (poulpy-core/src/oep/core_impl.rs:36-52,114-130) ---- */
/* Device scratch needed by the batched pipelines below (bytes; pass a pgb_alloc_device_bytes buffer). */
size_t pgb_glwe_keyswitch_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t a_base2k,
                                    const pgb_vmp_pmat *key, uint64_t key_base2k, uint64_t dsize, uint64_t batch);
/* CoreImpl::glwe_keyswitch (poulpy-core/src/keyswitching/glwe.rs:53-109, :207-239, :298-380; C1).
 * res/a are GLWE data VecZnx(rank+1, size); item b at data + b*stride.  key = GGLWEPrepared.data:
 * VmpPMat(dnum, rank_in, rank_out+1, key_size), shared by the batch. */
int pgb_glwe_keyswitch_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a, uint64_t a_base2k,
                               const pgb_vmp_pmat *key, uint64_t key_base2k, uint64_t dsize, const pgb_batch *bt,
                               void *scratch, size_t scratch_len);
size_t pgb_glwe_external_product_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t a_base2k,
                                           const pgb_vmp_pmat *ggsw, uint64_t ggsw_base2k, uint64_t dsize, uint64_t batch);
/* CoreImpl::glwe_external_product (poulpy-core/src/external_product/glwe.rs:99-141, :197-271; C2).
 * ggsw = GGSWPrepared.data: VmpPMat(dnum, rank+1, rank+1, size), shared by the batch. */
int pgb_glwe_external_product_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a,
                                      uint64_t a_base2k, const pgb_vmp_pmat *ggsw, uint64_t ggsw_base2k, uint64_t dsize,
                                      const pgb_batch *bt, void *scratch, size_t scratch_len);

/* CMux (poulpy-bin-fhe: glwe_sub, glwe_normalize_inplace, glwe_external_product_inplace, glwe_add_inplace, glwe_normalize_inplace).
 * t, f, res: GLWEs VecZnx(k + 1, .) in base 2^base2k; item b at data + b*stride (bt->stride_res for res, bt->stride_a for t, bt->stride_b
 * for f; t and f may use stride 0 to share one operand).  s: prepared GGSWs VmpPMat(dnum, k + 1, k + 1, s_size) in base 2^ggsw_base2k,
 * item b's selector at s->data + b*ggsw_stride (0 = one selector shared by the batch; otherwise a multiple of 16 of at least
 * pgb_bytes_of_vmp_pmat).  Per item:
 *   1. d[i] = t[i] - f[i] (wrapping i64) for i < res.size, a limb missing from an operand reads as 0;   2. d = vec_znx_normalize_assign(d);
 *   3. e = glwe_external_product(d, s_b) into res.size limbs of base2k (any dsize, mixed ggsw_base2k);
 *   4. e[i] += f[i] (wrapping i64) for i < min(res.size, f.size);   5. res = vec_znx_normalize_assign(e).
 * count in [1, 65535]; GLWE data and strides multiples of 16; scratch 256-byte aligned.  res must not overlap t, f, a selector or the
 * scratch (PGB_ERR_ALIAS); t and f are read-only and may overlap each other.  Every check runs before the first launch. */
size_t pgb_glwe_cmux_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t t_size, uint64_t f_size, uint64_t base2k,
                               const pgb_vmp_pmat *s, uint64_t ggsw_base2k, uint64_t dsize, uint64_t batch);
int pgb_glwe_cmux_batched(pgb_module *m, pgb_vec_znx *res, const pgb_vec_znx *t, const pgb_vec_znx *f, uint64_t base2k,
                          const pgb_vmp_pmat *s, uint64_t ggsw_stride, uint64_t ggsw_base2k, uint64_t dsize,
                          const pgb_batch *bt, void *scratch, size_t scratch_len);
/* Blind rotation of GLWEs by GGSW bits (a rotation by an encrypted integer, as poulpy-bin-fhe's BDD arithmetic does it): per item b,
 * acc_0 = a_b and, for i < n_bits with p_i = (step * 2^i) mod 2n (computed without overflow for any step),
 *   acc_{i+1} = cmux(t = X^(p_i) acc_i, f = acc_i, s_{b,i})   -- the five CMux steps above, into res.size limbs (X^p = vec_znx_rotate(p)
 *                                                                on every column);
 * res_b = acc_{n_bits}.  Selector s_{b,i} at s->data + b*ggsw_stride + i*bit_stride (64-bit byte offsets): ggsw_stride as for the CMux
 * (0 = one encrypted integer for the batch), bit_stride a multiple of 16 of at least one prepared GGSW when n_bits > 1.  bt->stride_res
 * for res, bt->stride_a for a (0 = one a, e.g. a LUT, rotated by every item's integer), bt->stride_b must be 0.  count in [1, 65535],
 * n_bits in [1, 64]; alignment, shapes and errors as for the CMux: res must not overlap a, any selector (b, i) or the scratch
 * (PGB_ERR_ALIAS); every check runs before the first launch.  The scratch holds one ping-pong accumulator (n_bits > 1) and the CMux's
 * scratch for res.size-limb operands. */
size_t pgb_glwe_blind_rotate_ggsw_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t base2k,
                                            const pgb_vmp_pmat *s, uint64_t ggsw_base2k, uint64_t dsize, uint64_t n_bits, uint64_t batch);
int pgb_glwe_blind_rotate_ggsw_batched(pgb_module *m, pgb_vec_znx *res, const pgb_vec_znx *a, uint64_t base2k, int64_t step,
                                       uint64_t n_bits, const pgb_vmp_pmat *s, uint64_t ggsw_stride, uint64_t bit_stride,
                                       uint64_t ggsw_base2k, uint64_t dsize, const pgb_batch *bt, void *scratch, size_t scratch_len);
/* CMux tree over GGSW bits (selection of one of 2^n_bits GLWEs by an encrypted integer: an encrypted-array read, or the table selection of
 * a lookup table read by vertical packing): per item b, with leaves g_{0,j} = a_b[j] at a->data + b*bt->stride_a + j*entry_stride
 * (j < 2^n_bits; stride_a = 0 shares one table across the batch; entry_stride a multiple of 16 of at least one GLWE of a.size limbs),
 *   g_{i+1,j} = cmux(t = g_{i,2j+1}, f = g_{i,2j}, s_{b,i})   for i < n_bits, j < 2^(n_bits-1-i)  -- the five CMux steps above, into
 *                                                               res.size limbs;
 * res_b = g_{n_bits,0}: with noise-free GGSW bits m_{b,i}, leaf sum_i m_{b,i} 2^i, normalised.  Selector s_{b,i} at s->data +
 * b*ggsw_stride + i*bit_stride, with the rules of pgb_glwe_blind_rotate_ggsw_batched (0 = one encrypted integer for the batch).
 * bt->stride_b must be 0, count in [1, 65535], n_bits in [1, 16]; res must not overlap the table, any selector or the scratch
 * (PGB_ERR_ALIAS); every check runs before the first launch.  Items run in chunks of whole items, each chunk the whole tree, one batched
 * CMux per level: _tmp_bytes(batch) is the scratch of a chunk of min(batch, floor(65535 / 2^(n_bits-1))) items, and the entry takes the
 * largest chunk whose _tmp_bytes fits scratch_len (PGB_ERR_SCRATCH when one item does not).  Results do not depend on the chunk. */
size_t pgb_glwe_cmux_tree_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t base2k, const pgb_vmp_pmat *s,
                                    uint64_t ggsw_base2k, uint64_t dsize, uint64_t n_bits, uint64_t batch);
int pgb_glwe_cmux_tree_batched(pgb_module *m, pgb_vec_znx *res, const pgb_vec_znx *a, uint64_t entry_stride, uint64_t base2k,
                               uint64_t n_bits, const pgb_vmp_pmat *s, uint64_t ggsw_stride, uint64_t bit_stride, uint64_t ggsw_base2k,
                               uint64_t dsize, const pgb_batch *bt, void *scratch, size_t scratch_len);
/* Binary decision diagram over GGSW bits: a levelled CMux circuit given as data (host memory, read during the call only; it may be freed
 * when the entry returns).  States 0 .. n_leaves-1 are the leaves; node k (level order: the level_count[0] nodes of level 0 first) is state
 * n_leaves + k.  Every child of a node of level i is a leaf or a node of a level < i; outputs[o] is any state. */
typedef struct {
    uint64_t n_leaves;           /* states 0 .. n_leaves-1 are the leaves */
    uint64_t n_levels;
    const uint32_t *level_bit;   /* [n_levels]: the bit every node of level i selects with */
    const uint32_t *level_count; /* [n_levels]: nodes in level i (>= 1) */
    const uint32_t *node_t;      /* [total nodes], level order: the state taken when the bit is 1 */
    const uint32_t *node_f;      /* [total nodes]: the state taken when the bit is 0 */
    uint64_t n_out;
    const uint32_t *outputs;     /* [n_out]: state indices */
} pgb_bdd_circuit;
/* Per item b: leaf j is a->data + b*bt->stride_a + j*entry_stride (a.size limbs; stride_a = 0 shares the leaves across the batch;
 * entry_stride a multiple of 16 of at least one GLWE of a.size limbs when n_leaves > 1); node k of level i is
 *   state[n_leaves + k] = cmux(t = state[node_t[k]], f = state[node_f[k]], s_{b, level_bit[i]})  -- the five CMux steps above, into
 *                                                                                                 res.size limbs;
 * output o goes to res->data + b*bt->stride_res + o*out_stride: a node's res.size limbs, or a leaf's first min(a.size, res.size) limbs with
 * the rest zeroed (no normalisation).  Selector s_{b,i} at s->data + b*ggsw_stride + i*bit_stride, with the rules of
 * pgb_glwe_blind_rotate_ggsw_batched (0 = one encrypted integer for the batch); level_bit[i] < n_bits <= 64.  bt->stride_b must be 0,
 * count in [1, 65535], every level width in [1, 65535], n_out >= 1; out_stride a multiple of 16 of at least one GLWE of res.size limbs when
 * n_out > 1, and bt->stride_res a multiple of 16 of at least (n_out-1)*out_stride plus one GLWE when count > 1.  res must not overlap the
 * leaves, any selector or the scratch (PGB_ERR_ALIAS).  Every check (null pointers, child, output and bit indices, widths, 128-bit extents,
 * aliasing, 256-byte scratch alignment) runs on the host arrays before the first launch.  Items run in chunks of whole items; a chunk of Bc
 * items keeps Bc * (widest level) <= 65535, and _tmp_bytes(batch) is the scratch of a chunk of min(batch, that cap) items: the circuit's
 * descriptor table, one block of Bc*level_count[i] GLWEs of res.size limbs per level, the linear copy of f and one CMux's scratch for the
 * widest level.  The entry takes the largest chunk whose _tmp_bytes fits scratch_len (PGB_ERR_SCRATCH when one item does not).  Results do
 * not depend on the chunk.  A chunk launches one CMux's launches per level plus one output copy. */
size_t pgb_glwe_bdd_eval_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t base2k, const pgb_vmp_pmat *s,
                                   uint64_t ggsw_base2k, uint64_t dsize, const pgb_bdd_circuit *c, uint64_t batch);
int pgb_glwe_bdd_eval_batched(pgb_module *m, pgb_vec_znx *res, uint64_t out_stride, const pgb_vec_znx *a, uint64_t entry_stride,
                              uint64_t base2k, uint64_t n_bits, const pgb_vmp_pmat *s, uint64_t ggsw_stride, uint64_t bit_stride,
                              uint64_t ggsw_base2k, uint64_t dsize, const pgb_bdd_circuit *c, const pgb_batch *bt, void *scratch,
                              size_t scratch_len);
/* glwe_pack (poulpy-core/src/glwe_packing.rs:15-170), batched: per item b, input j < n_in is the GLWE at a->data + b*bt->stride_a +
 * j*entry_stride (stride_a = 0 shares the inputs across the batch), and res_b (res->data + b*bt->stride_res) is the GLWE whose coefficient
 * index[j] carries the constant coefficient of input j: bit for bit what the host composition glwe_pack(ops, res, {index[j]: a_j},
 * log_gap_out) over the batched entries computes (pack_internal per pair of round i < log_n - log_gap_out, then glwe_trace with skip =
 * log_n - log_gap_out).  `index` is a HOST array read during the call only; indices are distinct, below n and multiples of 2^log_gap_out.
 * One layout throughout: a.size == res.size, one base2k for GLWEs and keys.  `keys` is a HOST array of log_n prepared automorphism keys of
 * one shape, keys[i] for pgb_trace_galois_element(i), cols_in = cols - 1, cols_out = cols.  The inputs are read-only.  n_in in [1, n],
 * log_gap_out <= log_n, nkeys >= log_n, count in [1, 65535], bt->stride_b == 0; data and strides multiples of 16, entry_stride at least one
 * GLWE when n_in > 1; res must not overlap the inputs, a key or the scratch (PGB_ERR_ALIAS); scratch 256-byte aligned.  Every check runs
 * before the first launch.  Round i of a chunk is one prep kernel, at most three batched automorphism calls under keys[i] (plain
 * glwe_automorphism for the pairs, op 0 for keys with only j, op 2 for keys with only j + t) and one combine kernel when pairs exist; then
 * the trace (or, without rounds, one copy).  Items run in chunks of whole items, Bc * (widest round) <= 65535; _tmp_bytes(batch) is the
 * scratch of a chunk of min(batch, that cap) items: the descriptor table, two ping-pong state blocks and the x block of Bc * (widest round)
 * GLWEs, the y block of Bc * (most pairs of a round) GLWEs, and the automorphism / trace scratch.  The entry takes the largest chunk whose
 * _tmp_bytes fits scratch_len (PGB_ERR_SCRATCH when one item does not); results do not depend on the chunk.  _tmp_bytes returns 0 for an
 * invalid map. */
size_t pgb_glwe_pack_tmp_bytes(const pgb_module *m, uint64_t size, uint64_t base2k, const pgb_vmp_pmat *key, uint64_t dsize,
                               const uint32_t *index, uint64_t n_in, uint64_t log_gap_out, uint64_t batch);
int pgb_glwe_pack_batched(pgb_module *m, pgb_vec_znx *res, const pgb_vec_znx *a, uint64_t entry_stride, const uint32_t *index,
                          uint64_t n_in, uint64_t log_gap_out, uint64_t base2k, const pgb_vmp_pmat *keys, uint64_t nkeys,
                          uint64_t dsize, const pgb_batch *bt, void *scratch, size_t scratch_len);

/* Pinned keys.  The single-kernel gadget products derive per-key forms of a prepared key before they run (NTT120: the collapsed key and
 * the bit bound of the key's coefficients, three small launches; FFT64: a re-laid-out copy, one launch).  Every buffer is caller-owned, so
 * the library cannot know that a key's bytes are unchanged between two calls -- unless the caller says so: after pgb_gadget_key_pin(key)
 * the module keeps those forms across calls (keyed on key->data and the call's shape) until pgb_gadget_key_unpin(key), module
 * destruction, or a pgb_vmp_prepare into that memory (which drops them).  Rewriting a pinned key's bytes by any other means without
 * unpinning it first is a contract violation.  Unpinned keys behave as before (forms re-derived on every call).  In the reference the
 * analogue is the lifetime of a `GGLWEPrepared` / `GGSWPrepared` value: prepared once, borrowed immutably by every product.
 * For a pinned key the host also learns the key's coefficient bound (one 4-byte read-back when the forms are built); when that bound
 * proves that the integers of the product stay below Q[0] Q[1] Q[2] / 2 the NTT120 gadget kernel works on three primes instead of four
 * (same results bit for bit: every input is still checked on the device; PGB_OPT_GADGET_PRIMES = 4 disables it). */
int pgb_gadget_key_pin(pgb_module *m, const pgb_vmp_pmat *key);
int pgb_gadget_key_unpin(pgb_module *m, const pgb_vmp_pmat *key);

/* Host-buffer front ends: `res_host` / `a_host` are ordinary host arrays of `count` GLWE VecZnx; the
 * library stages them through pinned memory in chunks, overlapping H2D, compute and D2H on the module's
 * streams, and returns when `res_host` is complete.  This is what a HalImpl/CoreImpl over host-resident
 * `Vec<u8>` buffers sees. */
int pgb_glwe_keyswitch_host(pgb_module *m, int64_t *res_host, uint64_t res_size, uint64_t res_base2k, const int64_t *a_host,
                            uint64_t a_size, uint64_t a_base2k, uint64_t rank_in, uint64_t rank_out,
                            const pgb_vmp_pmat *key, uint64_t key_base2k, uint64_t dsize, uint64_t count);
int pgb_glwe_external_product_host(pgb_module *m, int64_t *res_host, uint64_t res_size, uint64_t res_base2k,
                                   const int64_t *a_host, uint64_t a_size, uint64_t a_base2k, uint64_t rank,
                                   const pgb_vmp_pmat *ggsw, uint64_t ggsw_base2k, uint64_t dsize, uint64_t count);

/* One host call over several devices: `modules[i]` lives on its own CUDA device (or shares one), `keys[i]` is the replica of the prepared
 * key in that device's memory; the `count` ciphertexts are split contiguously over the modules and every shard runs
 * pgb_glwe_keyswitch_host on its own host thread.  This is what a Rust caller holding one `Module<B>` per GPU (Module is Sync + Send,
 * poulpy-hal/src/layouts/module.rs:103-104) does with a thread pool; no collective is involved. */
int pgb_glwe_keyswitch_host_sharded(pgb_module *const *modules, const pgb_vmp_pmat *keys, uint64_t n_modules, int64_t *res_host,
                                    uint64_t res_size, uint64_t res_base2k, const int64_t *a_host, uint64_t a_size, uint64_t a_base2k,
                                    uint64_t rank_in, uint64_t rank_out, uint64_t key_base2k, uint64_t dsize, uint64_t count);

/* ---- bivariate convolution (oep/hal_impl.rs:670-754; SURVEY 8f N2) ---------------------------------------------------
 * CnvPVecL / CnvPVecR (poulpy-hal/src/layouts/cnv_pvec.rs) are backend-owned prepared layouts; here both are DFT limbs in the
 * VecZnxDft layout, described by the same POD struct.  All *_tmp_bytes are 0. */
typedef pgb_vec_znx pgb_cnv_pvec;
size_t pgb_bytes_of_cnv_pvec_left(const pgb_module *m, uint64_t cols, uint64_t size);
size_t pgb_bytes_of_cnv_pvec_right(const pgb_module *m, uint64_t cols, uint64_t size);
size_t pgb_cnv_prepare_left_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size);
size_t pgb_cnv_prepare_right_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size);
size_t pgb_cnv_prepare_self_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size);
size_t pgb_cnv_apply_dft_tmp_bytes(const pgb_module *m, uint64_t cnv_offset, uint64_t res_size, uint64_t a_size, uint64_t b_size);
size_t pgb_cnv_pairwise_apply_dft_tmp_bytes(const pgb_module *m, uint64_t cnv_offset, uint64_t res_size, uint64_t a_size, uint64_t b_size);
size_t pgb_cnv_by_const_apply_tmp_bytes(const pgb_module *m, uint64_t cnv_offset, uint64_t res_size, uint64_t a_size, uint64_t b_size);
/* HalImpl::cnv_prepare_left :672 / cnv_prepare_right :679 / cnv_prepare_self :750 (reference/ntt120/convolution.rs:66-236):
 * forward transform of every column of `a`, the last active limb ANDed with `mask` first */
int pgb_cnv_prepare_left(pgb_module *m, pgb_cnv_pvec *res, const pgb_vec_znx *a, int64_t mask);
int pgb_cnv_prepare_right(pgb_module *m, pgb_cnv_pvec *res, const pgb_vec_znx *a, int64_t mask);
int pgb_cnv_prepare_self(pgb_module *m, pgb_cnv_pvec *left, pgb_cnv_pvec *right, const pgb_vec_znx *a, int64_t mask);
/* HalImpl::cnv_apply_dft :709 (convolution.rs:256-335): res[res_col, k] = sum_j a[a_col, k + off - j] (.) b[b_col, j] */
int pgb_cnv_apply_dft(pgb_module *m, uint64_t cnv_offset, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_cnv_pvec *a, uint64_t a_col,
                      const pgb_cnv_pvec *b, uint64_t b_col);
int pgb_cnv_apply_dft_batched(pgb_module *m, uint64_t cnv_offset, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_cnv_pvec *a,
                              uint64_t a_col, const pgb_cnv_pvec *b, uint64_t b_col, const pgb_batch *bt);
/* HalImpl::cnv_pairwise_apply_dft :733 (convolution.rs:441-557): (a[:, i] + a[:, j]) x (b[:, i] + b[:, j]) */
int pgb_cnv_pairwise_apply_dft(pgb_module *m, uint64_t cnv_offset, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_cnv_pvec *a,
                               const pgb_cnv_pvec *b, uint64_t col_i, uint64_t col_j);
int pgb_cnv_pairwise_apply_dft_batched(pgb_module *m, uint64_t cnv_offset, pgb_vec_znx_dft *res, uint64_t res_col, const pgb_cnv_pvec *a,
                                       const pgb_cnv_pvec *b, uint64_t col_i, uint64_t col_j, const pgb_batch *bt);
/* HalImpl::cnv_by_const_apply :695 (convolution.rs:361-410): coefficient-domain product with b_size HOST constants into the big type */
int pgb_cnv_by_const_apply(pgb_module *m, uint64_t cnv_offset, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col,
                           const int64_t *b, uint64_t b_size);

/* ---- coefficient-domain helpers of execute_standard (SURVEY 8f N1) ---- */
/* vec_znx_add_assign / sub_assign (poulpy-cpu-ref/src/reference/vec_znx/add.rs:60-82, sub.rs:60-82) */
int pgb_vec_znx_add_assign(pgb_module *m, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col);
int pgb_vec_znx_add_assign_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col,
                                   const pgb_batch *bt);
int pgb_vec_znx_sub_assign(pgb_module *m, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col);
int pgb_vec_znx_sub_assign_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col,
                                   const pgb_batch *bt);
/* vec_znx_mul_xp_minus_one (reference/vec_znx/mul_xp_minus_one.rs:13-22): res = X^p * a - a; res and a must not alias */
int pgb_vec_znx_mul_xp_minus_one(pgb_module *m, int64_t p, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col);
/* vec_znx_rsh_assign (HalImpl::vec_znx_rsh_assign, hal_impl.rs; reference/vec_znx/shift.rs:186-243): arithmetic right shift by k bits in base
 * 2^base2k, in place; ceil(k / base2k) must not exceed res.size (the reference panics) */
int pgb_vec_znx_rsh_assign(pgb_module *m, uint64_t base2k, uint64_t k, pgb_vec_znx *res, uint64_t res_col);
int pgb_vec_znx_rsh_assign_batched(pgb_module *m, uint64_t base2k, uint64_t k, pgb_vec_znx *res, uint64_t res_col, const pgb_batch *bt);
/* vec_znx_big_automorphism / _assign (HalImpl, hal_impl.rs; reference/ntt120/vec_znx_big.rs:1462-1529, reference/fft64/vec_znx_big.rs:140-188) */
int pgb_vec_znx_big_automorphism(pgb_module *m, int64_t p, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx_big *a, uint64_t a_col);
int pgb_vec_znx_big_automorphism_batched(pgb_module *m, int64_t p, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx_big *a,
                                         uint64_t a_col, const pgb_batch *bt);
size_t pgb_vec_znx_big_automorphism_assign_tmp_bytes(const pgb_module *m);
int pgb_vec_znx_big_automorphism_assign(pgb_module *m, int64_t p, pgb_vec_znx_big *res, uint64_t res_col);
/* vec_znx_big_sub_small_assign / _sub_small_negate_assign (HalImpl; reference/ntt120/vec_znx_big.rs:1285-1318): res -= a ; res = a - res */
int pgb_vec_znx_big_sub_small_assign(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col);
int pgb_vec_znx_big_sub_small_negate_assign(pgb_module *m, pgb_vec_znx_big *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col);
/* vec_znx_normalize_assign (reference/vec_znx/normalize.rs:403-425) */
int pgb_vec_znx_normalize_assign(pgb_module *m, uint64_t base2k, pgb_vec_znx *res, uint64_t res_col);
int pgb_vec_znx_normalize_assign_batched(pgb_module *m, uint64_t base2k, pgb_vec_znx *res, uint64_t res_col, const pgb_batch *bt);

/* ---- GLWE tensoring / relinearisation = CKKS multiplication (poulpy-core/src/operations/glwe.rs:699-818, :545-610;
 * poulpy-ckks/src/leveled/default/mul.rs:49-86; SURVEY 8f N2), batched and device resident ---- */
size_t pgb_glwe_tensor_apply_tmp_bytes(const pgb_module *m, uint64_t rank, uint64_t res_size, uint64_t res_base2k, uint64_t a_size,
                                       uint64_t b_size, uint64_t ab_base2k, uint64_t cnv_offset, uint64_t batch);
/* res: GLWETensor VecZnx with (rank+1)(rank+2)/2 columns; a, b: GLWE VecZnx of base2k `ab_base2k`, a.size == ceil(a_effective_k / ab_base2k) */
int pgb_glwe_tensor_apply_batched(pgb_module *m, uint64_t cnv_offset, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a,
                                  uint64_t a_effective_k, const pgb_vec_znx *b, uint64_t b_effective_k, uint64_t ab_base2k,
                                  const pgb_batch *bt, void *scratch, size_t scratch_len);
size_t pgb_glwe_tensor_relinearize_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t a_base2k,
                                             const pgb_vmp_pmat *tsk, uint64_t key_base2k, uint64_t dsize, uint64_t batch);
/* a: GLWETensor VecZnx; tsk: prepared tensor key = VmpPMat(dnum, rank(rank+1)/2, rank+1, size) */
int pgb_glwe_tensor_relinearize_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a, uint64_t a_base2k,
                                        const pgb_vmp_pmat *tsk, uint64_t key_base2k, uint64_t dsize, const pgb_batch *bt, void *scratch,
                                        size_t scratch_len);

/* ---- automorphisms (SURVEY 8f N4) ---- */
/* vec_znx_automorphism (poulpy-cpu-ref/src/reference/vec_znx/automorphism.rs:9-38): res = a(X^p), p odd; res and a must not alias */
int pgb_vec_znx_automorphism(pgb_module *m, int64_t p, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col);
int pgb_vec_znx_automorphism_batched(pgb_module *m, int64_t p, pgb_vec_znx *res, uint64_t res_col, const pgb_vec_znx *a, uint64_t a_col,
                                     const pgb_batch *bt);
/* glwe_automorphism (poulpy-core/src/automorphism/glwe_ct.rs:51-72): glwe_keyswitch with the automorphism key of Galois element p, then
 * X -> X^p on every column (what CKKS rotations / conjugation and the trace are made of) */
size_t pgb_glwe_automorphism_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t a_base2k, const pgb_vmp_pmat *key,
                                       uint64_t key_base2k, uint64_t dsize, uint64_t batch);
int pgb_glwe_automorphism_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a, uint64_t a_base2k,
                                  const pgb_vmp_pmat *key, uint64_t key_base2k, int64_t p, uint64_t dsize, const pgb_batch *bt, void *scratch,
                                  size_t scratch_len);

/* glwe_automorphism_add_assign (poulpy-core/src/automorphism/glwe_ct.rs:142-183): res += automorphism_p(key-switch(res)), the step the
 * trace is made of; glwe_trace_assign (poulpy-core/src/glwe_trace.rs:129-175): for i in skip..log_n { glwe_rsh(1); automorphism_add_assign
 * with the key of trace_galois_elements()[i] } (glwe_trace.rs:34-44).  `keys` is a HOST array of log_n prepared automorphism keys.
 * With one base2k on both sides and n = 2^10..2^12 (NTT120) / 2^9..2^12 (FFT64) the whole family is ONE launch of the gadget kernel per
 * batch (automorphism epilogue, DESIGN.md 3.4); the _tmp_bytes below include the staging of the outputs that the in-place forms need
 * there and, for the trace, the second GLWE buffer its rounds alternate with.  The NTT120 route reads one 4-byte flag count back per
 * call (stream synchronisation) to decide whether any ciphertext left the collapsed-key bound and the limb-wise sequence must redo the batch. */
size_t pgb_glwe_automorphism_add_assign_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t res_base2k, const pgb_vmp_pmat *key,
                                                  uint64_t key_base2k, uint64_t dsize, uint64_t batch);
int pgb_glwe_automorphism_add_assign_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vmp_pmat *key, uint64_t key_base2k,
                                             int64_t p, uint64_t dsize, const pgb_batch *bt, void *scratch, size_t scratch_len);
/* glwe_automorphism_add / _sub / _sub_negate (automorphism/glwe_ct.rs:95-275), out of place; op = 0: res = aut(ks(a)) + a, 1: aut(ks(a)) - a,
 * 2: a - aut(ks(a)); res == a gives the _assign forms; scratch as pgb_glwe_automorphism_add_assign_tmp_bytes */
int pgb_glwe_automorphism_op_batched(pgb_module *m, int op, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a, const pgb_vmp_pmat *key,
                                     uint64_t key_base2k, int64_t p, uint64_t dsize, const pgb_batch *bt, void *scratch, size_t scratch_len);
int64_t pgb_trace_galois_element(const pgb_module *m, uint64_t i);
size_t pgb_glwe_trace_assign_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t res_base2k, const pgb_vmp_pmat *key, uint64_t key_base2k,
                                       uint64_t dsize, uint64_t batch);
int pgb_glwe_trace_assign_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, uint64_t skip, const pgb_vmp_pmat *keys, uint64_t nkeys,
                                  uint64_t key_base2k, uint64_t dsize, const pgb_batch *bt, void *scratch, size_t scratch_len);

/* ggsw_expand_row (poulpy-core/src/conversion/gglwe_to_ggsw.rs:116-268; CoreImpl `ggsw_expand_row`): columns 1..rank of a GGSW from its
 * column-0 GLWEs and the tensor keys GGLWE(s[c] * s); `tsk` is a HOST array of rank prepared keys of identical shape */
size_t pgb_ggsw_expand_row_tmp_bytes(const pgb_module *m, uint64_t rank, uint64_t size, uint64_t res_base2k, const pgb_vmp_pmat *tsk,
                                     uint64_t tsk_base2k, uint64_t dsize, uint64_t batch);
int pgb_ggsw_expand_row_batched(pgb_module *m, pgb_mat_znx *ggsw, uint64_t res_base2k, const pgb_vmp_pmat *tsk, uint64_t ntsk, uint64_t tsk_base2k,
                                uint64_t dsize, const pgb_batch *bt, void *scratch, size_t scratch_len);

/* ---- CGGI blind rotation (poulpy-bin-fhe/src/blind_rotation/algorithms/cggi/algorithm.rs:275-368; C3) ---- */
/* x_pow_a table of the prepared key (cggi/key_prepared.rs:66-75): SvpPPol with 2n columns, col i = X^i. */
int pgb_cggi_x_pow_a(pgb_module *m, pgb_svp_ppol *res);
size_t pgb_cggi_blind_rotate_tmp_bytes(const pgb_module *m, uint64_t rank, uint64_t res_size, uint64_t dnum, uint64_t brk_size,
                                       uint64_t batch);
/* execute_block_binary over a batch of mod-switched LWEs.
 *   res    : `count` GLWE VecZnx(rank+1, res_size), stride bt->stride_res
 *   lwe_2n : device int64 [count][n_lwe+1] = (b, a_0..a_{n_lwe-1}) after mod_switch_2n (algorithms/mod.rs:136-176)
 *   lut    : VecZnx(1, lut_size) shared by the batch
 *   brk    : n_lwe prepared GGSWs, VmpPMat(dnum, rank+1, rank+1, brk_size) each, consecutive in memory
 *            (`brk->data` + i * bytes_of_vmp_pmat) */
int pgb_cggi_blind_rotate_batched(pgb_module *m, pgb_vec_znx *res, const int64_t *lwe_2n, uint64_t n_lwe, const pgb_vec_znx *lut,
                                  const pgb_vmp_pmat *brk, const pgb_svp_ppol *x_pow_a, uint64_t block_size, uint64_t base2k,
                                  const pgb_batch *bt, void *scratch, size_t scratch_len);
/* Host-buffer front end of the above = BlindRotationExecute::execute (cggi/algorithm.rs:88-117) for a caller whose LWE inputs and GLWE
 * outputs live in host memory: `lwe_host` = `count` one-column VecZnx(n_lwe + 1 coefficients (b, a_0, ..), lwe_size limbs of base
 * 2^lwe_base2k) back to back, `res_host` = `count` GLWE VecZnx(rank+1, res_size) back to back.  Uploads the LWEs, runs mod_switch_2n and
 * the rotation on the device in chunks and copies every finished chunk back while the next one computes; returns when res_host is
 * complete.  lut / brk / x_pow_a are the device-resident prepared objects of pgb_cggi_blind_rotate_batched; rot_left as in
 * pgb_cggi_mod_switch_2n_batched.  Pinned host buffers (pgb_alloc_pinned_bytes) make both copies asynchronous. */
int pgb_cggi_blind_rotate_host(pgb_module *m, int64_t *res_host, uint64_t rank, uint64_t res_size, const int64_t *lwe_host, uint64_t n_lwe,
                               uint64_t lwe_size, uint64_t lwe_base2k, int rot_left, const pgb_vec_znx *lut, const pgb_vmp_pmat *brk,
                               const pgb_svp_ppol *x_pow_a, uint64_t block_size, uint64_t base2k, uint64_t count);
/* execute_block_binary_extended (algorithm.rs:121-273): lut = `ext` VecZnx(1 col, lut_size) stored consecutively (LookupTable.data), lwe_2n
 * mod-switched to 2 * n * ext; res receives ring 0 of the accumulator */
size_t pgb_cggi_blind_rotate_extended_tmp_bytes(const pgb_module *m, uint64_t rank, uint64_t res_size, uint64_t dnum, uint64_t brk_size,
                                                uint64_t ext, uint64_t batch);
int pgb_cggi_blind_rotate_extended_batched(pgb_module *m, pgb_vec_znx *res, const int64_t *lwe_2n, uint64_t n_lwe, const pgb_vec_znx *lut,
                                           uint64_t ext, const pgb_vmp_pmat *brk, const pgb_svp_ppol *x_pow_a, uint64_t block_size,
                                           uint64_t base2k, const pgb_batch *bt, void *scratch, size_t scratch_len);

/* mod_switch_2n (algorithms/mod.rs:136-181) on the device: `lwe` = `count` one-column VecZnx of n_lwe + 1 coefficients (b, a_0, ...),
 * stride bt->stride_a; res = device int64 [count][n_lwe + 1]; two_n_domain = 2 * lut.domain_size(); rot_left = LookUpTableRotationDirection::Left. */
int pgb_cggi_mod_switch_2n_batched(pgb_module *m, int64_t *res, const pgb_vec_znx *lwe, uint64_t lwe_base2k, uint64_t two_n_domain,
                                   int rot_left, const pgb_batch *bt);
/* ---- LWE <-> GLWE (poulpy-core/src/conversion/glwe_to_lwe.rs, lwe_to_glwe.rs, keyswitching/lwe.rs) ----
 * An LWE is a one-column VecZnx of n = n_lwe + 1 coefficients per limb, (b, a_0, .., a_{n_lwe-1}), phase b + <a, s_lwe>, 1 <= n_lwe <= N;
 * its GLWE embedding is the rank-1 secret s_glwe(X) = s_lwe(X^-1).  Batches as everywhere (stride_res / stride_a, at least one item),
 * count in [1, 65535]; LWE data and strides are multiples of 8 bytes, GLWE data and strides multiples of 16, scratch 256-byte aligned.
 * There is no in-place form: any overlap of res and a is PGB_ERR_ALIAS.
 * sample_extract: a = rank-1 GLWE; limbs i < min(res.size, a.size) get (a[0][i][0], a[1][i][0..n_lwe)), the other limbs of res are zeroed.
 * lwe_keyswitch: key = VmpPMat(dnum, 1, 2, key_size) from embed(s_in) to embed(s_out); a is embedded into a rank-1 GLWE, key-switched with
 *   pgb_glwe_keyswitch_batched into res.size limbs of res_base2k and sample-extracted.
 * glwe_to_lwe: a = GLWE of rank k, key = VmpPMat(dnum, k, 2, key_size) to embed(s_lwe); key-switch to rank 1, then sample-extract.
 * lwe_to_glwe: res = GLWE of rank k, key = VmpPMat(dnum, 1, k + 1, key_size) from embed(s_lwe); embed, then key-switch into res.
 * The *_tmp_bytes take the arguments of pgb_glwe_keyswitch_tmp_bytes: the staged rank-1 GLWE(s) plus the inner key-switch's scratch. */
int pgb_lwe_sample_extract_batched(pgb_module *m, pgb_vec_znx *res, const pgb_vec_znx *a, const pgb_batch *bt);
size_t pgb_lwe_keyswitch_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t a_base2k, const pgb_vmp_pmat *key,
                                   uint64_t key_base2k, uint64_t dsize, uint64_t batch);
int pgb_lwe_keyswitch_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a, uint64_t a_base2k,
                              const pgb_vmp_pmat *key, uint64_t key_base2k, uint64_t dsize, const pgb_batch *bt, void *scratch, size_t scratch_len);
size_t pgb_glwe_to_lwe_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t a_base2k, const pgb_vmp_pmat *key,
                                 uint64_t key_base2k, uint64_t dsize, uint64_t batch);
int pgb_glwe_to_lwe_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a, uint64_t a_base2k,
                            const pgb_vmp_pmat *key, uint64_t key_base2k, uint64_t dsize, const pgb_batch *bt, void *scratch, size_t scratch_len);
/* glwe_to_lwe at many coefficients, one key-switch per item: per item b, g_b = glwe_keyswitch(a_b) into a staged rank-1 GLWE of res.size
 * limbs of res_base2k (the key, routes and scratch rule of pgb_glwe_to_lwe_batched), and for j < n_index the LWE at res->data +
 * b*bt->stride_res + j*entry_stride is lwe_sample_extract(vec_znx_rotate(-index[j], g_b)): for limbs l < min(res.size, g.size),
 * b' = g[l][0][idx] and a'_t = g[l][1][idx + t] (idx + t < N) or -g[l][1][idx + t - N]; the other limbs are zeroed.  index = {0} gives
 * pgb_glwe_to_lwe_batched bit for bit.  This is "key-switch, then rotate": it is not bit-identical to rotating a before the key-switch (a
 * rotation negates wrapped digits without renormalising, and the key-switch's final rounding need not be odd-symmetric), but both orders
 * agree modulo 2^(res.size * res_base2k) within one unit of the last limb.
 * `index` is a HOST array of n_index in [1, N] coefficients, each below N (duplicates allowed); entry_stride a multiple of 8 of at least one
 * LWE when n_index > 1; bt->stride_res a multiple of 8 of at least (n_index-1)*entry_stride plus one LWE when count > 1; res must not
 * overlap a over the whole extent (PGB_ERR_ALIAS).  Every check runs before the first launch.  Scratch: the index table (one upload per
 * call) at its head, then `batch` staged GLWEs, then the key-switch's scratch; _tmp_bytes takes n_index before the batch count. */
size_t pgb_glwe_to_lwe_indexed_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t a_base2k, const pgb_vmp_pmat *key,
                                         uint64_t key_base2k, uint64_t dsize, uint64_t n_index, uint64_t batch);
int pgb_glwe_to_lwe_indexed_batched(pgb_module *m, pgb_vec_znx *res, uint64_t entry_stride, uint64_t res_base2k, const pgb_vec_znx *a,
                                    uint64_t a_base2k, const uint32_t *index, uint64_t n_index, const pgb_vmp_pmat *key, uint64_t key_base2k,
                                    uint64_t dsize, const pgb_batch *bt, void *scratch, size_t scratch_len);
size_t pgb_lwe_to_glwe_tmp_bytes(const pgb_module *m, uint64_t res_size, uint64_t a_size, uint64_t a_base2k, const pgb_vmp_pmat *key,
                                 uint64_t key_base2k, uint64_t dsize, uint64_t batch);
int pgb_lwe_to_glwe_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, const pgb_vec_znx *a, uint64_t a_base2k,
                            const pgb_vmp_pmat *key, uint64_t key_base2k, uint64_t dsize, const pgb_batch *bt, void *scratch, size_t scratch_len);

/* execute_standard (algorithm.rs:370-443, block_size == 1 keys): per LWE coefficient one GGSW x GLWE external product, X^{a_i} - 1, add;
 * one glwe_normalize_assign at the end.  Same argument conventions as pgb_cggi_blind_rotate_batched. */
size_t pgb_cggi_blind_rotate_standard_tmp_bytes(const pgb_module *m, uint64_t rank, uint64_t res_size, uint64_t res_base2k,
                                                const pgb_vmp_pmat *brk, uint64_t brk_base2k, uint64_t batch);
int pgb_cggi_blind_rotate_standard_batched(pgb_module *m, pgb_vec_znx *res, uint64_t res_base2k, const int64_t *lwe_2n, uint64_t n_lwe,
                                           const pgb_vec_znx *lut, const pgb_vmp_pmat *brk, uint64_t brk_base2k, const pgb_batch *bt,
                                           void *scratch, size_t scratch_len);

#ifdef __cplusplus
}
#endif
#endif
