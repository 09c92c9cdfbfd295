// big.cu -- VecZnxBig kernels: base-2^K carry propagation (K7) and the i128/i64 element-wise helpers (R13/R14/F7).
//
// One thread owns one coefficient and walks the limbs from the least significant one, keeping the carry in
// registers (the reference keeps it in a 3n scratch: ntt120/vec_znx_big.rs:1022-1024).  Control flow depends only
// on the shapes, so it is uniform across the grid.  BigT = __int128 (NTT120 big) or int64_t (FFT64 big and plain
// VecZnx); the arithmetic restates
//   poulpy-cpu-ref/src/reference/znx/normalization.rs:4-21        get_digit / get_carry
//   poulpy-cpu-ref/src/reference/ntt120/vec_znx_big.rs:367-446    same-base2k path   (+ :600-667 fused +-=)
//   poulpy-cpu-ref/src/reference/ntt120/vec_znx_big.rs:453-597    cross-base2k path  (+ :670-803 fused +-=)
//   poulpy-cpu-ref/src/reference/vec_znx/normalize.rs:52-380      the i64 twins
// per coefficient instead of per slice.
#include "internal.h"
#include "znx.cuh"

__device__ __forceinline__ long long apply_op(int op, long long r, long long x) {
    if (op == 0) return x;
    return op > 0 ? (long long)((unsigned long long)r + (unsigned long long)x) : (long long)((unsigned long long)r - (unsigned long long)x);
}

struct NormArgs {
    LimbSet res, a; // limb_stride = bytes between consecutive limbs of the selected column
    uint32_t n;
    int res_size, a_size;
    int res_k, a_k; // base2k
    int lsh;
    // same-base2k plan
    int res_end, res_start, a_end, a_start;
    // cross-base2k plan
    int a_tot_bits, res_tot_bits, a_start_bit, res_start_bit;
    int op;
};

template <typename T> __global__ void __launch_bounds__(256) normalize_inter_kernel(NormArgs p) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    const char *ab = p.a.base + (size_t)blockIdx.y * p.a.batch_stride;
    char *rb = p.res.base + (size_t)blockIdx.y * p.res.batch_stride;
#define A_AT(j) (reinterpret_cast<const T *>(ab + (size_t)(j) * p.a.limb_stride)[i])
#define R_AT(j) (reinterpret_cast<long long *>(rb + (size_t)(j) * p.res.limb_stride)[i])
    const int K = p.res_k, lsh = p.lsh, w = lsh == 0 ? K : K - lsh, op = p.op;
    T c = 0;
    const int a_out = p.a_size - p.a_start;
    for (int j = 0; j < a_out; j++) {
        const T x = A_AT(p.a_size - j - 1);
        const T d = get_digit<T>(w, x);
        const T co = get_carry<T>(w, x, d);
        if (j == 0) c = co;
        else {
            const T s = wadd<T>(wshl<T>(d, lsh), c);
            c = wadd<T>(co, get_carry<T>(K, s, get_digit<T>(K, s)));
        }
    }
    if (op == 0)
        for (int j = p.res_start; j < p.res_size; j++) R_AT(j) = 0;
    const int mid = p.a_start > p.a_end ? p.a_start - p.a_end : 0;
    for (int j = 0; j < mid; j++) {
        const T x = A_AT(p.a_start - j - 1);
        const T d = get_digit<T>(w, x);
        const T co = get_carry<T>(w, x, d);
        const T s = wadd<T>(wshl<T>(d, lsh), c);
        const T out = get_digit<T>(K, s);
        long long &r = R_AT(p.res_start - j - 1);
        r = apply_op(op, op == 0 ? 0 : r, (long long)out);
        c = wadd<T>(co, get_carry<T>(K, s, out));
    }
    for (int j = 0; j < p.res_end; j++) {
        long long &r = R_AT(p.res_end - j - 1);
        const T out = get_digit<T>(K, c); // res limb is zero: digit of 0 shifted + carry
        r = apply_op(op, op == 0 ? 0 : r, (long long)out);
        c = get_carry<T>(K, c, out);
    }
#undef A_AT
#undef R_AT
}

// cross-base2k: verbatim per-coefficient port of the three-carry bit-repacking loop
template <typename T> __global__ void __launch_bounds__(256) normalize_cross_kernel(NormArgs p) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    const char *ab = p.a.base + (size_t)blockIdx.y * p.a.batch_stride;
    char *rb = p.res.base + (size_t)blockIdx.y * p.res.batch_stride;
#define A_AT(j) (reinterpret_cast<const T *>(ab + (size_t)(j) * p.a.limb_stride)[i])
#define R_AT(j) (reinterpret_cast<long long *>(rb + (size_t)(j) * p.res.limb_stride)[i])
    const int aK = p.a_k, rK = p.res_k, lsh = p.lsh, w = lsh == 0 ? aK : aK - lsh, op = p.op;
    const int addop = op == 0 ? 1 : op;
    T a_norm = 0, res_carry = 0, a_carry = 0;
    if (op == 0)
        for (int j = 0; j < p.res_size; j++) R_AT(j) = 0;
    if (p.res_start == 0) return;
    const int a_out = p.a_size - p.a_start;
    for (int j = 0; j < a_out; j++) {
        const T x = A_AT(p.a_size - j - 1);
        const T d = get_digit<T>(w, x);
        const T co = get_carry<T>(w, x, d);
        if (j == 0) a_carry = co;
        else {
            const T s = wadd<T>(wshl<T>(d, lsh), a_carry);
            a_carry = wadd<T>(co, get_carry<T>(aK, s, get_digit<T>(aK, s)));
        }
    }
    int res_acc_left = rK;
    int res_limb = p.res_start - 1;
    const int mid = p.a_start > p.a_end ? p.a_start - p.a_end : 0;
    bool done = false;
    for (int j = 0; j < mid && !done; j++) {
        const int a_limb = p.a_start - j - 1;
        int a_take_left = aK;
        { // nfc_middle_step_i128
            const T x = A_AT(a_limb);
            const T d = get_digit<T>(w, x);
            const T co = get_carry<T>(w, x, d);
            const T s = wadd<T>(wshl<T>(d, lsh), a_carry);
            const T out = get_digit<T>(aK, s);
            a_norm = out;
            a_carry = wadd<T>(co, get_carry<T>(aK, s, out));
        }
        if (j == 0) {
            if ((p.a_tot_bits - p.a_start_bit) % aK != 0) {
                const int take = (p.a_tot_bits - p.a_start_bit) % aK;
                a_norm >>= take;
                a_take_left -= take;
            } else if ((p.res_tot_bits - p.res_start_bit) % rK != 0) {
                res_acc_left -= (p.res_tot_bits - p.res_start_bit) % rK;
            }
        }
        for (;;) {
            long long &r = R_AT(res_limb);
            const int a_take = min(min(aK, a_take_left), res_acc_left);
            if (a_take != 0) {
                const int scale = rK - res_acc_left;
                const T d = get_digit<T>(a_take, a_norm);
                a_norm = get_carry<T>(a_take, a_norm, d);
                r = apply_op(addop, r, (long long)((unsigned long long)(long long)d << scale));
                a_take_left -= a_take;
                res_acc_left -= a_take;
            }
            if (res_acc_left == 0 || a_limb == 0) {
                if (a_limb == 0 && a_take_left == 0) {
                    a_carry = wadd<T>(a_carry, a_norm);
                    if (res_acc_left != 0) {
                        const int scale = rK - res_acc_left;
                        const T d = get_digit<T>(res_acc_left, a_carry);
                        a_carry = get_carry<T>(res_acc_left, a_carry, d);
                        r = apply_op(addop, r, (long long)((unsigned long long)(long long)d << scale));
                    }
                    { // nfc_middle_step_assign(res_base2k, 0, r, res_carry)
                        const T ri = (T)r;
                        const T d = get_digit<T>(rK, ri);
                        const T co = get_carry<T>(rK, ri, d);
                        const T s = wadd<T>(d, res_carry);
                        const T out = get_digit<T>(rK, s);
                        r = (long long)out;
                        res_carry = wadd<T>(co, get_carry<T>(rK, s, out));
                    }
                    res_carry = wadd<T>(res_carry, a_carry);
                    done = true;
                    break;
                }
                if (res_limb == 0) {
                    done = true;
                    break;
                }
                res_acc_left += rK;
                res_limb -= 1;
            }
            if (a_take_left == 0) {
                a_carry = wadd<T>(a_carry, a_norm);
                break;
            }
        }
    }
    if (p.res_end != 0) {
        T cu = (p.a_start == p.a_end) ? a_carry : res_carry;
        for (int j = 0; j < p.res_end; j++) {
            long long &r = R_AT(p.res_end - j - 1);
            const bool last = j == p.res_end - 1;
            if (op == 0) {
                const T ri = (T)r;
                const T d = get_digit<T>(rK, ri);
                const T s = wadd<T>(d, cu);
                const T out = get_digit<T>(rK, s);
                if (!last) cu = wadd<T>(get_carry<T>(rK, ri, d), get_carry<T>(rK, s, out));
                r = (long long)out;
            } else {
                const T out = get_digit<T>(rK, cu);
                r = apply_op(op, r, (long long)out);
                if (!last) cu = get_carry<T>(rK, cu, out);
            }
        }
    }
#undef A_AT
#undef R_AT
}

static inline int64_t clampi(int64_t v, int64_t lo, int64_t hi) { return v < lo ? lo : (v > hi ? hi : v); }

// big_is_i128: NTT120 big; otherwise i64 (FFT64 big or plain VecZnx)
int big_normalize(pgb_module *m, bool big_is_i128, LimbSet res, int res_size, int res_k, int64_t res_offset, LimbSet a, int a_size,
                  int a_k, int op, uint32_t batch) {
    if (batch == 0) return PGB_OK;
    PGB_REQUIRE(res_k >= 1 && res_k <= 63 && a_k >= 1 && a_k <= 63, "normalize: base2k out of range");
    NormArgs p;
    memset(&p, 0, sizeof p);
    p.res = res;
    p.a = a;
    p.n = (uint32_t)m->n;
    p.res_size = res_size;
    p.a_size = a_size;
    p.res_k = res_k;
    p.a_k = a_k;
    p.op = op;
    const int64_t base = a_k; // the reference derives lsh / limbs_offset from a's base in both paths (equal bases in `inter`)
    int64_t lsh = res_offset % base, lo = res_offset / base;
    if (res_offset < 0 && lsh != 0) {
        lsh = (lsh + base) % base;
        lo -= 1;
    }
    p.lsh = (int)lsh;
    ProfScope _ps(m, PROF_NORMALIZE);
    dim3 block(256), grid(((uint32_t)m->n + 255) / 256, batch);
    if (res_k == a_k) {
        p.res_end = (int)clampi(-lo, 0, res_size);
        p.res_start = (int)clampi((int64_t)a_size - lo, 0, res_size);
        p.a_end = (int)clampi(lo, 0, a_size);
        p.a_start = (int)clampi((int64_t)res_size + lo, 0, a_size);
        if (big_is_i128) normalize_inter_kernel<i128><<<grid, block, 0, m->stream>>>(p);
        else normalize_inter_kernel<long long><<<grid, block, 0, m->stream>>>(p);
    } else {
        const int64_t a_tot = (int64_t)a_size * a_k, res_tot = (int64_t)res_size * res_k;
        const int64_t res_end_bit = clampi(-lo * a_k, 0, res_tot);
        const int64_t res_start_bit = clampi(a_tot - lo * a_k, 0, res_tot);
        const int64_t a_end_bit = clampi(lo * a_k, 0, a_tot);
        const int64_t a_start_bit = clampi(res_tot + lo * a_k, 0, a_tot);
        p.a_tot_bits = (int)a_tot;
        p.res_tot_bits = (int)res_tot;
        p.a_start_bit = (int)a_start_bit;
        p.res_start_bit = (int)res_start_bit;
        p.res_end = (int)(res_end_bit / res_k);
        p.res_start = (int)((res_start_bit + res_k - 1) / res_k);
        p.a_end = (int)(a_end_bit / a_k);
        p.a_start = (int)((a_start_bit + a_k - 1) / a_k);
        if (big_is_i128) normalize_cross_kernel<i128><<<grid, block, 0, m->stream>>>(p);
        else normalize_cross_kernel<long long><<<grid, block, 0, m->stream>>>(p);
    }
    m->launches++;
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

// ---- small element-wise helpers on big limbs ------------------------------------------------------------
struct BigEwArgs {
    LimbSet dst, a;
    uint32_t n;
};
template <typename T, int OP> __global__ void __launch_bounds__(256) big_ew_kernel(BigEwArgs p) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    T *d = reinterpret_cast<T *>(p.dst.base + (size_t)blockIdx.z * p.dst.batch_stride + (size_t)blockIdx.y * p.dst.limb_stride) + i;
    if (OP == BIG_ZERO) {
        *d = 0;
        return;
    }
    const long long x = reinterpret_cast<const long long *>(p.a.base + (size_t)blockIdx.z * p.a.batch_stride + (size_t)blockIdx.y * p.a.limb_stride)[i];
    if (OP == BIG_ADD_SMALL) *d = wadd<T>(*d, (T)x);
    else if (OP == BIG_SUB_SMALL) *d = wsub<T>(*d, (T)x);
    else if (OP == BIG_SUB_SMALL_NEG) *d = wsub<T>((T)x, *d);
    else *d = (T)x;
}
// res = -res (wrapping) over limb sets: the tail of vec_znx_big_sub_small_negate_assign
template <typename T> __global__ void __launch_bounds__(256) big_neg_kernel(BigEwArgs p) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    T *d = reinterpret_cast<T *>(p.dst.base + (size_t)blockIdx.z * p.dst.batch_stride + (size_t)blockIdx.y * p.dst.limb_stride) + i;
    *d = wsub<T>((T)0, *d);
}

int big_ew(pgb_module *m, bool big_is_i128, int op, LimbSet dst, LimbSet a, uint32_t jobs, uint32_t batch) {
    if (jobs == 0 || batch == 0) return PGB_OK;
    ProfScope _ps(m, PROF_ELEMENTWISE);
    BigEwArgs p = {dst, a, (uint32_t)m->n};
    dim3 block(256), grid(((uint32_t)m->n + 255) / 256, jobs, batch);
#define LAUNCH(T, OP) big_ew_kernel<T, OP><<<grid, block, 0, m->stream>>>(p)
    if (big_is_i128) {
        if (op == BIG_ADD_SMALL) LAUNCH(i128, BIG_ADD_SMALL);
        else if (op == BIG_FROM_SMALL) LAUNCH(i128, BIG_FROM_SMALL);
        else if (op == BIG_SUB_SMALL) LAUNCH(i128, BIG_SUB_SMALL);
        else if (op == BIG_SUB_SMALL_NEG) LAUNCH(i128, BIG_SUB_SMALL_NEG);
        else if (op == BIG_NEG) big_neg_kernel<i128><<<grid, block, 0, m->stream>>>(p);
        else LAUNCH(i128, BIG_ZERO);
    } else {
        if (op == BIG_ADD_SMALL) LAUNCH(long long, BIG_ADD_SMALL);
        else if (op == BIG_FROM_SMALL) LAUNCH(long long, BIG_FROM_SMALL);
        else if (op == BIG_SUB_SMALL) LAUNCH(long long, BIG_SUB_SMALL);
        else if (op == BIG_SUB_SMALL_NEG) LAUNCH(long long, BIG_SUB_SMALL_NEG);
        else if (op == BIG_NEG) big_neg_kernel<long long><<<grid, block, 0, m->stream>>>(p);
        else LAUNCH(long long, BIG_ZERO);
    }
#undef LAUNCH
    m->launches++;
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

// ---- coefficient-domain rotate (reference/znx/rotate.rs:3-26): res = a * X^p mod (X^n + 1) -----------------
struct RotArgs {
    LimbSet dst, a;
    uint32_t n;
    const long long *p_dev; // optional per-batch rotation amounts (device), else p
    long long p;
    uint32_t p_stride;      // element stride between batch items in p_dev
};
__global__ void __launch_bounds__(256) rotate_kernel(RotArgs q) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; // destination index
    if (i >= q.n) return;
    const long long p = q.p_dev ? q.p_dev[(size_t)blockIdx.z * q.p_stride] : q.p;
    const long long *src = reinterpret_cast<const long long *>(q.a.base + (size_t)blockIdx.z * q.a.batch_stride + (size_t)blockIdx.y * q.a.limb_stride);
    long long *dst = reinterpret_cast<long long *>(q.dst.base + (size_t)blockIdx.z * q.dst.batch_stride + (size_t)blockIdx.y * q.dst.limb_stride);
    bool neg;
    const long long v = rotate_read([&](uint32_t k) { return src[k]; }, i, p, q.n, &neg);
    dst[i] = neg ? (long long)(0ull - (unsigned long long)v) : v;
}
int znx_rotate(pgb_module *m, LimbSet dst, LimbSet a, long long p, const long long *p_dev, uint32_t p_stride, uint32_t jobs, uint32_t batch) {
    if (jobs == 0 || batch == 0) return PGB_OK;
    ProfScope _ps(m, PROF_OTHER);
    RotArgs q = {dst, a, (uint32_t)m->n, p_dev, p, p_stride};
    dim3 block(256), grid(((uint32_t)m->n + 255) / 256, jobs, batch);
    rotate_kernel<<<grid, block, 0, m->stream>>>(q);
    m->launches++;
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

// i64 element-wise helpers of the coefficient domain: dst (op)= a, and dst = rotate(p, a) - a (vec_znx_mul_xp_minus_one)
struct ZnxEwArgs {
    LimbSet dst, a;
    uint32_t n;
    int op; // 0 add_assign, 1 sub_assign, 2 mul_xp_minus_one (dst = X^p a - a), 3 copy, 4 negate (dst = -a)
    const long long *p_dev;
    long long p;
    uint32_t p_stride;
};
__global__ void __launch_bounds__(256) znx_ew_kernel(ZnxEwArgs q) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= q.n) return;
    const long long *src = reinterpret_cast<const long long *>(q.a.base + (size_t)blockIdx.z * q.a.batch_stride + (size_t)blockIdx.y * q.a.limb_stride);
    long long *dst = reinterpret_cast<long long *>(q.dst.base + (size_t)blockIdx.z * q.dst.batch_stride + (size_t)blockIdx.y * q.dst.limb_stride);
    if (q.op == 0) {
        dst[i] = (long long)((unsigned long long)dst[i] + (unsigned long long)src[i]);
    } else if (q.op == 1) {
        dst[i] = (long long)((unsigned long long)dst[i] - (unsigned long long)src[i]);
    } else if (q.op == 3) {
        dst[i] = src[i];
    } else if (q.op == 4) {
        dst[i] = (long long)(0ull - (unsigned long long)src[i]);
    } else {
        const long long p = q.p_dev ? q.p_dev[(size_t)blockIdx.z * q.p_stride] : q.p;
        const uint32_t n = q.n, mp = (uint32_t)(p & (long long)(2 * n - 1));
        const uint32_t s = (i - mp) & (2 * n - 1); // coefficient s of a lands on i (negated when it wrapped once)
        const unsigned long long r = s < n ? (unsigned long long)src[s] : 0ull - (unsigned long long)src[s - n];
        dst[i] = (long long)(r - (unsigned long long)src[i]);
    }
}
int znx_ew(pgb_module *m, int op, LimbSet dst, LimbSet a, long long p, const long long *p_dev, uint32_t p_stride, uint32_t jobs, uint32_t batch) {
    if (jobs == 0 || batch == 0) return PGB_OK;
    ProfScope _ps(m, PROF_ELEMENTWISE);
    ZnxEwArgs q = {dst, a, (uint32_t)m->n, op, p_dev, p, p_stride};
    znx_ew_kernel<<<dim3(((uint32_t)m->n + 255) / 256, jobs, batch), 256, 0, m->stream>>>(q);
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

// vec_znx_automorphism (reference/znx/automorphism.rs:1-17): a(X) -> a(X^p); thread i scatters coefficient i to i*p mod 2n with the
// negacyclic sign (a permutation: race-free)
struct AutoArgs {
    LimbSet dst, a;
    uint32_t n;
    long long p;
};
template <typename T> __global__ void __launch_bounds__(256) znx_automorphism_kernel(AutoArgs q) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= q.n) return;
    const T *src = reinterpret_cast<const T *>(q.a.base + (size_t)blockIdx.z * q.a.batch_stride + (size_t)blockIdx.y * q.a.limb_stride);
    T *dst = reinterpret_cast<T *>(q.dst.base + (size_t)blockIdx.z * q.dst.batch_stride + (size_t)blockIdx.y * q.dst.limb_stride);
    const uint32_t mask = 2 * q.n - 1, p2n = (uint32_t)(q.p & (long long)mask);
    const uint32_t k = (uint32_t)(((unsigned long long)i * p2n) & mask);
    const T v = src[i];
    if (k < q.n) dst[k] = v;
    else dst[k - q.n] = (T)((typename BT<T>::U)0 - (typename BT<T>::U)v); // wrapping_neg
}
// big_is_i128: the limbs are i128 (NTT120 VecZnxBig, ntt120/vec_znx_big.rs:1462-1497) instead of i64 (VecZnx and the FFT64 VecZnxBig)
int znx_automorphism(pgb_module *m, LimbSet dst, LimbSet a, long long p, uint32_t jobs, uint32_t batch, bool big_is_i128) {
    if (jobs == 0 || batch == 0) return PGB_OK;
    ProfScope _ps(m, PROF_ELEMENTWISE);
    AutoArgs q = {dst, a, (uint32_t)m->n, p};
    const dim3 grid(((uint32_t)m->n + 255) / 256, jobs, batch);
    if (big_is_i128) znx_automorphism_kernel<i128><<<grid, 256, 0, m->stream>>>(q);
    else znx_automorphism_kernel<long long><<<grid, 256, 0, m->stream>>>(q);
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

// vec_znx_rsh_assign (reference/vec_znx/shift.rs:186-243): right shift by k bits in base 2^K, in place, one thread per coefficient walking
// the limbs with the carry in a register (rsh_assign_coeff, znx.cuh)
struct RshArgs {
    LimbSet r;
    uint32_t n;
    int size, K, k;
};
__global__ void __launch_bounds__(256) znx_rsh_assign_kernel(RshArgs q) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= q.n) return;
    char *rb = q.r.base + (size_t)blockIdx.y * q.r.batch_stride;
    rsh_assign_coeff([&](int j) -> long long & { return reinterpret_cast<long long *>(rb + (size_t)j * q.r.limb_stride)[i]; }, q.size, q.K, q.k);
}
int znx_rsh_assign(pgb_module *m, LimbSet r, int size, int base2k, int k, uint32_t batch, uint32_t words) {
    if (size == 0 || batch == 0) return PGB_OK;
    ProfScope _ps(m, PROF_NORMALIZE);
    const uint32_t nw = words ? words : (uint32_t)m->n; // words per limb to shift: n, or cols * n for all (adjacent) columns of a limb at once
    RshArgs q = {r, nw, size, base2k, k};
    znx_rsh_assign_kernel<<<dim3((nw + 255) / 256, batch), 256, 0, m->stream>>>(q);
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}

// raw byte-wise zero / copy over limb sets (both flavours)
struct RawArgs {
    LimbSet dst, a;
    uint32_t words; // uint4 words per limb
    int zero;
};
__global__ void __launch_bounds__(256) raw_kernel(RawArgs p) {
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= p.words) return;
    uint4 *d = reinterpret_cast<uint4 *>(p.dst.base + (size_t)blockIdx.z * p.dst.batch_stride + (size_t)blockIdx.y * p.dst.limb_stride) + u;
    if (p.zero) *d = make_uint4(0, 0, 0, 0);
    else *d = *(reinterpret_cast<const uint4 *>(p.a.base + (size_t)blockIdx.z * p.a.batch_stride + (size_t)blockIdx.y * p.a.limb_stride) + u);
}
int raw_limbs(pgb_module *m, bool zero, LimbSet dst, LimbSet a, uint64_t limb_bytes, uint32_t jobs, uint32_t batch) {
    if (jobs == 0 || batch == 0) return PGB_OK;
    ProfScope _ps(m, PROF_ELEMENTWISE);
    RawArgs p = {dst, a, (uint32_t)(limb_bytes / 16), zero ? 1 : 0};
    dim3 block(256), grid((p.words + 255) / 256, jobs, batch);
    raw_kernel<<<grid, block, 0, m->stream>>>(p);
    m->launches++;
    PGB_CHECK_CUDA(cudaGetLastError());
    return PGB_OK;
}
