// znx.cuh -- per-coefficient device code of the coefficient domain, shared by the kernels of big.cu and the packing kernels of pack.cu:
// the digit / carry arithmetic of reference/znx/normalization.rs:4-21, the index and sign of a negacyclic rotation, and the carry chains
// of vec_znx_rsh_assign and of the same-base2k vec_znx_normalize_assign on one coefficient.
#pragma once
#include "common.cuh"

template <typename T> struct BT;
template <> struct BT<i128> { typedef u128 U; static constexpr int BITS = 128; };
template <> struct BT<long long> { typedef unsigned long long U; static constexpr int BITS = 64; };

template <typename T> __device__ __forceinline__ T wadd(T a, T b) { return (T)((typename BT<T>::U)a + (typename BT<T>::U)b); }
template <typename T> __device__ __forceinline__ T wsub(T a, T b) { return (T)((typename BT<T>::U)a - (typename BT<T>::U)b); }
template <typename T> __device__ __forceinline__ T wshl(T a, int s) { return (T)((typename BT<T>::U)a << s); }
template <typename T> __device__ __forceinline__ T get_digit(int k, T x) {
    return (T)((typename BT<T>::U)x << (BT<T>::BITS - k)) >> (BT<T>::BITS - k);
}
template <typename T> __device__ __forceinline__ T get_carry(int k, T x, T d) { return wsub<T>(x, d) >> k; }

// rotate_kernel's read (reference/znx/rotate.rs:3-26): coefficient i of X^p a is ld(k) for the source index k of a, negated when *neg
template <typename Ld> __device__ __forceinline__ auto rotate_read(Ld ld, uint32_t i, long long p, uint32_t n, bool *neg) -> decltype(ld(0u)) {
    const uint32_t mp_2n = (uint32_t)(p & (long long)(2 * n - 1));
    const uint32_t mp_1n = mp_2n & (n - 1);
    const bool neg_first = mp_2n < n;
    decltype(ld(0u)) v;
    if (i < mp_1n) {
        v = ld(n - mp_1n + i);
        *neg = neg_first;
    } else {
        v = ld(i - mp_1n);
        *neg = !neg_first;
    }
    return v;
}
// the source index of coefficient i of X^p a, through rotate_read
__device__ __forceinline__ uint32_t rotate_src(uint32_t i, long long p, uint32_t n, bool *neg) {
    return rotate_read([](uint32_t k) { return k; }, i, p, n, neg);
}

// vec_znx_rsh_assign (reference/vec_znx/shift.rs:186-243) on one coefficient: R(j) is its word in limb j (a long long &).  Right shift by k
// bits in base 2^K with the carry in a register; the three loops follow the reference verbatim, including the order of its last loop (zero
// limb j, then step on limb steps-1-j), which is only the arithmetic shift for steps <= 1 or k a multiple of K.
template <typename Acc> __device__ __forceinline__ void rsh_assign_coeff(Acc R, int size, int K, int k) {
    typedef long long T;
    const int k_rem = k % K;
    const int steps = k / K + (k_rem ? 1 : 0), lsh = (K - k_rem) % K, w = lsh == 0 ? K : K - lsh;
    T c = 0;
    for (int j = 0; j < steps; j++) {
        const T x = R(size - j - 1);
        const T d = get_digit<T>(w, x), co = get_carry<T>(w, x, d);
        if (j == 0) c = co;
        else {
            const T s = wadd<T>(wshl<T>(d, lsh), c);
            c = wadd<T>(co, get_carry<T>(K, s, get_digit<T>(K, s)));
        }
    }
    for (int j = 0; j < size - steps; j++) {
        const T x = R(size - steps - j - 1);
        const T d = get_digit<T>(w, x), co = get_carry<T>(w, x, d);
        const T s = wadd<T>(wshl<T>(d, lsh), c);
        const T out = get_digit<T>(K, s);
        c = wadd<T>(co, get_carry<T>(K, s, out));
        R(size - j - 1) = out;
    }
    for (int j = 0; j < steps; j++) {
        R(j) = 0;
        const T x = R(steps - j - 1);
        const T d = get_digit<T>(w, x);
        const T s = wadd<T>(wshl<T>(d, lsh), c);
        const T out = get_digit<T>(K, s);
        if (j != 0) c = wadd<T>(get_carry<T>(w, x, d), get_carry<T>(K, s, out));
        R(steps - j - 1) = out;
    }
}

// vec_znx_normalize_assign (reference/vec_znx/normalize.rs:403-425) on one coefficient: the plan normalize_inter_kernel runs for equal
// base2k, equal sizes and offset 0 (lsh = 0, every limb in the middle loop), from the last limb up; the last carry is dropped.  in(j)
// reads limb j, out(j, v) writes its normalised value (the same word for the in-place form; limb j is read before it is written).
template <typename In, typename Out> __device__ __forceinline__ void normalize_coeff(In in, Out out, int size, int K) {
    typedef long long T;
    T c = 0;
    for (int j = 0; j < size; j++) {
        const T x = in(size - j - 1);
        const T d = get_digit<T>(K, x), co = get_carry<T>(K, x, d);
        const T s = wadd<T>(d, c);
        const T o = get_digit<T>(K, s);
        out(size - j - 1, o);
        c = wadd<T>(co, get_carry<T>(K, s, o));
    }
}
