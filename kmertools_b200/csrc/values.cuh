// values.cuh — the per-window decoder and the value semantics shared by every row format: byte -> 2-bit code,
// normalisation divisor and count -> output element.  kernels.cuh (dense rows) and sparse_kernels.cuh (CSR rows)
// both include it, so a dense and a sparse row hold the same bits for the same count.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace ktb {

constexpr int OUT_U32 = 0, OUT_F32 = 1, OUT_F64 = 2;
constexpr int NORM_COUNTS = 0, NORM_CLI = 1, NORM_PY = 2;

// ------------------------------------------------------------------------------------------------
// byte -> 2-bit code, 4 = ambiguous.  Same mapping as SEQ_NT4_TABLE (kmer/src/kmer.rs:6-15):
// bytes 0..3 -> themselves, A/a 0, C/c 1, G/g 2, T/t/U/u 3, everything else 4.  Arithmetic instead
// of a table: ((b>>1)^(b>>2))&3 sends A,C,G,T/U (either case) to 0,1,2,3.
__device__ __forceinline__ uint32_t nt4_code(uint32_t b) {
    const uint32_t u = b & 0xDFu;
    const uint32_t code = ((b >> 1) ^ (b >> 2)) & 3u;
    const bool letter = (u == 'A') | (u == 'C') | (u == 'G') | (u == 'T') | (u == 'U');
    return b < 4u ? b : (letter ? code : 4u);
}

// Correctly rounded c / d in f32 for integers 0 <= c <= d < 2^24: q0 = c * RN(1/d), one exact
// residual and one correction FMA.  Because c/d has a denominator below 2^24 it can never sit within
// 2^-49 (relative) of an f32 rounding boundary without being on it, so this equals
// (float)((double)c / (double)d), i.e. the reference's f64 quotient rounded once.  Checked
// exhaustively for d <= 4096 on the CPU in tests/test_host_logic.py (same FMA sequence in C).
__device__ __forceinline__ float quot_f32(float c, float d, float rinv) {
    const float q0 = c * rinv;
    const float rem = fmaf(-q0, d, c);
    return fmaf(rem, rinv, q0);
}

// divisor of the normalisation step as an integer (oligo.rs:255-257; pybindings/src/oligo.rs:58-66)
__device__ __forceinline__ uint64_t norm_divisor(uint64_t total, int norm_mode, int canonical) {
    uint64_t t = (norm_mode == NORM_PY && !canonical) ? 2 * total : total;
    return t > 1 ? t : 1;
}

template <int OUT> struct OutT;
template <> struct OutT<OUT_U32> { using type = uint32_t; };
template <> struct OutT<OUT_F32> { using type = float; };
template <> struct OutT<OUT_F64> { using type = double; };

// Converts one count to the output element.  dF/rinv are used for f32 when the divisor is exactly
// representable (< 2^24); otherwise, and for f64, the division is done in double like the reference.
template <int OUT>
__device__ __forceinline__ typename OutT<OUT>::type make_out(uint32_t cnt, bool norm, bool small_div,
                                                             float dF, float rinv, double dD) {
    if constexpr (OUT == OUT_U32) {
        return cnt;
    } else if constexpr (OUT == OUT_F32) {
        if (!norm) return (float)cnt;
        if (small_div) return quot_f32((float)cnt, dF, rinv);
        return (float)((double)cnt / dD);
    } else {
        if (!norm) return (double)cnt;
        return (double)cnt / dD;
    }
}

}  // namespace ktb
