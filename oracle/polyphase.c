/*
 * polyphase.c -- CPU definition of the polyphase resampling of batches
 * (af_batch_set_resampler, AF_RESAMPLE_POLYPHASE).
 *
 * TEST INFRASTRUCTURE ONLY, like oracle.c: the product never includes, links or
 * calls it.  The GPU's PCM is checked against it bit for bit; tests pin it to
 * scipy.signal.resample_poly and its tap table to scipy's firwin.
 *
 * Build: gcc -O2 -ffp-contract=off -fno-fast-math -fPIC -shared (polyphase.py
 * compiles it on first use).  The sum is an explicit fmaf chain, so no
 * contraction may add or remove roundings elsewhere.
 */
#include <math.h>
#include <stddef.h>
#include <stdint.h>

#define ORC_API __attribute__((visibility("default")))

/* h holds n_taps = 2L + 1 taps (the library's af_debug_polyphase_filter).
 *   y[n] = sum_k m[k] * h[n p + L - k q] over every k with
 *          0 <= n p + L - k q <= 2L, ascending k, m[k] = 0 outside [0, n_in),
 *          as acc = fmaf(m[k], h[i], acc) from +0.0f.
 * p == q == 1 copies (zero past n_in). */
ORC_API void orc_resample_polyphase(const float *mono, size_t n_in, uint32_t p, uint32_t q, const float *h,
                                    size_t n_taps, size_t n_out, float *y)
{
    const long long L = (long long)(n_taps - 1) / 2;
    for (size_t n = 0; n < n_out; ++n) {
        if (p == 1 && q == 1) { y[n] = n < n_in ? mono[n] : 0.0f; continue; }
        const long long t = (long long)n * p + L;
        const long long lo = t - 2 * L;                                 /* first k: ceil(lo / q) */
        long long k = lo >= 0 ? (lo + q - 1) / q : -((-lo) / (long long)q);
        float acc = 0.0f;
        for (; t - k * (long long)q >= 0; ++k) {
            const float m = k >= 0 && k < (long long)n_in ? mono[k] : 0.0f;
            acc = fmaf(m, h[t - k * (long long)q], acc);
        }
        y[n] = acc;
    }
}
