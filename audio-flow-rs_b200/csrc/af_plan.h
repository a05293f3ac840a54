// af_plan.h -- host-side planning: the chunk recurrence of the reference resampler, FFT / mel
// tables, the VAD threshold in the energy domain.  Pure host code (no CUDA calls).
#pragma once
#include <cstdint>
#include <vector>

#include "af_common.cuh"

namespace af {

// The f64 position recurrence of rubato 0.16.2 FastFixedIn::process_into_buffer as driven by
// resampler.rs:132-166 (128-frame chunks).  One instance == one resampler's position state.
struct RsRecurrence {
    uint32_t in_rate = 0, out_rate = 0;
    uint32_t p = 1, q = 1;        // in/out reduced: exact step = p / q
    double t = 1.0;               // 1.0 / (out / in), exactly as rubato computes it
    long end_idx = 0;             // chunk - (POLY + 1) - ceil(t)
    bool passthrough = false;
    bool exact = false;           // q is a power of two and t == p / q: the recurrence has no rounding
    double last_index = -4.0;     // -(POLYNOMIAL_LEN / 2)
    uint64_t chunks = 0;          // chunks processed so far
    uint64_t n_out = 0;           // outputs produced so far

    void init(uint32_t in, uint32_t out);
    // advance by one chunk; appends the f32 fractional offsets of its outputs to `frac` (if non-null)
    uint32_t step(std::vector<float> *frac);
    uint32_t mode() const { return passthrough ? RS_PASSTHROUGH : (exact ? RS_EXACT : RS_TABLE); }
};

// closed-form number of outputs after `chunks` chunks when the recurrence is exact
uint64_t rs_exact_count(const RsRecurrence &r, uint64_t chunks);

void build_fft_tables(FftTables *t);
// HTK mel filterbank, triangular, evaluated at bin centres, no normalisation; weights * 1/4
bool build_mel_tables(uint32_t n_mels, float f_min, float f_max, MelTables *t);
// smallest f32 e with 20*log10f(e) > threshold_db under the host libm; NaN if none
float vad_energy_threshold(float threshold_db);
// Launch order of the tiles of one fused launch over n_ctas CTAs, CTA c running the tiles at positions c, c + n_ctas,
// c + 2 n_ctas, ...: order[i] is the tile (index into steps) placed at position i, chosen so that the CTAs' step counts
// are as even as the fixed number of positions each CTA walks allows.  Never more steps on the busiest CTA than the
// identity order gives.
std::vector<uint32_t> balance_tile_order(const std::vector<uint32_t> &steps, uint32_t n_ctas);
// steps on the busiest CTA when the tiles run in that order
uint64_t tile_order_max_steps(const std::vector<uint32_t> &steps, const std::vector<uint32_t> &order, uint32_t n_ctas);

}  // namespace af
