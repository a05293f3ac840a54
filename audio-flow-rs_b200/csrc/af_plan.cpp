// af_plan.cpp -- host-side planning (see af_plan.h).
#include "af_plan.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>
#include <numeric>
#include <queue>

namespace af {

void RsRecurrence::init(uint32_t in, uint32_t out)
{
    in_rate = in; out_rate = out;
    passthrough = (in == out);                       // resampler.rs:33-40
    const uint32_t g = std::gcd(in, out);
    p = in / g; q = out / g;
    const double ratio = (double)out / (double)in;   // intended resample_ratio (SURVEY R4)
    t = 1.0 / ratio;
    end_idx = (long)RS_CHUNK - (RS_POLY + 1) - (long)std::ceil(t);
    exact = (q & (q - 1)) == 0 && q <= (1u << 20) && t == (double)p / (double)q;
    last_index = -(double)(RS_POLY / 2);
    chunks = 0; n_out = 0;
}

uint32_t RsRecurrence::step(std::vector<float> *frac)
{
    double idx = last_index;
    uint32_t n = 0;
    const double end = (double)end_idx;
    while (idx < end) {
        idx += t;
        const double fl = std::floor(idx);
        if (frac) frac->push_back((float)(idx - fl));
        ++n;
    }
    last_index = idx - (double)RS_CHUNK;
    chunks += 1;
    n_out += n;
    return n;
}

uint64_t rs_exact_count(const RsRecurrence &r, uint64_t chunks)
{
    if (chunks == 0) return 0;
    // outputs n >= 0 with -4 + n t < 128 (chunks - 1) + end_idx   <=>   n p < (128 chunks - 128 + end_idx + 4) q
    const uint64_t bound = (uint64_t)((long long)RS_CHUNK * (long long)chunks - RS_CHUNK + r.end_idx + 4);
    const __uint128_t num = (__uint128_t)bound * r.q;
    return (uint64_t)((num + r.p - 1) / r.p);
}

void build_fft_tables(FftTables *t)
{
    std::memset(t, 0, sizeof(*t));
    for (int n = 0; n < WIN; ++n) t->window[n] = (float)(0.5 - 0.5 * std::cos(2.0 * M_PI * (double)n / (double)WIN));
    for (int p = 0; p < 8; ++p)
        for (int l = 0; l < 16; ++l) {
            const int sa = 2 * p, sb = 2 * p + 1;
            const int ka = (sa >> 2) + 4 * (sa & 3), kb = (sb >> 2) + 4 * (sb & 3);
            const double aa = -2.0 * M_PI * (double)(l * ka) / 256.0, ab = -2.0 * M_PI * (double)(l * kb) / 256.0;
            t->tw1p[p * 16 + l] = make_float4((float)std::cos(aa), (float)std::cos(ab), (float)std::sin(aa), (float)std::sin(ab));
        }
    for (int r = 0; r < 4; ++r)
        for (int l = 0; l < 16; ++l) {
            const double aa = -2.0 * M_PI * (double)(l + 16 * r) / 512.0, ab = -2.0 * M_PI * (double)(l + 16 * (r + 4)) / 512.0;
            t->tw2p[r * 16 + l] = make_float4((float)std::cos(aa), (float)std::cos(ab), (float)std::sin(aa), (float)std::sin(ab));
        }
}

static double hz_to_mel_htk(double f) { return 2595.0 * std::log10(1.0 + f / 700.0); }
static double mel_to_hz_htk(double m) { return 700.0 * (std::pow(10.0, m / 2595.0) - 1.0); }

bool build_mel_tables(uint32_t n_mels, float f_min, float f_max, MelTables *t)
{
    std::memset(t, 0, sizeof(*t));
    if (n_mels == 0 || n_mels > MAX_MELS) return false;
    std::vector<double> pts(n_mels + 2);
    const double m_lo = hz_to_mel_htk((double)f_min), m_hi = hz_to_mel_htk((double)f_max);
    for (uint32_t i = 0; i < n_mels + 2; ++i)
        pts[i] = mel_to_hz_htk(m_lo + (m_hi - m_lo) * (double)i / (double)(n_mels + 1));
    // per-filter nonzero ranges
    std::vector<std::vector<float>> wts(n_mels);
    std::vector<int> los(n_mels, 0);
    for (uint32_t m = 0; m < n_mels; ++m) {
        int lo = -1, hi = -1;
        std::vector<float> w(NBIN, 0.0f);
        for (int k = 0; k < NBIN; ++k) {
            const double f = (double)k * (double)OUT_RATE / (double)NFFT;
            const double up = (f - pts[m]) / (pts[m + 1] - pts[m]);
            const double dn = (pts[m + 2] - f) / (pts[m + 2] - pts[m + 1]);
            double v = up < dn ? up : dn;
            if (v < 0.0) v = 0.0;
            w[k] = (float)v;
            if (w[k] != 0.0f) { if (lo < 0) lo = k; hi = k + 1; }
        }
        if (lo < 0) { lo = 0; hi = 0; }
        los[m] = lo;
        for (int k = lo; k < hi; ++k) wts[m].push_back(w[k] * 0.25f);    // pbuf holds 4 |X|^2
    }
    // every filter starts on a multiple of four bins (the mel warps read the power rows with LDS.128): zeros in front
    for (uint32_t m = 0; m < n_mels; ++m) {
        const int shift = los[m] & 3;
        if (shift) { wts[m].insert(wts[m].begin(), (size_t)shift, 0.0f); los[m] -= shift; }
    }
    // quads of adjacent filters share a trip count; weights interleaved per step: [a0..a3][b0..b3][c0..c3][d0..d3]
    const uint32_t cap16 = sizeof(t->w) / sizeof(float) / 16;
    const uint32_t n_quads = (n_mels + 3) / 4;
    uint32_t off16 = 0;
    std::vector<uint32_t> cost(n_quads, 0);
    uint32_t total = 0;
    for (uint32_t qd = 0; qd < n_quads; ++qd) {
        size_t longest = 0;
        for (uint32_t u = 0; u < 4; ++u)
            if (4 * qd + u < n_mels) longest = std::max(longest, wts[4 * qd + u].size());
        const uint32_t c4 = (uint32_t)((longest + 3) / 4);
        if (off16 + c4 > cap16) return false;
        MelQuad &Q = t->quad[qd];
        Q.c4 = c4; Q.woff = 64u * off16; Q.tcol = MEL_NO_TMEM;
        for (uint32_t u = 0; u < 4; ++u) {
            const uint32_t m = 4 * qd + u;
            if (m >= n_mels) { Q.off[u] = 0; continue; }                   // all-zero weights
            // the padded reads must stay inside the power row (PB_COLS floats): start earlier with zero weights in front
            int excess = los[m] + 4 * (int)c4 - PB_COLS;
            if (excess > 0) {
                excess = (excess + 3) & ~3;
                if (excess > los[m]) return false;
                wts[m].insert(wts[m].begin(), (size_t)excess, 0.0f);
                los[m] -= excess;
                if (wts[m].size() > 4 * (size_t)c4) return false;
            }
            Q.off[u] = 4u * (uint32_t)los[m];
            for (size_t k = 0; k < wts[m].size(); ++k) t->w[16 * (off16 + k / 4) + 4 * u + (k & 3)] = wts[m][k];
        }
        off16 += c4;
        cost[qd] = 24u * c4 + 40u;                     // warp instructions per quad in role_mel
        total += cost[qd];
    }
    t->n_w = (uint16_t)(16 * off16); t->n_mels = (uint16_t)n_mels;
    // split the filter quads over the mel warps by cost (greedy prefix split)
    uint32_t q = 0, acc = 0;
    t->quad_begin[0] = 0;
    for (int j = 1; j < MEL_WARPS; ++j) {
        const uint32_t target = (uint32_t)(((uint64_t)total * (uint64_t)j) / MEL_WARPS);
        while (q < n_quads && acc + cost[q] / 2 < target) acc += cost[q++];
        t->quad_begin[j] = (uint16_t)q;
    }
    t->quad_begin[MEL_WARPS] = (uint16_t)n_quads;
    // tensor-memory residence of the weights: mel warp j sits on scheduler j in every layout (warp_role) and can only
    // address the TMEM lane quarter j; a quad takes 16 columns per step after the FFT constants
    uint32_t next_col[4] = {TM_MEL0, TM_MEL0, TM_MEL0, TM_MEL0};
    for (int j = 0; j < MEL_WARPS; ++j) {
        uint32_t &col = next_col[j & 3];
        for (uint32_t qd = t->quad_begin[j]; qd < t->quad_begin[j + 1]; ++qd) {
            const uint32_t need = 16u * t->quad[qd].c4;
            if (t->quad[qd].c4 <= 8 && col + need <= TMEM_COLS) { t->quad[qd].tcol = col; col += need; }
        }
    }
    return true;
}

static inline float bits_to_f32(uint32_t b) { float f; std::memcpy(&f, &b, 4); return f; }

float vad_energy_threshold(float threshold_db)
{
    // energy_to_dbfs (vad.rs:171-176): e <= 0 -> -inf; else 20 * log10(e).  is_speech = dbfs > thr.
    auto speech = [&](float e) { return 20.0f * log10f(e) > threshold_db; };
    const uint32_t inf_bits = 0x7f800000u;
    if (!speech(bits_to_f32(inf_bits))) return std::numeric_limits<float>::quiet_NaN();
    uint32_t lo = 1, hi = inf_bits;              // invariant: speech(hi) true; everything below lo false
    if (speech(bits_to_f32(lo))) return bits_to_f32(lo);
    while (hi - lo > 1) {
        const uint32_t mid = lo + (hi - lo) / 2;
        if (speech(bits_to_f32(mid))) hi = mid; else lo = mid;
    }
    return bits_to_f32(hi);
}

uint64_t tile_order_max_steps(const std::vector<uint32_t> &steps, const std::vector<uint32_t> &order, uint32_t n_ctas)
{
    if (n_ctas == 0) return 0;
    std::vector<uint64_t> load(n_ctas, 0);
    for (size_t i = 0; i < order.size(); ++i) load[i % n_ctas] += steps[order[i]];
    return *std::max_element(load.begin(), load.end());
}

std::vector<uint32_t> balance_tile_order(const std::vector<uint32_t> &steps, uint32_t n_ctas)
{
    const size_t n = steps.size();
    std::vector<uint32_t> order(n);
    std::iota(order.begin(), order.end(), 0u);
    if (n_ctas == 0 || n <= n_ctas) return order;          // one tile per CTA at most: nothing to balance
    // CTA c walks a fixed number of positions (ceil or floor of n / n_ctas).  Longest tile first, each to the least
    // loaded CTA that still has a free position; ties go to the lower CTA index.
    std::vector<uint32_t> by_len(order);
    std::stable_sort(by_len.begin(), by_len.end(), [&](uint32_t a, uint32_t b) { return steps[a] > steps[b]; });
    std::vector<uint64_t> load(n_ctas, 0);
    std::vector<uint32_t> used(n_ctas, 0);
    std::vector<uint32_t> balanced(n);
    using Key = std::pair<uint64_t, uint32_t>;               // (load, CTA)
    std::priority_queue<Key, std::vector<Key>, std::greater<Key>> open;
    for (uint32_t c = 0; c < n_ctas; ++c) open.push({0, c});
    for (const uint32_t t : by_len) {
        const uint32_t c = open.top().second;
        open.pop();
        balanced[c + (size_t)used[c] * n_ctas] = t;
        load[c] += steps[t];
        if (c + (size_t)(++used[c]) * n_ctas < n) open.push({load[c], c});
    }
    if (tile_order_max_steps(steps, balanced, n_ctas) < tile_order_max_steps(steps, order, n_ctas)) order.swap(balanced);
    return order;
}

}  // namespace af
