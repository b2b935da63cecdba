// K7 — sample-rate conversion to 16 kHz on the device: the filter design and its table (SURVEY §8(f) row N3), what the reference
// obtains from librosa.load(sr=16000) / librosa.resample (/root/reference/easywakeword/wakeword.py:588, 866-870;
// examples/tune_threshold.py:33-47; soxr HQ underneath).  soxr is not restated bit for bit (see
// oracle/resample_restated.py: PARITY UNPINNED); the filter meets soxr HQ's published specification — linear
// phase, pass-band to 0.913 of the lower Nyquist, stop-band from 1.0, 125 dB — as one Kaiser-windowed-sinc
// polyphase stage:    out[n] = sum_k x[k] g(n M / L - k),   L / M = 16000 / sr_in in lowest terms.
//
// Table H[j][p] (float32, [2W][L], built on the host in double): tap of input sample k_c - W + 1 + j for phase p,
// k_c = floor(n M / L), p = n M mod L.  The FIR that evaluates it for ewk_resample and ewk_push_resampled is K8
// (ewk_resample_push.cuh).
#pragma once
#include <cmath>
#include <cstdint>
#include <vector>

#include <cuda_runtime.h>

namespace ewk {

constexpr int RS_TARGET = 16000;
constexpr int RS_MAX_PHASES = 4096;

struct ResampleDesign {
    int sr_in = 0, L = 0, M = 0, W = 0;
    double fc = 0, beta = 0;
};

inline long long rs_gcd(long long a, long long b) { while (b) { const long long t = a % b; a = b; b = t; } return a; }

inline double rs_bessel_i0(double x) {                       // power series, converges for every x used here
    double s = 1.0, term = 1.0;
    const double q = x * x / 4.0;
    for (int k = 1; k < 500; k++) {
        term *= q / ((double)k * (double)k);
        s += term;
        if (term < s * 1e-17) break;
    }
    return s;
}

// false when the ratio needs more than RS_MAX_PHASES phases
inline bool rs_design(int sr_in, ResampleDesign& d) {
    const long long g = rs_gcd(sr_in, RS_TARGET);
    d.sr_in = sr_in; d.L = (int)(RS_TARGET / g); d.M = (int)(sr_in / g);
    if (d.L > RS_MAX_PHASES) return false;
    const double lower = sr_in < RS_TARGET ? sr_in : RS_TARGET;
    const double f_pass = 0.913 * lower / 2.0, f_stop = lower / 2.0, att = 125.0;
    d.beta = 0.1102 * (att - 8.7);
    const double d_omega = 2.0 * M_PI * (f_stop - f_pass) / sr_in;
    const int n_taps = (int)std::ceil((att - 8.0) / (2.285 * d_omega));
    d.W = (n_taps + 1) / 2;
    d.fc = 0.5 * (f_pass + f_stop) / sr_in;
    return true;
}

inline void rs_build_table(const ResampleDesign& d, std::vector<float>& H) {
    H.assign((size_t)2 * d.W * d.L, 0.f);
    const double i0b = rs_bessel_i0(d.beta);
    for (int j = 0; j < 2 * d.W; j++)
        for (int p = 0; p < d.L; p++) {
            const double tau = (double)p / d.L + d.W - 1 - j, u = tau / d.W;
            double v = 0.0;
            if (std::fabs(u) < 1.0) {
                const double a = 2.0 * d.fc * tau * M_PI;
                const double sinc = a == 0.0 ? 1.0 : std::sin(a) / a;
                v = 2.0 * d.fc * sinc * rs_bessel_i0(d.beta * std::sqrt(1.0 - u * u)) / i0b;
            }
            H[(size_t)j * d.L + p] = (float)v;
        }
}

}  // namespace ewk
