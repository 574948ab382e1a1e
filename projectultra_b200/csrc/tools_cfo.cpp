// projectultra_b200/csrc/tools_cfo.cpp — the CFO injector of the reference's tools (tools/test_iwaveform.cpp:67-118, also
// tools/test_hf_modem.cpp): "radio tuning error" applied to the CLEAN transmit audio before the channel (test_iwaveform.cpp:501-506) --
// analytic signal through FFT -> zero negative frequencies -> inverse FFT over the next power of two, then a rotation by the float phase
// recurrence phase += 2 pi cfo / fs (wrapped into [-pi, pi]) and the real part.  Host code: the sweep driver applies it once per TX pool
// waveform (csrc/sweep.cu), exactly where the tool applies it, so it costs nothing per trial; fresh-payload frames take the batched
// device version (tools_cfo_gpu.cu), which this function is the reference of.  Arithmetic: the reference's own radix-2 FFT
// (src/dsp/fft.cpp:76-121, the build without FFTW: float twiddles exp(-2 pi i k / N) from a float angle, butterflies in std::complex<float>,
// 1/N on the inverse) restated operation for operation; pinned bit for bit against the compiled reference FFT class in
// tests/test_tools_cfo.py (oracle/ref_build/ref_harness.cpp: ref_tools_apply_cfo).  The payload-independent tables (twiddles, rotator)
// are built by tools_cfo_twiddles / tools_cfo_rotator, which the batched device injector (tools_cfo_gpu.cu) shares.
#include <cmath>
#include <complex>
#include <vector>

#include "pu_internal.h"

namespace pu {
namespace {
using cfloat = std::complex<float>;

void fft_ref(std::vector<cfloat>& data, const std::vector<cfloat>& tw, bool inverse) {
    const size_t size = data.size();
    for (size_t i = 0, j = 0; i + 1 < size; ++i) {            // bit-reversal permutation (fft.cpp:91-97)
        if (i < j) std::swap(data[i], data[j]);
        size_t k = size / 2;
        while (k <= j) { j -= k; k /= 2; }
        j += k;
    }
    for (size_t len = 2; len <= size; len *= 2) {             // butterflies (:100-112)
        const size_t half = len / 2, step = size / len;
        for (size_t i = 0; i < size; i += len)
            for (size_t k = 0; k < half; ++k) {
                cfloat w = tw[k * step];
                if (inverse) w = std::conj(w);
                const cfloat t = w * data[i + k + half];
                data[i + k + half] = data[i + k] - t;
                data[i + k] = data[i + k] + t;
            }
    }
    if (inverse) {                                            // (:115-120)
        const float scale = 1.0f / size;
        for (auto& v : data) v *= scale;
    }
}
}  // namespace

void tools_cfo_twiddles(size_t fft_size, std::complex<float>* tw) {
    for (size_t k = 0; k < fft_size / 2; ++k) {               // fft.cpp:76-80
        const float angle = -2.0f * M_PI * k / fft_size;
        tw[k] = cfloat(std::cos(angle), std::sin(angle));
    }
}

void tools_cfo_rotator(size_t N, float cfo_hz, float sample_rate, std::complex<float>* rot) {
    float phase = 0.0f;
    const float phase_inc = 2.0f * static_cast<float>(M_PI) * cfo_hz / sample_rate;   // (:106)
    for (size_t i = 0; i < N; ++i) {
        rot[i] = cfloat(std::cos(phase), std::sin(phase));
        phase += phase_inc;
        if (phase > M_PI) phase -= 2.0f * M_PI;               // float -= double, as the tool writes it (:112-113)
        else if (phase < -M_PI) phase += 2.0f * M_PI;
    }
}

void tools_apply_cfo(float* samples, size_t N, float cfo_hz, float sample_rate) {
    if (N < 128 || std::abs(cfo_hz) < 0.001f) return;         // test_iwaveform.cpp:68
    size_t fft_size = 1;
    while (fft_size < N) fft_size *= 2;
    std::vector<cfloat> tw(fft_size / 2), rot(N);
    tools_cfo_twiddles(fft_size, tw.data());
    tools_cfo_rotator(N, cfo_hz, sample_rate, rot.data());
    std::vector<cfloat> a(fft_size, cfloat(0, 0));
    for (size_t i = 0; i < N; ++i) a[i] = cfloat(samples[i], 0);
    fft_ref(a, tw, false);
    for (size_t i = 1; i < fft_size / 2; ++i) a[i] *= 2.0f;                       // double the positive frequencies (:88-90)
    for (size_t i = fft_size / 2 + 1; i < fft_size; ++i) a[i] = cfloat(0, 0);     // zero the negative ones (:91-93)
    fft_ref(a, tw, true);
    for (size_t i = 0; i < N; ++i) samples[i] = std::real(a[i] * rot[i]);
}
}  // namespace pu

extern "C" pu_status pu_tools_apply_cfo(float* samples, size_t n, float cfo_hz, float sample_rate) {
    PU_REQUIRE(samples || n == 0, "pu_tools_apply_cfo: NULL samples");
    PU_REQUIRE(sample_rate > 0, "pu_tools_apply_cfo: bad sample rate");
    PU_REQUIRE(n <= (size_t(1) << 26), "pu_tools_apply_cfo: more than 2^26 samples");
    pu::tools_apply_cfo(samples, n, cfo_hz, sample_rate);
    return PU_OK;
}

// sizeof of the public PODs (include/pu/pu_capi.h: pu_abi_sizes): a binding that mirrors a struct by hand can check itself
extern "C" int pu_abi_sizes(uint32_t out[8]) {
    if (!out) return 0;
    const uint32_t v[8] = {sizeof(pu_modem_config), sizeof(pu_dpsk_config), sizeof(pu_mcdpsk_config), sizeof(pu_channel_config),
                           sizeof(pu_sweep_mode),   sizeof(pu_sweep_desc),  sizeof(pu_sweep_stats),   0};
    for (int i = 0; i < 8; ++i) out[i] = v[i];
    return 7;
}
