// selector.cu — host side of the channel bank: filter design, per-group stream bookkeeping, launches.
//
// Mirrors the parameter math of the reference's Decimator / Selector (csdr/chain/selector.py:21-26,
// 37-51,115-130,138-140,159-166) and the demodulator wiring of csdr/chain/analog.py:11-127.
// Filter design follows SURVEY.md Appendix A.1 (double precision, rounded once to float32).
#include "selector_kernels.cuh"
#include "fastconv.cuh"
#include "ingress.cuh"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <complex>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <map>
#include <memory>
#include <mutex>
#include <vector>

using namespace owrx;

namespace {

// ---------------------------------------------------------------- filter design (A.1)
int filter_len(double transition)
{
    int len = (int)(4.0 / transition);
    if ((len & 1) == 0) len += 1;
    return len;
}

void design_lowpass(std::vector<double>& h, int len, double fc)
{
    h.assign((size_t)len, 0.0);
    const int mid = len / 2;
    auto win = [](double r) { return 0.54 - 0.46 * cos(2.0 * M_PI * (0.5 + r / 2.0)); };
    h[mid] = 2.0 * M_PI * fc * win(0.0);
    for (int i = 1; i <= mid; i++) {
        const double v = sin(2.0 * M_PI * fc * i) / i * win((double)i / mid);
        h[mid + i] = v;
        h[mid - i] = v;
    }
    double sum = 0.0;
    for (double v : h) sum += v;
    for (double& v : h) v /= sum;
}

void design_bandpass(std::vector<float2>& out, int len, double lo, double hi)
{
    std::vector<double> h;
    design_lowpass(h, len, (hi - lo) / 2.0);
    const double centre = (hi + lo) / 2.0;
    out.resize((size_t)len);
    for (int i = 0; i < len; i++) {
        const double ph = 2.0 * M_PI * centre * i;
        out[i] = make_float2((float)(h[i] * cos(ph)), (float)(h[i] * sin(ph)));
    }
}

// in-place forward FFT, power-of-two length (host side: band-pass partition spectra)
void fft_pow2(std::vector<std::complex<double>>& a)
{
    const size_t n = a.size();
    for (size_t i = 1, j = 0; i < n; i++) {
        size_t bit = n >> 1;
        for (; j & bit; bit >>= 1) j ^= bit;
        j ^= bit;
        if (i < j) std::swap(a[i], a[j]);
    }
    // twiddles of one size are computed once (setBandpass transforms 25 partitions per call, from websocket threads)
    static std::mutex tw_mu;
    static std::map<size_t, std::vector<std::complex<double>>> tw_cache;
    const std::complex<double>* tw;
    {
        std::lock_guard<std::mutex> lk(tw_mu);
        auto& t = tw_cache[n];
        if (t.empty()) {
            t.reserve(n);
            for (size_t len = 2; len <= n; len <<= 1) {
                const double ang = -2.0 * M_PI / (double)len;
                for (size_t k = 0; k < len / 2; k++) t.emplace_back(cos(ang * (double)k), sin(ang * (double)k));
            }
        }
        tw = t.data();
    }
    for (size_t len = 2; len <= n; len <<= 1) {
        const std::complex<double>* tl = tw + (len / 2 - 1);               // stages are stored back to back: 1 + 2 + 4 + ...
        for (size_t i = 0; i < n; i += len)
            for (size_t k = 0; k < len / 2; k++) {
                const std::complex<double> w = tl[k];
                const std::complex<double> u = a[i + k], v = a[i + k + len / 2] * w;
                a[i + k] = u + v;
                a[i + k + len / 2] = u - v;
            }
    }
}

// NfmDeemphasis taps — spec-defined (upstream tables unrecoverable): frequency-sampled
// A(f) = 1 (<=400 Hz), 400/f (<=4 kHz), 0 above; Hamming window; unity gain at 400 Hz.
void design_nfm_deemphasis(std::vector<float>& out, int sample_rate)
{
    const int len = sample_rate >= 24000 ? 199 : 79, M = 8192, mid = len / 2;
    const double fs = sample_rate;
    std::vector<double> h((size_t)len);
    for (int n = 0; n < len; n++) {
        double acc = 0.0;
        for (int k = 0; k <= M / 2; k++) {
            const double f = k * fs / M;
            const double a = f <= 400.0 ? 1.0 : (f <= 4000.0 ? 400.0 / f : 0.0);
            const double c = (k == 0 || k == M / 2) ? 0.5 : 1.0;
            acc += c * a * cos(2.0 * M_PI * k * (double)(n - mid) / M);
        }
        h[n] = acc * 2.0 / M * (0.54 - 0.46 * cos(2.0 * M_PI * n / (double)(len - 1)));
    }
    double g = 0.0;
    for (int n = 0; n < len; n++) g += h[n] * cos(2.0 * M_PI * 400.0 / fs * (n - mid));
    out.resize((size_t)len);
    for (int n = 0; n < len; n++) out[n] = (float)(h[n] / g);
}

// AudioResampler(in, out) prototype — spec-defined (libsamplerate's converter is not recoverable): L/M = out/in reduced,
// Kaiser-windowed sinc at the rate L*in with a 96 dB stop band, transition 0.1*min(in, out) and cutoff 0.45*min(in, out);
// K taps per phase, N = L*K, sum h = L.  Returns false for a ratio whose N exceeds 65536.  Written to `tab` as the polyphase
// table tab[p * K + j] = h[p + j * L], rounded once to float.
bool design_audio_resampler(int in_rate, int out_rate, int* L, int* M, int* K, std::vector<float>* tab)
{
    long long a = in_rate, b = out_rate;
    while (b) { const long long t = a % b; a = b; b = t; }
    const long long l = out_rate / a, m = in_rate / a;
    const double A = 96.0, beta = 0.1102 * (A - 8.7);
    const double f_lo = std::min(in_rate, out_rate), fs = (double)l * in_rate;
    const double df = 0.1 * f_lo / fs, fc = 0.45 * f_lo / fs;
    const double k = ceil(((A - 7.95) / (14.36 * df) + 1.0) / (double)l);
    if (k * (double)l > 65536.0) return false;
    *L = (int)l; *M = (int)m; *K = (int)k;
    if (!tab) return true;
    auto i0 = [](double x) {
        double sum = 1.0, term = 1.0;
        for (int j = 1; j < 500; j++) {
            term *= (x / (2.0 * j)) * (x / (2.0 * j));
            sum += term;
            if (term < 1e-17 * sum) break;
        }
        return sum;
    };
    const int n = *L * *K;
    const double i0b = i0(beta), c = (n - 1) / 2.0;
    std::vector<double> h((size_t)n);
    double sum = 0.0;
    for (int i = 0; i < n; i++) {
        const double t = 2.0 * fc * (i - c);
        const double sinc = t == 0.0 ? 1.0 : sin(M_PI * t) / (M_PI * t);
        const double r = n > 1 ? 2.0 * i / (n - 1) - 1.0 : 0.0;
        h[(size_t)i] = 2.0 * fc * sinc * i0(beta * sqrt(std::max(0.0, 1.0 - r * r))) / i0b;
        sum += h[(size_t)i];
    }
    tab->resize((size_t)n);
    for (int p = 0; p < *L; p++)
        for (int j = 0; j < *K; j++) (*tab)[(size_t)p * *K + j] = (float)(h[(size_t)p + (size_t)j * *L] * (double)l / sum);
    return true;
}

// ---------------------------------------------------------------- stage buffer with history
// rows of `slots * width` floats; rows [0, fill) hold absolute indices [abs_end - fill, abs_end).
struct StageBuf {
    float* d[2] = {nullptr, nullptr};
    // recorded by the split-phase drain (owrx_bank_drain_begin, through drain_enqueue) after the transpose that read buffer b;
    // the next writer of that buffer waits for it.  Created on first use; an event that was never recorded does not block.
    cudaEvent_t drained[2] = {nullptr, nullptr};
    int cur = 0, width = 1, slots = 0;
    size_t hist = 0, cap_rows = 0, fill = 0;
    long long abs_end = 0;

    size_t row_floats() const { return (size_t)slots * width; }
    float* rows(size_t r = 0) const { return d[cur] + r * row_floats(); }
    float* row_abs(long long a) const { return d[cur] + (size_t)(a - (abs_end - (long long)fill)) * row_floats(); }
    float* append_ptr() const { return rows(fill); }

    int init(int width_, int slots_, size_t hist_, size_t cap_new)
    {
        release();
        width = width_; slots = slots_; hist = hist_; cap_rows = hist_ + cap_new;
        for (int b = 0; b < 2; b++) {
            OWRX_CUDA(cudaMalloc((void**)&d[b], cap_rows * row_floats() * sizeof(float)));
            OWRX_CUDA(cudaMemset(d[b], 0, cap_rows * row_floats() * sizeof(float)));
        }
        cur = 0; fill = hist; abs_end = 0;     // `hist` zero rows precede the stream start
        return OWRX_OK;
    }
    int ensure_new(size_t n_new, cudaStream_t st)
    {
        if (fill + n_new <= cap_rows) return OWRX_OK;
        const size_t ncap = std::max(fill + n_new, cap_rows * 2);
        for (int b = 0; b < 2; b++) {
            float* nb = nullptr;
            OWRX_CUDA(cudaMalloc((void**)&nb, ncap * row_floats() * sizeof(float)));
            OWRX_CUDA(cudaMemsetAsync(nb, 0, ncap * row_floats() * sizeof(float), st));
            if (b == cur && fill) OWRX_CUDA(cudaMemcpyAsync(nb, d[b], fill * row_floats() * sizeof(float), cudaMemcpyDeviceToDevice, st));
            OWRX_CUDA(cudaStreamSynchronize(st));
            cudaFree(d[b]);
            d[b] = nb;
        }
        cap_rows = ncap;
        return OWRX_OK;
    }
    void appended(size_t n) { fill += n; abs_end += (long long)n; }
    // keep the newest `keep` rows (<= fill) at the front of the other buffer
    int roll(size_t keep, cudaStream_t st)
    {
        keep = std::min(keep, fill);
        if (keep == fill) return OWRX_OK;
        if (keep) OWRX_CUDA(cudaMemcpyAsync(d[cur ^ 1], rows(fill - keep), keep * row_floats() * sizeof(float), cudaMemcpyDeviceToDevice, st));
        cur ^= 1;
        fill = keep;
        return OWRX_OK;
    }
    void release()
    {
        for (int b = 0; b < 2; b++) { if (d[b]) cudaFree(d[b]); d[b] = nullptr; }
        for (int b = 0; b < 2; b++) { if (drained[b]) cudaEventDestroy(drained[b]); drained[b] = nullptr; }
        cap_rows = fill = 0;
    }
    // the current buffer has been read by work enqueued on `st` so far
    int mark_drained(cudaStream_t st)
    {
        if (!drained[cur]) OWRX_CUDA(cudaEventCreateWithFlags(&drained[cur], cudaEventDisableTiming));
        OWRX_CUDA(cudaEventRecord(drained[cur], st));
        return OWRX_OK;
    }
    // `st` is about to write the current buffer
    int wait_drained(cudaStream_t st) const
    {
        if (drained[cur]) OWRX_CUDA(cudaStreamWaitEvent(st, drained[cur], 0));
        return OWRX_OK;
    }
};

// flat FIFO of floats: one bulk append per feed, bulk pop
struct FQ {
    std::vector<float> v;
    size_t off = 0;
    size_t size() const { return v.size() - off; }
    void push(const float* p, size_t n)
    {
        if (off && off >= v.size() / 2) { v.erase(v.begin(), v.begin() + (ptrdiff_t)off); off = 0; }
        v.insert(v.end(), p, p + n);
    }
    void push_back(float x) { v.push_back(x); }
    size_t pop(float* out, size_t max_floats, size_t unit)
    {
        size_t take = std::min(max_floats, size());
        take -= take % unit;
        std::copy(v.begin() + (ptrdiff_t)off, v.begin() + (ptrdiff_t)(off + take), out);
        off += take;
        if (off == v.size()) { v.clear(); off = 0; }
        return take;
    }
};

struct Chan {
    int id = -1;
    int group = -1, slot = -1;
    double rate = 0.0, phase = 0.0;        // phase (turns) just before the next unconsumed sample
    bool bp_enabled = false;
    double bp_lo = 0.0, bp_hi = 0.0;
    bool bp_dirty = false;                 // a designed band-pass waits in bp_stage for the next block boundary
    std::vector<float2> bp_stage;          // Tb taps followed by the bpP x 256 partition spectra
    ChanCfg cfg{};
    owrx_chan_spec_t spec{};
    float agc_initial = 1.0f;
    int audio_fmt = OWRX_AUDIO_F32;
    int mpx_fmt = OWRX_MPX_OFF;
    int atap_fmt = OWRX_MPX_OFF;           // owrx_chan_set_audio_tap
    int rs_in = 0, rs_out = 0;             // owrx_chan_set_audio_resampler: 0 = none
    bool rs_dirty = false;                 // the resampler (re)starts at the next block boundary (apply_pending)
    unsigned long long gen = 0;            // bank-unique: tells this client from a later one that gets the same id
    FQ q_audio, q_demod, q_if, q_power;
    std::vector<unsigned char> q_bytes, q_mpx, q_atap;
    size_t last_audio = 0;
};

// one tapped channel of a block (owrx_chan_set_mpx / _audio_tap): where its run sits in the staging region and whom it belongs to
struct TapRun {
    int chan, fmt, run;
    unsigned long long gen;
};

// A per-channel tap gathered by tap_gather_kernel: the tapped slots of the block being issued (rebuilt at every block
// boundary) and a staging region per block parity of `cap` rows per run; the split-phase drain's copy of a region is awaited
// through `drained` before the region is written again
struct TapStage {
    std::vector<TapRun> runs;
    int nf = 0, ns = 0;
    unsigned char* d[2] = {nullptr, nullptr};
    size_t cap = 0, bytes = 0;
    size_t rows = 0;                                 // rows gathered in this feed
    cudaEvent_t drained[2] = {nullptr, nullptr};

    // the block's layout: F32 runs, then S16 runs, in slot order; returns the slot's run
    void clear() { runs.clear(); nf = ns = 0; }
    int add(int chan, int fmt, unsigned long long gen)
    {
        const int run = fmt == OWRX_MPX_F32 ? nf++ : (fmt == OWRX_MPX_S16 ? ns++ : 0);
        if (fmt != OWRX_MPX_OFF) runs.push_back(TapRun{chan, fmt, run, gen});
        return run;
    }
    // start of a feed: room for `low` new rows per run (the layout is this block's)
    int provision(size_t low)
    {
        rows = 0;
        if (runs.empty()) return OWRX_OK;
        const size_t c = std::max(cap, (low + 7) / 8 * 8);
        const size_t b = c * (4 * (size_t)nf + 2 * (size_t)ns);
        if (c != cap || b > bytes) {
            OWRX_CUDA(cudaDeviceSynchronize());
            for (int k = 0; k < 2; k++) { cudaFree(d[k]); d[k] = nullptr; }
            cap = bytes = 0;
            for (int k = 0; k < 2; k++) OWRX_CUDA(cudaMalloc((void**)&d[k], b));
            cap = c; bytes = b;
        }
        return OWRX_OK;
    }
    // new rows [in, in + n) of every tapped slot -> staging region `cur`, on `st`
    template <typename Sel>
    int gather(owrx_bank_stats_t& stats, const float* in, int slots, size_t n, Sel sel, int cur, cudaStream_t st)
    {
        if (rows + n > cap) return fail(OWRX_E_STATE, "tap staging under-provisioned");
        if (drained[cur]) OWRX_CUDA(cudaStreamWaitEvent(st, drained[cur], 0));
        const long long r0 = (long long)rows;
        const long long tiles = (r0 + (long long)n + MG_R - 1) / MG_R - r0 / MG_R;
        tap_gather_kernel<<<dim3((unsigned)(slots / 32), (unsigned)std::min<long long>(tiles, 65535)), 256, 0, st>>>(
            in, slots, (int)n, sel, r0, (long long)cap, nf, d[cur]);
        OWRX_LAUNCH_CHECK();
        stats.kernel_launches++;
        rows += n;
        return OWRX_OK;
    }
    // the split-phase drain's copy of region `cur` has been enqueued on `st`
    int mark_drained(int cur, cudaStream_t st)
    {
        if (!drained[cur]) OWRX_CUDA(cudaEventCreateWithFlags(&drained[cur], cudaEventDisableTiming));
        OWRX_CUDA(cudaEventRecord(drained[cur], st));
        return OWRX_OK;
    }
    void release()
    {
        for (int k = 0; k < 2; k++) {
            cudaFree(d[k]); d[k] = nullptr;
            if (drained[k]) cudaEventDestroy(drained[k]);
            drained[k] = nullptr;
        }
        cap = bytes = 0;
    }
};

struct Group {
    owrx_chan_spec_t spec{};
    bool wfm = false;
    int D = 1, T = 1, nseg = 1, nrs = 1, RB = 1;
    double frac = 1.0;
    bool has_frac = false;
    int Tb = 1, sq_len = 1, Td = 1, Tpre = 0;
    double wfm_rate = 1.0;
    float alpha = 0.f;
    int slots = 0;                                   // capacity, multiple of K3_CG
    std::vector<int> slot_chan;
    // device tables
    float* d_taps = nullptr; float* d_deemph = nullptr; float* d_pre = nullptr;
    double* d_rate = nullptr; double* d_phase = nullptr; float2* d_w = nullptr;
    float2* d_bp = nullptr;
    int* d_bp_en2[2] = {nullptr, nullptr};           // per-slot tables are double-buffered by block parity (see group_begin_feed)
    int* d_bp_en = nullptr;                          // = d_bp_en2[cur]
    // K4F partitioned-FFT band-pass (fastconv.cuh): H[p][256][slots], scratch spectra
    int bpP = 1;
    float2* d_bp_H = nullptr; float2* d_bp_X = nullptr; float2* d_bp_Y = nullptr;
    size_t bp_blocks_cap = 0;
    ChanCfg* d_cfg2[2] = {nullptr, nullptr};
    ChanCfg* d_cfg = nullptr;                        // = d_cfg2[cur]
    ChanState* d_state = nullptr;
    TailStash* d_stash = nullptr;                    // fused tail: state the next feed starts from (tail_front -> tail_commit)
    std::vector<double> h_rate, h_phase; std::vector<float2> h_w;
    std::vector<int> h_bp_en; std::vector<ChanCfg> h_cfg;
    bool cfg_stale[2] = {true, true};                // host tables changed since that copy was uploaded
    int cur = 0;                                     // parity of the block being issued
    std::map<int, SlotPatch> pend;                   // per-slot state patches waiting for the next block boundary
    bool bp_pending = false;                         // some channel has a staged band-pass
    SlotPatch* d_patch[2] = {nullptr, nullptr}; int patch_cap = 0;     // device staging: [0] tail stream, [1] serial stream
    float2* d_bp_stage = nullptr; int* d_bp_stage_slots = nullptr; int bp_stage_cap = 0;
    // page-locked host staging of the designed band-passes, one per block parity: a pageable source of this size (76 KB per
    // 3125-tap design) would make cudaMemcpyAsync wait for the stream; the event says the copy that last read it has run
    unsigned char* h_bp_pin[2] = {nullptr, nullptr}; size_t h_bp_pin_cap[2] = {0, 0};
    cudaEvent_t bp_pin_ev[2] = {nullptr, nullptr};
    // stream position
    size_t in_off = 0;                               // streaming: offset of the next block in the bank's IQ buffer
    size_t dev_lead = 0;                             // device path: samples at the head of the next block this group has consumed already
    long long frac_m = 0, wfm_m = 0, sq_abs = 0;
    StageBuf s1, s2, s3, f1, f1p, f1b, f2, f3;
    float2* d_partial = nullptr; size_t partial_cap = 0;
    unsigned char* d_gate = nullptr; float* d_power = nullptr; float* d_dcmean = nullptr; float* d_dcprev = nullptr;
    size_t blocks_cap = 0;
    long long sq_block_abs = 0;                      // squelch blocks processed so far (S-meter report interval)
    long long sq_block_first = 0;                    // sq_block_abs at the start of this feed
    // last run
    size_t last_audio = 0, last_demod = 0, last_if = 0, last_blocks = 0;
    size_t dr_audio = 0, dr_demod = 0, dr_if = 0, dr_blocks = 0;    // of those, already copied to the host queues
    bool dr_final = false;                           // the feed's client-audio bytes and multiplex tap are in the queues
    size_t pass_audio = 0;                           // audio rows produced by the last tail pass
    size_t feed_blocks = 0;                          // squelch blocks processed so far in this feed
    size_t pend_rows = 0;                            // FirDecimate rows appended to s1 since the last tail pass
    long long pend_first = 0;
    // client audio tail (Convert / AdpcmEncoder), and the resampler in front of it
    std::vector<int> h_tail_mode;
    std::vector<RsCfg> h_rs;
    RsCfg* d_rs_cfg2[2] = {nullptr, nullptr};
    RsCfg* d_rs_cfg = nullptr;                       // = d_rs_cfg2[cur]
    int* d_tail_mode2[2] = {nullptr, nullptr};
    int* d_tail_mode = nullptr;                      // = d_tail_mode2[cur]
    TailState* d_tail = nullptr; int* d_tail_count = nullptr;
    int16_t* d_tail_s16 = nullptr; unsigned char* d_tail_bytes = nullptr;
    size_t tail_rows_cap = 0; int tail_cap = 0;
    bool any_tail = false, tail_ran = false;
    // client-audio resampler (audio_resample_kernel): some slot has one (per-slot state in ChanCfg::rs_*), the largest L/M of
    // them, its outputs of this feed (rows of d_rs and of the int16 scratch), and the feed's first absolute audio row.  f3 keeps
    // the K - 1 rows the resampler looks back over its passes (f3.hist).
    bool any_rs = false, rs_pending = false;
    double rs_up = 1.0;
    float* d_rs = nullptr;
    size_t rs_rows = 0;
    long long audio_af = 0;
    // K3F fast-convolution channeliser (fastconv.cuh): tables are built lazily on the first eligible pass
    bool fc_ok = false;
    FcShape fc{};
    float* d_fc_h = nullptr; float2* d_fc_tab = nullptr; float4* d_fc_F = nullptr; float2* d_fc_Z = nullptr;
    float fc_tab_scale = 1.0f;                                 // fp16 x 2 operand form: the table's power of two
    float* d_fc_scale = nullptr;                               // [0] spectra scale of the pass, [1] output scale, [2] running max (bits)
    int* d_fc_slots = nullptr; double* d_fc_rates = nullptr;
    size_t fc_blocks_cap = 0;
    std::vector<double> fc_tab_rate;                 // per slot: Shift rate its table column was built for (NaN = none)
    // tensor-core form (fastconv_tc.cu): bf16 operand planes of the table and of the branch spectra
    void* d_fc_tabp = nullptr; void* d_fc_Fp = nullptr; size_t fc_blocks_cap_tc = 0;
    std::vector<double> fc_tabp_rate;
    std::vector<float> fc_taps;                      // h[t] rounded to float (same values K3 uses)
    // taps (tap_gather_kernel): the WFM multiplex tap of f1 (ChanCfg::mpx / mpx_run), and the demodulated-audio tap of f3,
    // whose (format, run) per slot is a per-parity table of its own
    TapStage mpx, atap;
    std::vector<TapFmt> h_atap;
    TapFmt* d_atap2[2] = {nullptr, nullptr};
    TapFmt* d_atap = nullptr;                        // = d_atap2[cur]
};

// ---------------------------------------------------------------- output drain
// Every path that moves outputs to the host queues (the host feed per chunk and at its end, deferred drain, owrx_bank_drain,
// owrx_bank_drain_begin / _end) takes the same three steps: drain_items lists what is to move, one item per (group, output);
// drain_enqueue stages the list on a stream; drain_deliver pushes the staged bytes into the queues once the copies have landed.
enum DrainKind { DRAIN_AUDIO, DRAIN_DEMOD, DRAIN_IF, DRAIN_POWER, DRAIN_BYTES, DRAIN_MPX, DRAIN_ATAP };

// the client a slot (DRAIN_MPX / _ATAP: a run) belongs to when the drain is listed; delivery skips it once that client has left
struct DrainTo {
    int chan;
    unsigned long long gen;
    int fmt;                     // DRAIN_BYTES: the client-audio format; DRAIN_MPX / _ATAP: the tap format
    size_t n;                    // DRAIN_BYTES: S16 samples of the slot; DRAIN_MPX / _ATAP: the run's first byte in the item
};

struct DrainItem {
    DrainKind kind;
    Group* g = nullptr;          // read by drain_enqueue only (the client-audio scratch, the parity of the tap regions)
    TapStage* tap = nullptr;     // MPX / ATAP: the staging the runs are copied from (drain_enqueue only)
    const float* src = nullptr;  // AUDIO / DEMOD / IF: the first row to move; POWER: the first block
    StageBuf* buf = nullptr;     // AUDIO / DEMOD / IF: the buffer src lies in
    size_t n = 0;                // rows of `slots` elements of `width` floats (POWER: blocks; BYTES: int16 rows; taps: rows per run)
    int slots = 0, width = 1;
    size_t cap = 0;              // BYTES: ADPCM bytes per slot; taps: rows per run of the gather region
    long long phase = 0;         // POWER: absolute squelch block of block 0
    size_t bytes = 0, off = 0;   // size and offset in the staging (drain_enqueue)
    std::vector<DrainTo> to;     // per slot (taps: per run)
    bool transposed() const { return kind == DRAIN_AUDIO || kind == DRAIN_DEMOD || kind == DRAIN_IF; }
};

// page-locked host staging and device transpose scratch of a drain; grows while no drain is in flight on it
struct DrainStage {
    unsigned char* h = nullptr;
    unsigned char* d = nullptr;
    size_t h_cap = 0, d_cap = 0;

    int reserve(size_t h_bytes, size_t d_bytes)
    {
        if (h_bytes > h_cap) {
            if (h) cudaFreeHost(h);
            h = nullptr; h_cap = 0;
            OWRX_CUDA(cudaMallocHost((void**)&h, h_bytes));
            h_cap = h_bytes;
        }
        if (d_bytes > d_cap) {
            cudaFree(d); d = nullptr; d_cap = 0;
            OWRX_CUDA(cudaMalloc((void**)&d, d_bytes));
            d_cap = d_bytes;
        }
        return OWRX_OK;
    }
    void release()
    {
        if (h) cudaFreeHost(h);
        cudaFree(d);
        h = nullptr; d = nullptr; h_cap = d_cap = 0;
    }
};

}  // namespace

struct owrx_bank {
    int device = 0, sm_count = 0;
    double input_rate = 0.0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::mutex mu;
    std::vector<std::unique_ptr<Chan>> chans;
    unsigned long long chan_gen = 0;                 // Chan::gen of the latest client
    std::vector<std::unique_ptr<Group>> groups;
    int out_mask = OWRX_OUT_AUDIO;
    // streaming wideband buffer
    float2* d_iq[2] = {nullptr, nullptr};
    int iq_cur = 0;
    size_t iq_cap = 0, iq_fill = 0;
    // staging of the synchronous drains, and of the split-phase drain (owrx_bank_drain_begin / _end): a synchronous drain
    // between _begin and _end must not clobber the copies in flight; adrain_items is the list they deliver
    DrainStage stage, adrain_stage;
    std::vector<DrainItem> adrain_items;
    bool adrain_pending = false;
    cudaEvent_t adrain_done = nullptr;                         // the D2H copies have landed
    owrx_bank_stats_t stats{};
    // H2D copy stream for the chunked host path; side stream + events for the pipelined device path
    cudaStream_t copy_stream = nullptr, side_stream = nullptr, serial_stream = nullptr;
    std::vector<cudaEvent_t> chunk_events;
    cudaEvent_t fir_done = nullptr, ptail_done[2] = {nullptr, nullptr}, tail_done[2] = {nullptr, nullptr}, dev_done = nullptr;
    bool pipelined = false, reserve_sm = false;
    std::vector<cudaEvent_t> fir_events, drain_events;
    cudaStream_t drain_stream = nullptr;
    unsigned long long calls = 0;
    // optional per-kernel timing of K3 (CUDA events on the launching stream)
    bool profile = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;
    std::vector<int> prof_tags;
    size_t prof_used = 0;
    std::vector<size_t> prof_open;                   // brackets begun and not ended yet, innermost last (a tap gather inside the tail's)
    double prof_ms[OWRX_PROF_KINDS] = {};
    uint64_t prof_launches[OWRX_PROF_KINDS] = {};
    int fir_mode = OWRX_FIR_AUTO, bp_mode = OWRX_FIR_AUTO;
    unsigned char* d_raw = nullptr; size_t raw_cap = 0;   // staging for raw (non-float) ingress chunks (owrx_bank_feed_fmt)
    // deferred drain (owrx_bank_set_deferred_drain): a feed returns once its work is enqueued; its last outputs reach the
    // host queues at the start of the next feed — after that feed's uploads are under way — or in owrx_bank_flush
    bool deferred = false, pending_final = false;
    int fir_form_used = 0;                           // form of the latest Shift + FirDecimate pass (owrx_bank_fir_form)
    // forms the parity tests force at shapes where the cost models would not pick them (read from the environment at creation,
    // like fir_mode)
    bool tail_fused = true;                          // OWRX_TAIL_FUSED=0: the seven-kernel low-rate tail
    int fc_m = 0;                                    // OWRX_FC_M = 64 | 256: branch FFT size of new groups (fc_pick_fft_size)
    int fc_levels = 0;                               // OWRX_FC_TC_FMT = f16x2 | bf16x3: operand split of new groups (fc_pick_tc_levels)
    int fc_tc_form = -1;                             // OWRX_FC_TC_FORM = 0 | 1: blocks | slots in the MMA's M (fc_launch_contract_tc)
    size_t last_consumed = 0;                        // device path: samples of the last block every group is done with
    // groups whose last client left: out of the feed loops at once, their device memory released by a later call once the
    // event (recorded behind everything issued while the group was live) has completed — no device synchronisation
    std::vector<std::pair<std::unique_ptr<Group>, cudaEvent_t>> graveyard;
    cudaStream_t ctl_stream = nullptr;
    unsigned long long feeds = 0;                    // host-path feeds so far (parity of the per-slot table copies)
    // client-audio resampler polyphase tables, one per (L, M) for the bank's lifetime (RsCfg::tab points into them)
    struct RsTab { float* d; int K; };
    std::map<std::pair<int, int>, RsTab> rs_tabs;
};

namespace {

template <typename T> int dev_alloc(T** p, size_t n)
{
    *p = nullptr;
    OWRX_CUDA(cudaMalloc((void**)p, std::max<size_t>(n, 1) * sizeof(T)));
    OWRX_CUDA(cudaMemset(*p, 0, std::max<size_t>(n, 1) * sizeof(T)));
    return OWRX_OK;
}

void group_release(Group* g)
{
    cudaFree(g->d_taps); cudaFree(g->d_deemph); cudaFree(g->d_pre);
    cudaFree(g->d_rate); cudaFree(g->d_phase); cudaFree(g->d_w);
    cudaFree(g->d_bp); cudaFree(g->d_bp_en2[0]); cudaFree(g->d_bp_en2[1]); cudaFree(g->d_cfg2[0]); cudaFree(g->d_cfg2[1]);
    cudaFree(g->d_state); cudaFree(g->d_stash); cudaFree(g->d_patch[0]); cudaFree(g->d_patch[1]);
    cudaFree(g->d_bp_stage); cudaFree(g->d_bp_stage_slots);
    for (int k = 0; k < 2; k++) {
        if (g->h_bp_pin[k]) cudaFreeHost(g->h_bp_pin[k]);
        if (g->bp_pin_ev[k]) cudaEventDestroy(g->bp_pin_ev[k]);
    }
    cudaFree(g->d_bp_H); cudaFree(g->d_bp_X); cudaFree(g->d_bp_Y);
    cudaFree(g->d_partial); cudaFree(g->d_gate); cudaFree(g->d_power); cudaFree(g->d_dcmean); cudaFree(g->d_dcprev);
    cudaFree(g->d_tail_mode2[0]); cudaFree(g->d_tail_mode2[1]); cudaFree(g->d_rs_cfg2[0]); cudaFree(g->d_rs_cfg2[1]); cudaFree(g->d_tail); cudaFree(g->d_tail_count); cudaFree(g->d_tail_s16);
    cudaFree(g->d_tail_bytes); cudaFree(g->d_rs);
    cudaFree(g->d_fc_h); cudaFree(g->d_fc_tab); cudaFree(g->d_fc_F); cudaFree(g->d_fc_Z); cudaFree(g->d_fc_slots); cudaFree(g->d_fc_rates);
    cudaFree(g->d_fc_scale);
    cudaFree(g->d_fc_tabp); cudaFree(g->d_fc_Fp);
    g->mpx.release(); g->atap.release();
    cudaFree(g->d_atap2[0]); cudaFree(g->d_atap2[1]);
    g->s1.release(); g->s2.release(); g->s3.release(); g->f1.release(); g->f1p.release(); g->f1b.release(); g->f2.release(); g->f3.release();
}

// Selector / Decimator parameter math (csdr/chain/selector.py:21-26,37-51,115-126): the spec a plain
// Selector(inputRate, outputRate) hands to pycsdr.
owrx_chan_spec_t spec_from_rates(double input_rate, double output_rate)
{
    owrx_chan_spec_t sp{};
    double orate = output_rate > input_rate ? input_rate : output_rate;
    const double d = input_rate / orate;
    sp.decimation = (int)d;
    sp.fraction = (input_rate / sp.decimation) / orate;
    sp.transition = 0.15 * (orate / input_rate);
    sp.cutoff = 0.5 * sp.decimation / (input_rate / orate);
    sp.bp_transition = 320.0 / orate;                                  // Selector._buildBandpass, selector.py:115-117
    sp.squelch_length = std::max(1, (int)(orate / 16));                // Selector._buildSquelch, selector.py:119-121
    sp.deemph_rate = (int)orate;                                       // NfmDeemphasis(sampleRate), analog.py:43
    return sp;
}

bool spec_equal(const owrx_chan_spec_t& a, const owrx_chan_spec_t& b)
{
    return a.decimation == b.decimation && a.transition == b.transition && a.cutoff == b.cutoff && a.fraction == b.fraction &&
           a.bp_transition == b.bp_transition && a.squelch_length == b.squelch_length && a.deemph_rate == b.deemph_rate &&
           a.wfm == b.wfm && (!a.wfm || (a.wfm_decimation == b.wfm_decimation && a.wfm_audio_rate == b.wfm_audio_rate && a.wfm_tau == b.wfm_tau));
}

int spec_validate(const owrx_chan_spec_t& sp)
{
    if (sp.decimation < 1) return fail(OWRX_E_INVALID, "decimation must be >= 1");
    if (!(sp.transition > 0.0 && sp.transition <= 4.0)) return fail(OWRX_E_INVALID, "bad FirDecimate transition %g", sp.transition);
    if (!(sp.cutoff > 0.0)) return fail(OWRX_E_INVALID, "bad FirDecimate cutoff %g", sp.cutoff);
    if (!(sp.fraction >= 1.0)) return fail(OWRX_E_INVALID, "fraction must be >= 1");
    if (!(sp.bp_transition > 0.0 && sp.bp_transition < 2.0)) return fail(OWRX_E_INVALID, "bad Bandpass transition %g", sp.bp_transition);
    if (sp.squelch_length < 1) return fail(OWRX_E_INVALID, "bad Squelch length");
    if (sp.deemph_rate < 1) return fail(OWRX_E_INVALID, "bad de-emphasis rate");
    if (sp.wfm && !(sp.wfm_decimation > 1.03 && sp.wfm_audio_rate > 0 && sp.wfm_tau > 0.0)) return fail(OWRX_E_INVALID, "bad WFM parameters");
    return OWRX_OK;
}

int group_create(owrx_bank* bank, const owrx_chan_spec_t& sp, int* index)
{
    int vrc = spec_validate(sp);
    if (vrc != OWRX_OK) return vrc;
    std::unique_ptr<Group> g(new Group());
    g->spec = sp;
    const bool wfm = sp.wfm != 0;
    g->wfm = wfm;
    g->D = sp.decimation;
    g->frac = sp.fraction;
    g->has_frac = g->frac != 1.0;
    const double cutoff = sp.cutoff;
    g->T = filter_len(sp.transition);
    const int P = (g->T + g->D - 1) / g->D;
    g->nseg = (P + K3_PP - 1) / K3_PP;
    g->nrs = (g->D + K3_RBMAX - 1) / K3_RBMAX;
    g->RB = (g->D + g->nrs - 1) / g->nrs;
    g->Tb = filter_len(sp.bp_transition);
    g->bpP = (g->Tb + BPF_H - 1) / BPF_H;
    g->sq_len = sp.squelch_length;
    g->slots = K3_CG;
    g->slot_chan.assign((size_t)g->slots, -1);

    // FirDecimate taps in polyphase layout [nseg][D][28]
    std::vector<double> h;
    design_lowpass(h, g->T, cutoff / g->D);
    std::vector<float> ht((size_t)g->nseg * g->D * K3_PP, 0.f);
    for (int t = 0; t < g->T; t++) {
        const int p = t / g->D, r = t % g->D;
        ht[((size_t)(p / K3_PP) * g->D + r) * K3_PP + (p % K3_PP)] = (float)h[t];
    }
    g->fc_taps.resize((size_t)g->T);
    for (int t = 0; t < g->T; t++) g->fc_taps[(size_t)t] = (float)h[t];
    const int fcM = fc_pick_fft_size(g->D, P, bank->fc_m);
    g->fc = FcShape{g->D, g->T, P, fcM - P + 1, (g->D + FC_DPAD - 1) / FC_DPAD * FC_DPAD, g->slots, fcM, fc_pick_tc_levels(g->D, bank->fc_levels)};
    g->fc_tab_scale = fc_tab_scale(g->fc, g->fc_taps.data());
    g->fc_ok = g->D >= 8 && P <= fcM / 2;
    int rc;
    if ((rc = dev_alloc(&g->d_taps, ht.size())) != OWRX_OK) return rc;
    OWRX_CUDA(cudaMemcpy(g->d_taps, ht.data(), ht.size() * sizeof(float), cudaMemcpyHostToDevice));

    std::vector<float> de;
    design_nfm_deemphasis(de, sp.deemph_rate);                           // NfmDeemphasis(sampleRate), analog.py:43
    g->Td = (int)de.size();
    if ((rc = dev_alloc(&g->d_deemph, de.size())) != OWRX_OK) return rc;
    OWRX_CUDA(cudaMemcpy(g->d_deemph, de.data(), de.size() * sizeof(float), cudaMemcpyHostToDevice));
    if (wfm) {
        g->wfm_rate = sp.wfm_decimation;                                 // analog.py:66: 250000.0 / sampleRate
        g->Tpre = filter_len(0.03);
        std::vector<double> pre;
        design_lowpass(pre, g->Tpre, 0.5 / (g->wfm_rate - 0.03));
        std::vector<float> pf(pre.begin(), pre.end());
        if ((rc = dev_alloc(&g->d_pre, pf.size())) != OWRX_OK) return rc;
        OWRX_CUDA(cudaMemcpy(g->d_pre, pf.data(), pf.size() * sizeof(float), cudaMemcpyHostToDevice));
        const double dt = 1.0 / (double)sp.wfm_audio_rate;
        g->alpha = (float)(dt / (sp.wfm_tau + dt));                      // WfmDeemphasis, SURVEY A.11
    }
    const size_t S = (size_t)g->slots;
    if ((rc = dev_alloc(&g->d_rate, S)) || (rc = dev_alloc(&g->d_phase, S)) || (rc = dev_alloc(&g->d_w, S)) ||
        (rc = dev_alloc(&g->d_bp, S * g->Tb)) || (rc = dev_alloc(&g->d_bp_H, S * (size_t)g->bpP * FC_M)) ||
        (rc = dev_alloc(&g->d_bp_en2[0], S)) || (rc = dev_alloc(&g->d_bp_en2[1], S)) || (rc = dev_alloc(&g->d_cfg2[0], S)) ||
        (rc = dev_alloc(&g->d_cfg2[1], S)) || (rc = dev_alloc(&g->d_state, S)) || (rc = dev_alloc(&g->d_tail_mode2[0], S)) ||
        (rc = dev_alloc(&g->d_tail_mode2[1], S)) || (rc = dev_alloc(&g->d_tail, S)) || (rc = dev_alloc(&g->d_tail_count, S)) ||
        (rc = dev_alloc(&g->d_rs_cfg2[0], S)) || (rc = dev_alloc(&g->d_rs_cfg2[1], S)) ||
        (rc = dev_alloc(&g->d_atap2[0], S)) || (rc = dev_alloc(&g->d_atap2[1], S)) || (rc = dev_alloc(&g->d_stash, S)))
        return rc;
    g->d_cfg = g->d_cfg2[0]; g->d_bp_en = g->d_bp_en2[0]; g->d_tail_mode = g->d_tail_mode2[0]; g->d_rs_cfg = g->d_rs_cfg2[0];
    g->d_atap = g->d_atap2[0];
    g->h_tail_mode.assign(S, 0);
    g->h_rs.assign(S, RsCfg{});
    g->h_atap.assign(S, TapFmt{OWRX_MPX_OFF, 0});
    g->h_rate.assign(S, 0.0); g->h_phase.assign(S, 0.0); g->h_w.assign(S, make_float2(1.f, 0.f));
    g->h_bp_en.assign(S, 0);
    ChanCfg idle{}; idle.kind = OWRX_DEMOD_NONE; idle.agc_ref = 0.8f; idle.agc_max = 1.f; idle.agc_thr = 0.8f;
    g->h_cfg.assign(S, idle);

    const size_t cap = 4096;
    // band-pass input history: Tb-1 taps back, plus the register-blocked kernel's window overshoot (2*BP_RB + padding of T)
    // band-pass input history: Tb-1 taps back plus the register-blocked kernel's window overshoot, or the P+1 hops of the
    // partitioned-FFT form
    const size_t bp_hist = std::max<size_t>((size_t)(g->Tb + 3 * BP_RB), (size_t)BPF_H * (size_t)(g->bpP + 1));
    if ((rc = g->s1.init(2, g->slots, bp_hist, cap)) != OWRX_OK) return rc;
    if (g->has_frac && (rc = g->s2.init(2, g->slots, bp_hist, cap)) != OWRX_OK) return rc;
    if ((rc = g->s3.init(2, g->slots, (size_t)g->sq_len, cap)) != OWRX_OK) return rc;
    if ((rc = g->f1.init(1, g->slots, 256, cap)) != OWRX_OK) return rc;
    if (wfm && (rc = g->f1p.init(1, g->slots, 32, cap)) != OWRX_OK) return rc;
    if (wfm && (rc = g->f1b.init(1, g->slots, 0, cap)) != OWRX_OK) return rc;
    if ((rc = g->f2.init(1, g->slots, 0, cap)) != OWRX_OK) return rc;
    if ((rc = g->f3.init(1, g->slots, 0, cap)) != OWRX_OK) return rc;
    g->in_off = bank->iq_fill;          // a new group starts with the next incoming sample
    for (size_t i = 0; i < bank->groups.size(); i++) {
        if (!bank->groups[i]) { *index = (int)i; bank->groups[i] = std::move(g); return OWRX_OK; }
    }
    *index = (int)bank->groups.size();
    bank->groups.push_back(std::move(g));
    return OWRX_OK;
}

// A group nobody listens to any more leaves the feed loops now; its buffers are freed by reap_groups once everything
// that was issued while it was live has run (event behind the bank's own streams and the caller's last block).
int retire_group(owrx_bank* bank, int gi)
{
    std::unique_ptr<Group> g = std::move(bank->groups[(size_t)gi]);
    bank->groups[(size_t)gi].reset();
    cudaEvent_t ev = nullptr;
    OWRX_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    for (cudaStream_t s : {bank->stream, bank->side_stream, bank->serial_stream, bank->copy_stream, bank->drain_stream}) {
        OWRX_CUDA(cudaEventRecord(ev, s));
        OWRX_CUDA(cudaStreamWaitEvent(bank->ctl_stream, ev, 0));
    }
    OWRX_CUDA(cudaStreamWaitEvent(bank->ctl_stream, bank->dev_done, 0));       // the caller's stream (device path)
    OWRX_CUDA(cudaEventRecord(ev, bank->ctl_stream));
    bank->graveyard.emplace_back(std::move(g), ev);
    return OWRX_OK;
}

void reap_groups(owrx_bank* bank, bool wait)
{
    for (size_t i = 0; i < bank->graveyard.size();) {
        auto& e = bank->graveyard[i];
        if (wait) cudaEventSynchronize(e.second);
        if (cudaEventQuery(e.second) != cudaSuccess) { i++; continue; }
        group_release(e.first.get());
        cudaEventDestroy(e.second);
        bank->graveyard.erase(bank->graveyard.begin() + (ptrdiff_t)i);
    }
}

int find_group(owrx_bank* bank, const owrx_chan_spec_t& sp)
{
    for (size_t i = 0; i < bank->groups.size(); i++) {
        Group* g = bank->groups[i].get();
        if (g && spec_equal(g->spec, sp)) return (int)i;
    }
    return -1;
}

void agc_defaults(ChanCfg& c, int kind, int profile)
{
    c.kind = kind;
    c.agc_ref = 0.8f;
    c.agc_attack = 0.1f;
    c.agc_decay = profile == OWRX_AGC_FAST ? 0.001f : 0.0001f;
    c.agc_hang_time = profile == OWRX_AGC_FAST ? 200 : 600;
    c.agc_max = kind == OWRX_DEMOD_NFM ? 3.0f : 65535.0f;               // NFm: agc.setMaxGain(3), analog.py:39
    c.active = 1;
    // exact threshold form of "abs(v)*gain/ref > 1": the largest a with (float)(a / ref) <= 1
    float a = c.agc_ref;
    while (a / c.agc_ref <= 1.0f) a = nextafterf(a, INFINITY);
    c.agc_thr = nextafterf(a, 0.0f);
}

float agc_initial_gain(int kind) { return kind == OWRX_DEMOD_AM ? 200.0f : 1.0f; }   // Am: setInitialGain(200), analog.py:15

void add_patch(Group* g, int slot, int flags, float agc_gain)
{
    SlotPatch& p = g->pend[slot];
    p.slot = slot;
    if (flags & (PATCH_AGC_RESET | PATCH_AGC_GAIN)) p.agc_gain = agc_gain;
    if ((flags & PATCH_AGC_RESET) && (p.flags & PATCH_AGC_GAIN)) p.flags &= ~PATCH_AGC_GAIN;
    p.flags |= flags;
}

int place_channel(owrx_bank* bank, Chan* ch, int gi)
{
    Group* g = bank->groups[(size_t)gi].get();
    int slot = -1;
    for (int s = 0; s < g->slots; s++) if (g->slot_chan[(size_t)s] < 0) { slot = s; break; }
    if (slot < 0) return fail(OWRX_E_STATE, "group full");     // caller grows before placing
    g->slot_chan[(size_t)slot] = ch->id;
    ch->group = gi; ch->slot = slot;
    // a new client's modules start with empty histories and fresh state (the reference builds fresh pycsdr modules): recorded
    // here, applied stream-ordered at the next block boundary (group_begin_feed) — no device synchronisation
    add_patch(g, slot, PATCH_DEMOD | PATCH_AGC_RESET | PATCH_TAIL | PATCH_SQUELCH | PATCH_HISTORY, ch->agc_initial);
    g->h_cfg[(size_t)slot] = ch->cfg;
    g->h_bp_en[(size_t)slot] = 0;
    g->h_tail_mode[(size_t)slot] = ch->audio_fmt;
    g->h_rs[(size_t)slot] = RsCfg{};
    g->cfg_stale[0] = g->cfg_stale[1] = true;
    if (ch->rs_in) { ch->rs_dirty = true; g->rs_pending = true; }    // a moved resampler restarts from empty history
    return OWRX_OK;
}

// grow a group's slot capacity by K3_CG, re-laying out every per-slot table and stage buffer
int group_grow(owrx_bank* bank, Group* g)
{
    // re-laying out every table of the group: rare (every 64th client of a class) and the one control operation that
    // quiesces the device — block kernels on the pipeline's other streams may still read the old arrays
    (void)bank;
    OWRX_CUDA(cudaDeviceSynchronize());
    const int os = g->slots, ns = os + K3_CG;
    auto regrow = [&](auto** p, size_t rows) -> int {
        using T = typename std::remove_pointer<typename std::remove_pointer<decltype(p)>::type>::type;
        T* nb = nullptr;
        int rc = dev_alloc(&nb, rows * (size_t)ns);
        if (rc != OWRX_OK) return rc;
        OWRX_CUDA(cudaMemcpy2D(nb, (size_t)ns * sizeof(T), *p, (size_t)os * sizeof(T), (size_t)os * sizeof(T), rows, cudaMemcpyDeviceToDevice));
        cudaFree(*p);
        *p = nb;
        return OWRX_OK;
    };
    int rc;
    if ((rc = regrow(&g->d_rate, 1)) || (rc = regrow(&g->d_phase, 1)) || (rc = regrow(&g->d_w, 1)) ||
        (rc = regrow(&g->d_bp, (size_t)g->Tb)) || (rc = regrow(&g->d_bp_H, (size_t)g->bpP * FC_M)) ||
        (rc = regrow(&g->d_bp_en2[0], 1)) || (rc = regrow(&g->d_bp_en2[1], 1)) || (rc = regrow(&g->d_cfg2[0], 1)) ||
        (rc = regrow(&g->d_cfg2[1], 1)) || (rc = regrow(&g->d_state, 1)) || (rc = regrow(&g->d_tail_mode2[0], 1)) ||
        (rc = regrow(&g->d_tail_mode2[1], 1)) || (rc = regrow(&g->d_tail, 1)) || (rc = regrow(&g->d_tail_count, 1)) ||
        (rc = regrow(&g->d_rs_cfg2[0], 1)) || (rc = regrow(&g->d_rs_cfg2[1], 1)) ||
        (rc = regrow(&g->d_atap2[0], 1)) || (rc = regrow(&g->d_atap2[1], 1)) || (rc = regrow(&g->d_stash, 1)))
        return rc;
    g->d_cfg = g->d_cfg2[g->cur]; g->d_bp_en = g->d_bp_en2[g->cur]; g->d_tail_mode = g->d_tail_mode2[g->cur];
    g->d_rs_cfg = g->d_rs_cfg2[g->cur]; g->d_atap = g->d_atap2[g->cur];
    cudaFree(g->d_tail_s16); cudaFree(g->d_tail_bytes); cudaFree(g->d_rs);
    g->d_tail_s16 = nullptr; g->d_tail_bytes = nullptr; g->d_rs = nullptr; g->tail_rows_cap = 0; g->tail_cap = 0;
    auto regrow_buf = [&](StageBuf& b) -> int {
        if (!b.d[0]) return OWRX_OK;
        for (int k = 0; k < 2; k++) {
            float* nb = nullptr;
            const size_t orf = (size_t)os * b.width, nrf = (size_t)ns * b.width;
            int rc2 = dev_alloc(&nb, b.cap_rows * nrf);
            if (rc2 != OWRX_OK) return rc2;
            OWRX_CUDA(cudaMemcpy2D(nb, nrf * sizeof(float), b.d[k], orf * sizeof(float), orf * sizeof(float), b.cap_rows, cudaMemcpyDeviceToDevice));
            cudaFree(b.d[k]);
            b.d[k] = nb;
        }
        b.slots = ns;
        return OWRX_OK;
    };
    if ((rc = regrow_buf(g->s1)) || (rc = regrow_buf(g->s2)) || (rc = regrow_buf(g->s3)) || (rc = regrow_buf(g->f1)) || (rc = regrow_buf(g->f1p)) ||
        (rc = regrow_buf(g->f1b)) || (rc = regrow_buf(g->f2)) || (rc = regrow_buf(g->f3)))
        return rc;
    cudaFree(g->d_partial); g->d_partial = nullptr; g->partial_cap = 0;
    cudaFree(g->d_bp_X); cudaFree(g->d_bp_Y);
    g->d_bp_X = nullptr; g->d_bp_Y = nullptr; g->bp_blocks_cap = 0;
    cudaFree(g->d_gate); cudaFree(g->d_power); cudaFree(g->d_dcmean); cudaFree(g->d_dcprev);
    g->d_gate = nullptr; g->d_power = nullptr; g->d_dcmean = nullptr; g->d_dcprev = nullptr; g->blocks_cap = 0;
    // fast-convolution tables are laid out per slot count: rebuild lazily
    cudaFree(g->d_fc_tab); cudaFree(g->d_fc_Z); cudaFree(g->d_fc_slots); cudaFree(g->d_fc_rates); cudaFree(g->d_fc_tabp);
    g->d_fc_tab = nullptr; g->d_fc_Z = nullptr; g->d_fc_slots = nullptr; g->d_fc_rates = nullptr; g->d_fc_tabp = nullptr;
    g->fc_tabp_rate.clear();
    g->fc.slots = ns;
    g->fc_tab_rate.clear();
    g->slots = ns;
    g->slot_chan.resize((size_t)ns, -1);
    g->h_rate.resize((size_t)ns, 0.0); g->h_phase.resize((size_t)ns, 0.0); g->h_w.resize((size_t)ns, make_float2(1.f, 0.f));
    g->h_bp_en.resize((size_t)ns, 0);
    g->h_tail_mode.resize((size_t)ns, 0);
    g->h_rs.resize((size_t)ns, RsCfg{});
    g->h_atap.resize((size_t)ns, TapFmt{OWRX_MPX_OFF, 0});
    ChanCfg idle{}; idle.kind = OWRX_DEMOD_NONE; idle.agc_ref = 0.8f; idle.agc_max = 1.f; idle.agc_thr = 0.8f;
    g->h_cfg.resize((size_t)ns, idle);
    g->cfg_stale[0] = g->cfg_stale[1] = true;
    return OWRX_OK;
}

// Bandpass.setBandpass: the taps (and their partition spectra for the K4F form) are designed on the host and staged in the
// channel; they reach the per-slot tables at the next block boundary (apply_pending), ordered on the stream that reads them
// pure host arithmetic, no bank state: callers run it WITHOUT the bank mutex (a 3125-tap design is ~0.2 ms of host time)
void design_bandpass_stage(std::vector<float2>& stage, int Tb, int bpP, double lo, double hi)
{
    std::vector<float2> taps;
    design_bandpass(taps, Tb, lo, hi);                                   // Bandpass.setBandpass, selector.py:159-166
    const size_t nH = (size_t)bpP * FC_M;
    stage.resize((size_t)Tb + nH);
    std::copy(taps.begin(), taps.end(), stage.begin());
    // partition spectra H[p] = FFT_256([taps[128p .. 128p+127] | 0]) of the SAME float32 taps (double arithmetic, rounded once)
    std::vector<std::complex<double>> buf((size_t)FC_M);
    for (int p = 0; p < bpP; p++) {
        for (int u = 0; u < FC_M; u++) {
            const int t = p * BPF_H + u;
            buf[(size_t)u] = (u < BPF_H && t < Tb) ? std::complex<double>(taps[(size_t)t].x, taps[(size_t)t].y) : std::complex<double>(0.0, 0.0);
        }
        fft_pow2(buf);
        for (int q = 0; q < FC_M; q++)
            stage[(size_t)Tb + (size_t)p * FC_M + q] = make_float2((float)buf[(size_t)q].real(), (float)buf[(size_t)q].imag());
    }
}

// `designed` (optional): a stage designed outside the mutex for exactly this group's (Tb, bpP)
int upload_bandpass(owrx_bank* bank, Chan* ch, std::vector<float2>* designed = nullptr)
{
    Group* g = bank->groups[(size_t)ch->group].get();
    g->h_bp_en[(size_t)ch->slot] = ch->bp_enabled ? 1 : 0;
    g->cfg_stale[0] = g->cfg_stale[1] = true;
    if (!ch->bp_enabled) return OWRX_OK;
    if (designed && designed->size() == (size_t)g->Tb + (size_t)g->bpP * FC_M) ch->bp_stage.swap(*designed);
    else design_bandpass_stage(ch->bp_stage, g->Tb, g->bpP, ch->bp_lo, ch->bp_hi);
    ch->bp_dirty = true;
    g->bp_pending = true;
    return OWRX_OK;
}

// Everything the control path recorded since the last block, as stream-ordered device work.  st_fir owns the FirDecimate
// output history (s1), st_tail every other stage history, the band-pass tables, the squelch / demodulator state and the
// per-slot tables of this block's parity, st_serial the Agc and audio-tail state.  Called after the history rolls.
int apply_pending(owrx_bank* bank, Group* g, cudaStream_t st_fir, cudaStream_t st_tail, cudaStream_t st_serial)
{
    const int S = g->slots;
    if (!g->pend.empty()) {
        std::vector<SlotPatch> v;
        int any_tail_flags = 0, any_serial_flags = 0;
        for (auto& kv : g->pend) {
            v.push_back(kv.second);
            any_tail_flags |= kv.second.flags & (PATCH_DEMOD | PATCH_SQUELCH);
            any_serial_flags |= kv.second.flags & (PATCH_AGC_RESET | PATCH_AGC_GAIN | PATCH_TAIL);
        }
        if ((int)v.size() > g->patch_cap) {
            // first use / more pending slots than ever before: the staging arrays grow (cudaFree waits for their readers)
            const int cap = std::max(S, (int)v.size());
            for (int k = 0; k < 2; k++) {
                cudaFree(g->d_patch[k]); g->d_patch[k] = nullptr;
                OWRX_CUDA(cudaMalloc((void**)&g->d_patch[k], (size_t)cap * sizeof(SlotPatch)));
            }
            g->patch_cap = cap;
        }
        const int n = (int)v.size();
        // pageable sources: cudaMemcpyAsync stages them before it returns, the vector may go
        if (any_tail_flags) {
            OWRX_CUDA(cudaMemcpyAsync(g->d_patch[0], v.data(), (size_t)n * sizeof(SlotPatch), cudaMemcpyHostToDevice, st_tail));
            slot_patch_kernel<<<(n + 127) / 128, 128, 0, st_tail>>>(g->d_patch[0], n, PATCH_DEMOD | PATCH_SQUELCH, g->d_state, g->d_tail);
            OWRX_LAUNCH_CHECK();
            bank->stats.kernel_launches++;
        }
        if (any_serial_flags) {
            OWRX_CUDA(cudaMemcpyAsync(g->d_patch[1], v.data(), (size_t)n * sizeof(SlotPatch), cudaMemcpyHostToDevice, st_serial));
            slot_patch_kernel<<<(n + 127) / 128, 128, 0, st_serial>>>(g->d_patch[1], n, PATCH_AGC_RESET | PATCH_AGC_GAIN | PATCH_TAIL, g->d_state,
                                                                     g->d_tail);
            OWRX_LAUNCH_CHECK();
            bank->stats.kernel_launches++;
        }
        for (const SlotPatch& sp : v) {
            if (!(sp.flags & PATCH_HISTORY)) continue;
            struct { StageBuf* b; cudaStream_t st; } bufs[] = {{&g->s1, st_fir}, {&g->s2, st_tail}, {&g->s3, st_tail}, {&g->f1, st_tail},
                                                              {&g->f1p, st_tail}};
            for (auto& e : bufs) {
                StageBuf* b = e.b;
                if (!b->d[b->cur] || !b->fill) continue;
                OWRX_CUDA(cudaMemset2DAsync(b->d[b->cur] + (size_t)sp.slot * b->width, b->row_floats() * sizeof(float), 0,
                                            (size_t)b->width * sizeof(float), b->fill, e.st));
            }
        }
        g->pend.clear();
    }
    if (g->bp_pending) {
        const size_t per = (size_t)g->Tb + (size_t)g->bpP * FC_M;
        std::vector<Chan*> todo;
        std::vector<int> slots;
        for (int s = 0; s < S; s++) {
            const int cid = g->slot_chan[(size_t)s];
            if (cid < 0) continue;
            Chan* ch = bank->chans[(size_t)cid].get();
            if (!ch || !ch->bp_dirty) continue;
            if (ch->bp_stage.size() == per) { todo.push_back(ch); slots.push_back(s); }
            ch->bp_dirty = false;
        }
        if (!slots.empty()) {
            const int q = g->cur;
            const size_t n = slots.size(), bytes = n * per * sizeof(float2) + n * sizeof(int);
            if (!g->bp_pin_ev[q]) OWRX_CUDA(cudaEventCreateWithFlags(&g->bp_pin_ev[q], cudaEventDisableTiming));
            OWRX_CUDA(cudaEventSynchronize(g->bp_pin_ev[q]));
            if (bytes > g->h_bp_pin_cap[q]) {
                const size_t cap = std::max(bytes, (size_t)16 * (per * sizeof(float2) + sizeof(int)));
                if (g->h_bp_pin[q]) cudaFreeHost(g->h_bp_pin[q]);
                g->h_bp_pin[q] = nullptr; g->h_bp_pin_cap[q] = 0;
                OWRX_CUDA(cudaHostAlloc((void**)&g->h_bp_pin[q], cap, cudaHostAllocDefault));
                g->h_bp_pin_cap[q] = cap;
            }
            if ((int)n > g->bp_stage_cap) {
                const int cap = std::max((int)n, std::min(S, 16));
                cudaFree(g->d_bp_stage); cudaFree(g->d_bp_stage_slots);
                g->d_bp_stage = nullptr; g->d_bp_stage_slots = nullptr; g->bp_stage_cap = 0;
                OWRX_CUDA(cudaMalloc((void**)&g->d_bp_stage, (size_t)cap * per * sizeof(float2)));
                OWRX_CUDA(cudaMalloc((void**)&g->d_bp_stage_slots, (size_t)cap * sizeof(int)));
                g->bp_stage_cap = cap;
            }
            float2* hs = reinterpret_cast<float2*>(g->h_bp_pin[q]);
            int* hi = reinterpret_cast<int*>(g->h_bp_pin[q] + n * per * sizeof(float2));
            for (size_t i = 0; i < n; i++) {
                memcpy(hs + i * per, todo[i]->bp_stage.data(), per * sizeof(float2));
                hi[i] = slots[i];
            }
            OWRX_CUDA(cudaMemcpyAsync(g->d_bp_stage, hs, n * per * sizeof(float2), cudaMemcpyHostToDevice, st_tail));
            OWRX_CUDA(cudaMemcpyAsync(g->d_bp_stage_slots, hi, n * sizeof(int), cudaMemcpyHostToDevice, st_tail));
            OWRX_CUDA(cudaEventRecord(g->bp_pin_ev[q], st_tail));
            bp_scatter_kernel<<<dim3((unsigned)((per + 255) / 256), (unsigned)n), 256, 0, st_tail>>>(
                g->d_bp_stage, g->d_bp_stage_slots, g->Tb, (int)((size_t)g->bpP * FC_M), S, g->d_bp, g->d_bp_H);
            OWRX_LAUNCH_CHECK();
            bank->stats.kernel_launches++;
        }
        g->bp_pending = false;
    }
    // tap layouts of this block (ChanCfg::mpx / mpx_run for the multiplex tap, h_atap for the audio tap)
    g->mpx.clear(); g->atap.clear();
    for (int s = 0; s < S; s++) {
        const int cid = g->slot_chan[(size_t)s];
        const Chan* ch = cid >= 0 ? bank->chans[(size_t)cid].get() : nullptr;
        if (g->wfm) {
            const int fmt = ch ? ch->mpx_fmt : OWRX_MPX_OFF;
            const int run = g->mpx.add(cid, fmt, ch ? ch->gen : 0);
            ChanCfg& c = g->h_cfg[(size_t)s];
            if (c.mpx != fmt || c.mpx_run != run) {
                c.mpx = fmt; c.mpx_run = run;
                g->cfg_stale[0] = g->cfg_stale[1] = true;
            }
        }
        const int fmt = ch ? ch->atap_fmt : OWRX_MPX_OFF;
        const int run = g->atap.add(cid, fmt, ch ? ch->gen : 0);
        TapFmt& a = g->h_atap[(size_t)s];
        if (a.fmt != fmt || a.run != run) {
            a = TapFmt{fmt, run};
            g->cfg_stale[0] = g->cfg_stale[1] = true;
        }
    }
    if (g->rs_pending) {
        // resamplers set, changed or moved since the last block start from empty history at this block's first audio row
        for (int s = 0; s < S; s++) {
            const int cid = g->slot_chan[(size_t)s];
            Chan* ch = cid >= 0 ? bank->chans[(size_t)cid].get() : nullptr;
            if (!ch || !ch->rs_dirty) continue;
            RsCfg c{};
            c.origin = g->f3.abs_end;
            if (ch->rs_in) {
                int L = 0, M = 0, K = 0;
                design_audio_resampler(ch->rs_in, ch->rs_out, &L, &M, &K, nullptr);
                const auto& t = bank->rs_tabs.at(std::make_pair(L, M));         // built by the setter
                c.L = L; c.M = M; c.K = t.K; c.tab = t.d;
            }
            g->h_rs[(size_t)s] = c;
            ch->rs_dirty = false;
            g->cfg_stale[0] = g->cfg_stale[1] = true;
        }
        g->rs_pending = false;
    }
    g->any_rs = false; g->rs_up = 1.0;
    size_t rs_hist = 0;
    for (const RsCfg& c : g->h_rs) {
        if (!c.L) continue;
        g->any_rs = true;
        g->rs_up = std::max(g->rs_up, (double)c.L / c.M);
        rs_hist = std::max(rs_hist, (size_t)c.K);
    }
    g->f3.hist = rs_hist;                            // kept by the next roll (K - 1 rows back from a pass's first output)
    // per-slot tables of this block's parity: a block still in flight on the other streams keeps reading the other copy
    g->d_cfg = g->d_cfg2[g->cur]; g->d_bp_en = g->d_bp_en2[g->cur]; g->d_tail_mode = g->d_tail_mode2[g->cur];
    g->d_rs_cfg = g->d_rs_cfg2[g->cur]; g->d_atap = g->d_atap2[g->cur];
    if (g->cfg_stale[g->cur]) {
        OWRX_CUDA(cudaMemcpyAsync(g->d_cfg, g->h_cfg.data(), (size_t)S * sizeof(ChanCfg), cudaMemcpyHostToDevice, st_tail));
        OWRX_CUDA(cudaMemcpyAsync(g->d_bp_en, g->h_bp_en.data(), (size_t)S * sizeof(int), cudaMemcpyHostToDevice, st_tail));
        OWRX_CUDA(cudaMemcpyAsync(g->d_tail_mode, g->h_tail_mode.data(), (size_t)S * sizeof(int), cudaMemcpyHostToDevice, st_tail));
        OWRX_CUDA(cudaMemcpyAsync(g->d_rs_cfg, g->h_rs.data(), (size_t)S * sizeof(RsCfg), cudaMemcpyHostToDevice, st_tail));
        OWRX_CUDA(cudaMemcpyAsync(g->d_atap, g->h_atap.data(), (size_t)S * sizeof(TapFmt), cudaMemcpyHostToDevice, st_tail));
        g->cfg_stale[g->cur] = false;
    }
    g->any_tail = false;
    for (int m : g->h_tail_mode) if (m) g->any_tail = true;
    return OWRX_OK;
}

inline dim3 grid2d(int slots, size_t rows) { return dim3((unsigned)((slots + 31) / 32), (unsigned)((rows + 3) / 4)); }
const dim3 kBlock2d(32, 4);
constexpr size_t kRowChunk = 4 * 65535;

// optional CUDA-event bracket around a kernel of kind `tag` (OWRX_PROF_*) on its launching stream
int prof_mark(owrx_bank* bank, int tag, cudaStream_t st, bool begin)
{
    if (!bank->profile) return OWRX_OK;
    if (begin) {
        if (bank->prof_used == bank->prof_events.size()) {
            cudaEvent_t a, b;
            OWRX_CUDA(cudaEventCreate(&a));
            OWRX_CUDA(cudaEventCreate(&b));
            bank->prof_events.emplace_back(a, b);
            bank->prof_tags.push_back(tag);
        }
        bank->prof_tags[bank->prof_used] = tag;
        OWRX_CUDA(cudaEventRecord(bank->prof_events[bank->prof_used].first, st));
        bank->prof_open.push_back(bank->prof_used++);
    } else {
        OWRX_CUDA(cudaEventRecord(bank->prof_events[bank->prof_open.back()].second, st));
        bank->prof_open.pop_back();
    }
    return OWRX_OK;
}

// K3F: Shift + FirDecimate of one group by polyphase fast convolution (fastconv.cuh); same outputs as the direct
// K3 pass.  `iq`, `n_avail`, the d_rate/d_phase tables and s1 capacity are already set up by group_fir.
int group_fir_fastconv(owrx_bank* bank, Group* g, const float2* iq, size_t n_avail, size_t n_k, cudaStream_t st, bool tc)
{
    const int S = g->slots;
    int rc;
    FcShape& sh = g->fc;
    if (!g->d_fc_h) {
        OWRX_CUDA(cudaMalloc((void**)&g->d_fc_h, g->fc_taps.size() * sizeof(float)));
        OWRX_CUDA(cudaMemcpyAsync(g->d_fc_h, g->fc_taps.data(), g->fc_taps.size() * sizeof(float), cudaMemcpyHostToDevice, st));
    }
    if (!g->d_fc_slots) {
        OWRX_CUDA(cudaMalloc((void**)&g->d_fc_slots, (size_t)S * sizeof(int)));
        OWRX_CUDA(cudaMalloc((void**)&g->d_fc_rates, (size_t)S * sizeof(double)));
    }
    // zero-fill on `st` (a non-blocking stream: a legacy-stream cudaMemset would not be ordered before the table kernel)
    if (!tc && !g->d_fc_tab) {
        const size_t tab_bytes = (size_t)sh.M * sh.Dp * S * sizeof(float2);
        OWRX_CUDA(cudaMalloc((void**)&g->d_fc_tab, tab_bytes));
        OWRX_CUDA(cudaMemsetAsync(g->d_fc_tab, 0, tab_bytes, st));
        g->fc_tab_rate.assign((size_t)S, NAN);
    }
    if (tc && !g->d_fc_tabp) {
        const size_t tab_bytes = (size_t)fc_tc_planes(sh) * fc_tc_plane_elems_tab(sh) * 2;
        OWRX_CUDA(cudaMalloc(&g->d_fc_tabp, tab_bytes));
        OWRX_CUDA(cudaMemsetAsync(g->d_fc_tabp, 0, tab_bytes, st));
        g->fc_tabp_rate.assign((size_t)S, NAN);
    }
    // ---- (re)build the table columns of retuned / new channels
    {
        std::vector<double>& built = tc ? g->fc_tabp_rate : g->fc_tab_rate;
        std::vector<int> sl;
        std::vector<double> rt;
        for (int s = 0; s < S; s++) {
            const int cid = g->slot_chan[(size_t)s];
            if (cid < 0) continue;
            const double r = bank->chans[(size_t)cid]->rate;
            if (built[(size_t)s] == r) continue;
            built[(size_t)s] = r;
            sl.push_back(s);
            rt.push_back(r);
        }
        if (!sl.empty()) {
            // the staging arrays may still be read by an earlier table launch on another stream: order on the device
            OWRX_CUDA(cudaMemcpyAsync(g->d_fc_slots, sl.data(), sl.size() * sizeof(int), cudaMemcpyHostToDevice, st));
            OWRX_CUDA(cudaMemcpyAsync(g->d_fc_rates, rt.data(), rt.size() * sizeof(double), cudaMemcpyHostToDevice, st));
            // (small pageable sources are staged by the runtime before cudaMemcpyAsync returns: no stream wait, the vectors may go)
            rc = tc ? fc_launch_table_tc(sh, g->d_fc_h, g->d_fc_slots, g->d_fc_rates, (int)sl.size(), g->d_fc_tabp, g->fc_tab_scale, st)
                    : fc_launch_table(sh, g->d_fc_h, g->d_fc_slots, g->d_fc_rates, (int)sl.size(), g->d_fc_tab, st);
            if (rc != OWRX_OK) return rc;
            bank->stats.kernel_launches++;
        }
    }
    // ---- scratch for up to Bmax blocks per pass (branch spectra: 16 B per complex as packed-FMA operands, 12 B as bf16 planes)
    const size_t blocks_total = (n_k + (size_t)sh.Kb - 1) / (size_t)sh.Kb;
    const size_t per_block = (size_t)sh.M * sh.Dp * (tc ? (size_t)fc_tc_planes(sh) * 2 : sizeof(float4));
    // (a pass is cut when its spectra exceed 1 GB: every cut re-reads the table)
    const size_t Bmax = std::max<size_t>(1, std::min<size_t>(4096, ((size_t)1 << 30) / per_block));
    const size_t need = std::min(blocks_total, Bmax);
    const size_t z_cap = std::max(g->fc_blocks_cap, g->fc_blocks_cap_tc);
    if (need > z_cap || (!tc && need > g->fc_blocks_cap) || (tc && need > g->fc_blocks_cap_tc)) {
        OWRX_CUDA(cudaStreamSynchronize(st));
        if (need > z_cap) { cudaFree(g->d_fc_Z); g->d_fc_Z = nullptr; }
        if (!tc) {
            cudaFree(g->d_fc_F); g->d_fc_F = nullptr; g->fc_blocks_cap = 0;
            OWRX_CUDA(cudaMalloc((void**)&g->d_fc_F, need * per_block));
            g->fc_blocks_cap = need;
        } else {
            cudaFree(g->d_fc_Fp); g->d_fc_Fp = nullptr; g->fc_blocks_cap_tc = 0;
            OWRX_CUDA(cudaMalloc(&g->d_fc_Fp, need * per_block));
            g->fc_blocks_cap_tc = need;
        }
    }
    if (!g->d_fc_Z) {
        const size_t cap = std::max(g->fc_blocks_cap, g->fc_blocks_cap_tc);
        OWRX_CUDA(cudaMalloc((void**)&g->d_fc_Z, (size_t)FC_MAXSPLIT * cap * (size_t)sh.M * S * sizeof(float2)));
    }
    float2* out = reinterpret_cast<float2*>(g->s1.append_ptr());
    const bool scaled = tc && sh.tc_levels == 2;
    if (scaled) {
        // operand scaling of the pass (fp16 x 2 form: one read of the input for its largest magnitude; bf16 x 3 needs none)
        if (!g->d_fc_scale) OWRX_CUDA(cudaMalloc((void**)&g->d_fc_scale, 4 * sizeof(float)));
        // (timed with the forward FFTs: the scaling pass is part of what the shared front costs)
        if ((rc = prof_mark(bank, OWRX_PROF_FC_FORWARD, st, true)) != OWRX_OK) return rc;
        if ((rc = fc_launch_scale(sh, iq, (long long)n_avail, g->fc_tab_scale, reinterpret_cast<unsigned*>(g->d_fc_scale + 2), g->d_fc_scale, st)) != OWRX_OK)
            return rc;
        if ((rc = prof_mark(bank, OWRX_PROF_FC_FORWARD, st, false)) != OWRX_OK) return rc;
        bank->stats.kernel_launches += 2;
    }
    for (size_t b0 = 0; b0 < blocks_total; b0 += Bmax) {
        const int B = (int)std::min(Bmax, blocks_total - b0);
        const size_t s_off = b0 * (size_t)sh.Kb * (size_t)sh.D;
        if ((rc = prof_mark(bank, OWRX_PROF_FC_FORWARD, st, true)) != OWRX_OK) return rc;
        rc = tc ? fc_launch_forward_tc(sh, iq + s_off, (long long)(n_avail - s_off), B, g->d_fc_Fp, scaled ? g->d_fc_scale : nullptr, st)
                : fc_launch_forward(sh, iq + s_off, (long long)(n_avail - s_off), B, g->d_fc_F, st);
        if (rc != OWRX_OK) return rc;
        if ((rc = prof_mark(bank, OWRX_PROF_FC_FORWARD, st, false)) != OWRX_OK) return rc;
        if ((rc = prof_mark(bank, OWRX_PROF_FC_CONTRACT, st, true)) != OWRX_OK) return rc;
        int nsplit = 1;
        rc = tc ? fc_launch_contract_tc(sh, g->d_fc_Fp, g->d_fc_tabp, B, g->d_fc_Z, bank->sm_count, bank->fc_tc_form, &nsplit, st)
                : fc_launch_contract(sh, g->d_fc_F, g->d_fc_tab, B, g->d_fc_Z, bank->sm_count, &nsplit, st);
        if (rc != OWRX_OK) return rc;
        if ((rc = prof_mark(bank, OWRX_PROF_FC_CONTRACT, st, false)) != OWRX_OK) return rc;
        if ((rc = prof_mark(bank, OWRX_PROF_FC_INVERSE, st, true)) != OWRX_OK) return rc;
        if ((rc = fc_launch_inverse(sh, g->d_fc_Z, nsplit, B, g->d_rate, g->d_phase, (long long)(b0 * (size_t)sh.Kb), (long long)n_k, out,
                                    scaled ? g->d_fc_scale + 1 : nullptr, st)) != OWRX_OK)
            return rc;
        if ((rc = prof_mark(bank, OWRX_PROF_FC_INVERSE, st, false)) != OWRX_OK) return rc;
        bank->stats.kernel_launches += 3;
    }
    return OWRX_OK;
}

// K3 pass of one group over `n_avail` wideband samples starting at `iq` (device), on stream `st`:
// Shift + FirDecimate for every channel, appended to s1.  May be called several times (chunked host
// feeds) before group_tail runs the remaining stages over all pending rows.
// Returns the number of wideband samples consumed (n_k * D).
int group_fir(owrx_bank* bank, Group* g, const float2* iq, size_t n_avail, size_t* consumed, cudaStream_t st)
{
    *consumed = 0;
    if (n_avail < (size_t)g->T) return OWRX_OK;
    const size_t n_k = (n_avail - (size_t)g->T) / (size_t)g->D + 1;
    if (n_k > (size_t)0x7fffffff) return fail(OWRX_E_INVALID, "block too large");
    const int S = g->slots;
    int rc;

    // ---- per-launch channel tables
    for (int s = 0; s < S; s++) {
        const int cid = g->slot_chan[(size_t)s];
        if (cid < 0) { g->h_rate[(size_t)s] = 0.0; g->h_phase[(size_t)s] = 0.0; g->h_w[(size_t)s] = make_float2(1.f, 0.f); continue; }
        Chan* ch = bank->chans[(size_t)cid].get();
        g->h_rate[(size_t)s] = ch->rate;
        g->h_phase[(size_t)s] = ch->phase;
        const double a = 2.0 * M_PI * (ch->rate - floor(ch->rate));
        g->h_w[(size_t)s] = make_float2((float)cos(a), (float)sin(a));
    }
    OWRX_CUDA(cudaMemcpyAsync(g->d_rate, g->h_rate.data(), (size_t)S * sizeof(double), cudaMemcpyHostToDevice, st));
    OWRX_CUDA(cudaMemcpyAsync(g->d_phase, g->h_phase.data(), (size_t)S * sizeof(double), cudaMemcpyHostToDevice, st));
    OWRX_CUDA(cudaMemcpyAsync(g->d_w, g->h_w.data(), (size_t)S * sizeof(float2), cudaMemcpyHostToDevice, st));

    const bool fastconv = g->fc_ok && bank->fir_mode != OWRX_FIR_DIRECT && (bank->fir_mode >= OWRX_FIR_FASTCONV || n_k >= 64);
    if (fastconv) {
        // contraction on the tensor cores once a pass holds enough overlap-save blocks B for the S slots of the group.  Per
        // (bin, branch) the FP32-pipe form costs 8 B S FLOP at ~35 TFLOP/s (it is FMA-bound; its table is 8 bytes per entry),
        // the tensor-core form moves 12 (B + S) bytes at ~3.3 TB/s for short passes (table 12 bytes per entry, read once per
        // pass): tensor cores win for B > ~21 at 64 slots and B > ~18 at 128.  Measured: C3 (128 slots, B = 15) 0.57 ms on
        // the FP32 pipe vs 0.69 ms on the tensor cores; C2 (64 slots, B = 88) 0.29 vs 0.10 ms.
        const size_t fc_blocks = (n_k + (size_t)g->fc.Kb - 1) / (size_t)g->fc.Kb;
        const double fp32_cost = 8.0 * (double)fc_blocks * S / 35e12, tc_cost = 4.0 * g->fc.tc_levels * ((double)fc_blocks + S) / 3.3e12;
        const bool tc = bank->fir_mode == OWRX_FIR_FASTCONV_TC || (bank->fir_mode == OWRX_FIR_AUTO && fp32_cost > tc_cost);
        bank->fir_form_used = tc ? OWRX_FIR_FASTCONV_TC : OWRX_FIR_FASTCONV;
        if ((rc = g->s1.ensure_new(n_k, st)) != OWRX_OK) return rc;
        if ((rc = group_fir_fastconv(bank, g, iq, n_avail, n_k, st, tc)) != OWRX_OK) return rc;
    } else {
    bank->fir_form_used = OWRX_FIR_DIRECT;
    // ---- K3: Shift + FirDecimate
    const int nparts = g->nseg * g->nrs;
    const int ncg = S / K3_CG;
    const size_t fixed = (size_t)nparts * ncg;
    // input-stationary ranges of JB blocks (>= 28 so that an output straddles at most two ranges)
    const size_t n_blocks = n_k + K3_PP - 1;
    const size_t sms = (size_t)bank->sm_count - (bank->reserve_sm ? 1 : 0);
    size_t n_ranges = std::max<size_t>(1, sms / fixed);
    n_ranges = std::min(n_ranges, std::max<size_t>(1, n_blocks / K3_PP));
    const int JB = (int)((n_blocks + n_ranges - 1) / n_ranges);
    n_ranges = (n_blocks + JB - 1) / JB;
    const size_t pneed = (size_t)nparts * n_k * S + (size_t)nparts * n_ranges * (K3_PP - 1) * S;
    if (pneed > g->partial_cap) {
        cudaFree(g->d_partial); g->d_partial = nullptr; g->partial_cap = 0;
        OWRX_CUDA(cudaMalloc((void**)&g->d_partial, pneed * sizeof(float2)));
        g->partial_cap = pneed;
    }
    if ((rc = g->s1.ensure_new(n_k, st)) != OWRX_OK) return rc;
    K3Params p;
    p.iq = iq; p.n_lim = (long long)n_avail; p.taps = g->d_taps;
    p.ch_rate = g->d_rate; p.ch_phase = g->d_phase; p.ch_w = g->d_w;
    p.partial = g->d_partial;
    p.side = g->d_partial + (size_t)nparts * n_k * S;
    p.D = g->D; p.nseg = g->nseg; p.nrs = g->nrs; p.RB = g->RB; p.JB = JB; p.n_blocks = (int)n_blocks; p.n_k = (int)n_k; p.slots = S;
    const size_t smem = (size_t)g->RB * K3_PP * sizeof(float) + 2 * (size_t)g->RB * sizeof(float2) + 2 * K3_NW * 128 * sizeof(float);
    if ((rc = prof_mark(bank, OWRX_PROF_K3_DIRECT, st, true)) != OWRX_OK) return rc;
    if ((rc = launch_fir_decimate(p, dim3((unsigned)(n_ranges * nparts), (unsigned)ncg), smem, st)) != OWRX_OK) return rc;
    if ((rc = prof_mark(bank, OWRX_PROF_K3_DIRECT, st, false)) != OWRX_OK) return rc;
    bank->stats.kernel_launches++;
    {
        const size_t total = n_k * (size_t)S;
        fir_reduce_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(p.partial, p.side, nparts, (int)n_ranges, JB, (int)n_k, S,
                                                                           reinterpret_cast<float2*>(g->s1.append_ptr()));
        OWRX_LAUNCH_CHECK();
        bank->stats.kernel_launches++;
    }
    }
    if (g->pend_rows == 0) g->pend_first = g->s1.abs_end;
    g->s1.appended(n_k);
    g->pend_rows += n_k;
    *consumed = n_k * (size_t)g->D;

    // ---- advance NCO phases
    for (int s = 0; s < S; s++) {
        const int cid = g->slot_chan[(size_t)s];
        if (cid < 0) continue;
        Chan* ch = bank->chans[(size_t)cid].get();
        double ph = ch->phase + ch->rate * (double)(*consumed);
        ch->phase = ph - floor(ph);
    }
    return OWRX_OK;
}

// Every stage after FirDecimate, over the s1 rows appended since the last call, on stream `st`.
int group_tail(owrx_bank* bank, Group* g, cudaStream_t st)
{
    g->pass_audio = 0;
    const size_t n_k = g->pend_rows;
    const long long s1_first = g->pend_first;
    g->pend_rows = 0;
    if (!n_k) return OWRX_OK;
    const int S = g->slots;
    int rc;

    // ---- FractionalDecimator (complex)
    const StageBuf* bp_in = &g->s1;
    long long bp_first = s1_first;
    size_t n2 = n_k;
    if (g->has_frac) {
        // count outputs m with ceil(5 + m*rate) + 6 < s1.abs_end (same double arithmetic as the kernel)
        size_t cnt = 0;
        while (true) {
            const double where = 5.0 + (double)(g->frac_m + (long long)cnt) * g->frac;
            if ((long long)ceil(where) + 6 >= g->s1.abs_end) break;
            cnt++;
        }
        n2 = cnt;
        if ((rc = g->s2.ensure_new(n2, st)) != OWRX_OK) return rc;
        for (size_t o = 0; o < n2; o += kRowChunk) {
            const size_t c = std::min(kRowChunk, n2 - o);
            fracdec_cf_kernel<<<grid2d(S, c), kBlock2d, 0, st>>>(
                reinterpret_cast<const float2*>(g->s1.rows()), g->s1.abs_end - (long long)g->s1.fill, S, nullptr, g->frac,
                g->frac_m + (long long)o, (int)c, S, reinterpret_cast<float2*>(g->s2.append_ptr()) + o * S);
            OWRX_LAUNCH_CHECK();
            bank->stats.kernel_launches++;
        }
        bp_first = g->s2.abs_end;
        g->s2.appended(n2);
        g->frac_m += (long long)n2;
        bp_in = &g->s2;
    }

    // ---- Bandpass -> s3 (selector output / IF)
    if ((rc = g->s3.ensure_new(n2, st)) != OWRX_OK) return rc;
    // long band-pass filters only (the 250 kHz WFM IF: 3125 taps): for the 151-tap filters of the 12 kHz classes the direct
    // form is cheap and keeps full relative precision on near-zero samples (start-up transients feed a scale-free FmDemod)
    const bool bp_fft = g->bpP > 4 && bank->bp_mode != OWRX_FIR_DIRECT && (bank->bp_mode == OWRX_FIR_FASTCONV || n2 >= 4 * (size_t)BPF_H);
    if (bp_fft) {
        // K4F: partitioned overlap-save on 256-point FFTs, in passes of at most kBpBlocks hops
        const size_t kBpBlocks = std::max<size_t>(1, ((size_t)96 << 20) / ((size_t)FC_M * S * sizeof(float2)));
        const size_t blocks_total = (n2 + BPF_H - 1) / BPF_H;
        const size_t need = std::min(blocks_total, kBpBlocks);
        if (need > g->bp_blocks_cap) {
            OWRX_CUDA(cudaStreamSynchronize(st));
            cudaFree(g->d_bp_X); cudaFree(g->d_bp_Y);
            g->d_bp_X = nullptr; g->d_bp_Y = nullptr; g->bp_blocks_cap = 0;
            OWRX_CUDA(cudaMalloc((void**)&g->d_bp_X, (need + (size_t)g->bpP) * FC_M * S * sizeof(float2)));
            OWRX_CUDA(cudaMalloc((void**)&g->d_bp_Y, need * FC_M * S * sizeof(float2)));
            g->bp_blocks_cap = need;
        }
        for (size_t b0 = 0; b0 < blocks_total; b0 += kBpBlocks) {
            const int nblk = (int)std::min(kBpBlocks, blocks_total - b0);
            const size_t o = b0 * BPF_H;
            const float2* src = reinterpret_cast<const float2*>(bp_in->row_abs(bp_first + (long long)o));
            const int rows_here = (int)std::min<size_t>((size_t)nblk * BPF_H, n2 - o);
            if ((rc = bpf_launch_forward(src, S, (int)(n2 - o) - 1, g->bpP, nblk, g->d_bp_X, st)) != OWRX_OK) return rc;
            if ((rc = bpf_launch_mac(g->d_bp_X, g->d_bp_H, S, g->bpP, nblk, g->d_bp_Y, st)) != OWRX_OK) return rc;
            if ((rc = bpf_launch_inverse(g->d_bp_Y, src, g->d_bp_en, S, nblk, rows_here,
                                         reinterpret_cast<float2*>(g->s3.append_ptr()) + o * S, st)) != OWRX_OK)
                return rc;
            bank->stats.kernel_launches += 3;
        }
    } else
    for (size_t o = 0; o < n2; o += kRowChunk * BP_RB) {
        const size_t c = std::min(kRowChunk * BP_RB, n2 - o);
        bandpass_kernel<<<grid2d(S, (c + BP_RB - 1) / BP_RB), kBlock2d, 0, st>>>(
            reinterpret_cast<const float2*>(bp_in->row_abs(bp_first + (long long)o)), S, nullptr, g->d_bp, g->d_bp_en, g->Tb,
            (int)c, S, reinterpret_cast<float2*>(g->s3.append_ptr()) + o * S);
        OWRX_LAUNCH_CHECK();
        bank->stats.kernel_launches++;
    }
    g->s3.appended(n2);
    g->last_if += n2;

    // ---- Squelch over whole blocks
    const size_t pending = (size_t)(g->s3.abs_end - g->sq_abs);
    const size_t nb = pending / (size_t)g->sq_len;
    const size_t n4 = nb * (size_t)g->sq_len;
    g->last_blocks += nb;
    g->sq_block_abs += (long long)nb;
    if (nb) {
        if (g->feed_blocks + nb > g->blocks_cap) return fail(OWRX_E_STATE, "squelch scratch under-provisioned");
        // per-block scratch of this pass sits behind the blocks of earlier passes of the same feed
        unsigned char* const d_gate = g->d_gate + g->feed_blocks * (size_t)S;
        float* const d_power = g->d_power + g->feed_blocks * (size_t)S;
        float* const d_dcmean = g->d_dcmean + g->feed_blocks * (size_t)S;
        g->feed_blocks += nb;
        const float2* sq_in = reinterpret_cast<const float2*>(g->s3.row_abs(g->sq_abs));
        const int hang_blocks = 2;                                       // hangLength = 2*blockLength, selector.py:124
        // one launch for Squelch + demodulator front + DcBlock means (tail_front_kernel) unless OWRX_TAIL_FUSED=0 asks for the
        // seven-kernel evaluation (kept as the second opinion: tests/test_gpu_selector.py runs both)
        // the fused front re-derives the block powers its gate needs in EVERY CTA of a block: fine while a squelch block is one or
        // two CTAs long (12 kHz: 750 rows), 7x redundant reads for the 15 625-row blocks of a 250 kHz WFM IF (C5: 190 us vs 60 us)
        const bool fused = bank->tail_fused && nb <= 65535 && g->sq_len <= 2 * TF_ROWS;
        if ((rc = g->f1.ensure_new(n4, st)) != OWRX_OK) return rc;
        if (fused) {
            const unsigned zsplit = (unsigned)((g->sq_len + TF_ROWS - 1) / TF_ROWS);
            tail_front_kernel<<<dim3((unsigned)(S / 32), (unsigned)nb, zsplit), 256, 0, st>>>(
                sq_in, S, (int)nb, g->sq_len, 5, hang_blocks, g->d_cfg, g->d_state, d_power, d_gate, g->f1.append_ptr(), d_dcmean,
                g->d_dcprev, g->d_stash);
            OWRX_LAUNCH_CHECK();
            tail_commit_kernel<<<(S + 127) / 128, 128, 0, st>>>(S, (int)nb, g->d_cfg, d_dcmean, g->d_stash, g->d_state);
            OWRX_LAUNCH_CHECK();
            bank->stats.kernel_launches += 2;
        } else {
        squelch_power_kernel<<<dim3((unsigned)(S / 32), (unsigned)nb), 256, 0, st>>>(sq_in, S, (int)nb, g->sq_len, 5, d_power);
        OWRX_LAUNCH_CHECK();
        squelch_gate_kernel<<<(S + 127) / 128, 128, 0, st>>>(d_power, S, (int)nb, hang_blocks, g->d_cfg, g->d_state, d_gate);
        OWRX_LAUNCH_CHECK();
        // ---- demodulator front -> f1
        {
            // single logical launch split in row chunks that are multiples of sq_len
            const size_t chunk_rows = std::max<size_t>((size_t)g->sq_len, (kRowChunk / (size_t)g->sq_len) * (size_t)g->sq_len);
            for (size_t o = 0; o < n4; o += chunk_rows) {
                const size_t c = std::min(chunk_rows, n4 - o);
                // FM needs the previous row: for o > 0 it is in the buffer; state is only used at o == 0
                demod_front_kernel<<<grid2d(S, c), kBlock2d, 0, st>>>(sq_in + o * S, S, (int)c, g->sq_len,
                                                                      d_gate + (o / (size_t)g->sq_len) * S, g->d_cfg,
                                                                      g->d_state, g->f1.append_ptr() + o * S);
                OWRX_LAUNCH_CHECK();
                if (o + c < n4) {
                    // make the carried "last gated sample" right for the next chunk
                    demod_front_commit_kernel<<<(S + 127) / 128, 128, 0, st>>>(sq_in + o * S, S, (int)c, g->sq_len,
                                                                              d_gate + (o / (size_t)g->sq_len) * S, g->d_state);
                    OWRX_LAUNCH_CHECK();
                }
            }
            demod_front_commit_kernel<<<(S + 127) / 128, 128, 0, st>>>(sq_in, S, (int)n4, g->sq_len, d_gate, g->d_state);
            OWRX_LAUNCH_CHECK();
        }
        bank->stats.kernel_launches += 3;
        }
        const long long f1_first = g->f1.abs_end;
        g->f1.appended(n4);
        g->sq_abs += (long long)n4;
        if (g->wfm && !g->mpx.runs.empty()) {
            // ---- multiplex tap: the tapped slots' new f1 rows -> their staging runs (on the stream that owns f1, before it rolls)
            if ((rc = prof_mark(bank, OWRX_PROF_TAP, st, true)) != OWRX_OK) return rc;
            if ((rc = g->mpx.gather(bank->stats, g->f1.row_abs(f1_first), S, n4, MpxTapSel{g->d_cfg}, g->cur, st)) != OWRX_OK) return rc;
            if ((rc = prof_mark(bank, OWRX_PROF_TAP, st, false)) != OWRX_OK) return rc;
        }

        size_t n_audio = 0;
        if (!g->wfm) {
            // ---- demodulator back: NfmDeemphasis / DcBlock / copy -> f2 (pre-AGC)
            if (!fused) {
                dc_mean_kernel<<<dim3((unsigned)(S / 32), (unsigned)nb), 256, 0, st>>>(g->f1.row_abs(f1_first), S, (int)nb,
                                                                                            g->sq_len, g->d_cfg, g->d_state,
                                                                                            d_dcmean, g->d_dcprev);
                OWRX_LAUNCH_CHECK();
            }
            if ((rc = g->f2.ensure_new(n4, st)) != OWRX_OK) return rc;
            const size_t chunk_rows = std::max<size_t>((size_t)g->sq_len, (kRowChunk / (size_t)g->sq_len) * (size_t)g->sq_len);
            for (size_t o = 0; o < n4; o += chunk_rows) {
                const size_t c = std::min(chunk_rows, n4 - o);
                demod_back_kernel<<<grid2d(S, (c + DB_RB - 1) / DB_RB), kBlock2d, 0, st>>>(g->f1.row_abs(f1_first + (long long)o), S, (int)c, g->sq_len,
                                                                     g->d_deemph, g->Td, g->d_cfg,
                                                                     d_dcmean + (o / (size_t)g->sq_len) * S,
                                                                     o == 0 ? g->d_dcprev : d_dcmean + (o / (size_t)g->sq_len - 1) * S,
                                                                     g->f2.append_ptr() + o * S);
                OWRX_LAUNCH_CHECK();
            }
            if (!fused) {
                dc_commit_kernel<<<(S + 127) / 128, 128, 0, st>>>(S, (int)nb, g->d_cfg, d_dcmean, g->d_state);
                OWRX_LAUNCH_CHECK();
            }
            bank->stats.kernel_launches += fused ? 1 : 3;
            g->f2.appended(n4);
            n_audio = n4;
        } else {
            // ---- WFM: prefilter (133-tap LPF, once per input index) -> 12-point Lagrange to the audio rate -> de-emphasis
            const long long v_end = g->f1.abs_end - (long long)(g->Tpre - 1);      // prefilter looks Tpre-1 samples ahead
            const size_t nv = v_end > g->f1p.abs_end ? (size_t)(v_end - g->f1p.abs_end) : 0;
            if (nv) {
                if ((rc = g->f1p.ensure_new(nv, st)) != OWRX_OK) return rc;
                const float* src = g->f1.row_abs(g->f1p.abs_end);
                const int last_row = (int)(g->f1.abs_end - 1 - g->f1p.abs_end);
                for (size_t o = 0; o < nv; o += kRowChunk * BP_RB) {
                    const size_t c = std::min(kRowChunk * BP_RB, nv - o);
                    fir_fwd_f_kernel<<<grid2d(S, (c + BP_RB - 1) / BP_RB), kBlock2d, 0, st>>>(src + o * S, S, (int)c, last_row - (int)o, g->d_pre,
                                                                                           g->Tpre, g->f1p.append_ptr() + o * S);
                    OWRX_LAUNCH_CHECK();
                }
                g->f1p.appended(nv);
            }
            size_t cnt = 0;
            while (true) {
                const double where = 5.0 + (double)(g->wfm_m + (long long)cnt) * g->wfm_rate;
                if ((long long)ceil(where) + 6 >= g->f1p.abs_end) break;
                cnt++;
            }
            if ((rc = g->f1b.ensure_new(cnt, st)) != OWRX_OK) return rc;
            if ((rc = g->f2.ensure_new(cnt, st)) != OWRX_OK) return rc;
            for (size_t o = 0; o < cnt; o += kRowChunk) {
                const size_t c = std::min(kRowChunk, cnt - o);
                fracdec_f_kernel<<<grid2d(S, c), kBlock2d, 0, st>>>(g->f1p.rows(), g->f1p.abs_end - (long long)g->f1p.fill, S,
                                                                    g->wfm_rate, g->wfm_m + (long long)o, (int)c, nullptr, 0,
                                                                    g->f1b.append_ptr() + o * S);
                OWRX_LAUNCH_CHECK();
            }
            if (cnt) {
                wfm_deemph_kernel<<<S / IIR_CH, IIR_TL, 0, st>>>(g->f1b.append_ptr(), S, (int)cnt, g->alpha, g->d_state,
                                                                  g->f2.append_ptr());
                OWRX_LAUNCH_CHECK();
            }
            bank->stats.kernel_launches += 2;
            g->wfm_m += (long long)cnt;
            g->f2.appended(cnt);
            n_audio = cnt;
        }
        g->last_demod += n_audio;
        g->last_audio += n_audio;
        g->pass_audio = n_audio;
    }
    return OWRX_OK;
}

// The sample-serial end of the chain (Agc, then the client audio tail) over the rows group_tail produced.
// One warp per 32 channels: negligible resources, so it may run on a side stream beside the next K3 pass.
int group_tail_serial(owrx_bank* bank, Group* g, cudaStream_t st)
{
    const int S = g->slots;
    const size_t n_audio = g->pass_audio;
    int rc;
    {
        // ---- Agc -> f3
        if (n_audio) {
            if ((rc = g->f3.ensure_new(n_audio, st)) != OWRX_OK) return rc;
            if ((rc = prof_mark(bank, OWRX_PROF_AGC, st, true)) != OWRX_OK) return rc;
            if (g->wfm) {
                // the WFm chain has no Agc (csdr/chain/analog.py:55-67): the audio is the de-emphasised signal
                OWRX_CUDA(cudaMemcpyAsync(g->f3.append_ptr(), g->f2.rows(g->f2.fill - n_audio), n_audio * (size_t)S * sizeof(float),
                                          cudaMemcpyDeviceToDevice, st));
            } else {
                // The Agc is a latency-bound dependent chain (one warp per channel): every cycle another kernel's warps take
                // on its scheduler stretches it.  Its CTAs therefore claim 160 KB of dynamic shared memory they do not use
                // (189 KB with their own buffers), so that neither a contraction CTA (>= 58 KB since the 16-branch stages) nor
                // a 66 KB FFT CTA can share their SM (measured inside the three-stream pipeline, C2, with a 100 KB claim while
                // the contraction needed 177 KB: Agc stage 0.32 -> 0.26 ms, step 0.34 -> 0.32 ms).  OWRX_AGC_PAD_KB overrides.
                static const int agc_pad = (getenv("OWRX_AGC_PAD_KB") ? atoi(getenv("OWRX_AGC_PAD_KB")) : 160) << 10;
                if (agc_pad) OWRX_CUDA(cudaFuncSetAttribute(agc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, agc_pad));
                agc_kernel<<<S / AGC_CH, AGC_TL, agc_pad, st>>>(g->f2.rows(g->f2.fill - n_audio), S, (int)n_audio, g->d_cfg, g->d_state,
                                                           g->f3.append_ptr());
                OWRX_LAUNCH_CHECK();
            }
            if ((rc = prof_mark(bank, OWRX_PROF_AGC, st, false)) != OWRX_OK) return rc;
            bank->stats.kernel_launches++;
            g->f3.appended(n_audio);
            if (!g->atap.runs.empty()) {
                // ---- audio tap: the tapped slots' new f3 rows -> their staging runs (on the stream that writes f3, before it rolls)
                if ((rc = prof_mark(bank, OWRX_PROF_TAP, st, true)) != OWRX_OK) return rc;
                if ((rc = g->atap.gather(bank->stats, g->f3.rows(g->f3.fill - n_audio), S, n_audio, AudioTapSel{g->d_atap}, g->cur, st)) != OWRX_OK)
                    return rc;
                if ((rc = prof_mark(bank, OWRX_PROF_TAP, st, false)) != OWRX_OK) return rc;
            }
            if (g->any_tail) {
                // ---- client audio tail: [AudioResampler + Limit] Convert(FLOAT, SHORT) [+ AdpcmEncoder(sync=True)]; appends
                // behind earlier passes.  a0: absolute audio row of this pass's first row; the feed's rows start at audio_af.
                const long long a0 = g->f3.abs_end - (long long)n_audio;
                if (g->last_audio > g->tail_rows_cap) return fail(OWRX_E_STATE, "audio tail scratch under-provisioned");
                if (g->any_rs) {
                    // per-slot output counts follow from (L, M, origin) alone: the host sizes the launch without a read-back
                    long long most = 0;
                    for (const RsCfg& c : g->h_rs) {
                        if (!c.L) continue;
                        g->rs_rows = std::max(g->rs_rows, (size_t)(rs_outputs(c, a0 + (long long)n_audio) - rs_outputs(c, g->audio_af)));
                        most = std::max(most, rs_outputs(c, a0 + (long long)n_audio) - rs_outputs(c, a0));
                    }
                    if (g->rs_rows > g->tail_rows_cap) return fail(OWRX_E_STATE, "audio resampler scratch under-provisioned");
                    const long long per_cta = (long long)RS_WARPS * RS_T;
                    const unsigned gy = (unsigned)std::max(1LL, std::min(65535LL, (most + per_cta - 1) / per_cta));
                    if ((rc = prof_mark(bank, OWRX_PROF_RESAMPLE, st, true)) != OWRX_OK) return rc;
                    audio_resample_kernel<<<dim3((unsigned)(S / 32), gy), 32 * RS_WARPS, 0, st>>>(
                        g->f3.rows(0), g->f3.abs_end - (long long)g->f3.fill, S, g->d_rs_cfg, g->d_tail_mode, a0, (int)n_audio,
                        g->audio_af, g->d_rs);
                    OWRX_LAUNCH_CHECK();
                    if ((rc = prof_mark(bank, OWRX_PROF_RESAMPLE, st, false)) != OWRX_OK) return rc;
                    bank->stats.kernel_launches++;
                }
                audio_tail_kernel<<<(S + 31) / 32, 128, 0, st>>>(g->f3.rows(g->f3.fill - n_audio), S, (int)n_audio, g->d_tail_mode,
                                                               g->d_tail, g->d_tail_s16, g->d_tail_bytes, g->d_tail_count, g->tail_cap,
                                                               g->d_rs, g->any_rs ? g->d_rs_cfg : nullptr, a0, g->audio_af);
                OWRX_LAUNCH_CHECK();
                bank->stats.kernel_launches++;
                g->tail_ran = true;
            }
        }
    }
    return OWRX_OK;
}

// rows of the client-audio tail's scratch for a feed of up to `low` audio rows: a resampled slot may produce more (L > M)
size_t tail_rows(const Group* g, size_t low)
{
    return g->any_rs ? std::max(low, (size_t)ceil((double)low * g->rs_up) + 2) : low;
}

// (re)allocates the audio tail's scratch: int16 rows, ADPCM bytes per slot and, with a resampler, the resampled float rows
int alloc_tail(Group* g, size_t rows)
{
    const size_t S = (size_t)g->slots;
    const int cap = (int)(rows / 2 + 8 * (rows / 2002 + 2) + 16);
    cudaFree(g->d_tail_s16); cudaFree(g->d_tail_bytes); cudaFree(g->d_rs);
    g->d_tail_s16 = nullptr; g->d_tail_bytes = nullptr; g->d_rs = nullptr; g->tail_rows_cap = 0; g->tail_cap = 0;
    OWRX_CUDA(cudaMalloc((void**)&g->d_tail_s16, rows * S * sizeof(int16_t)));
    OWRX_CUDA(cudaMalloc((void**)&g->d_tail_bytes, (size_t)cap * S));
    if (g->any_rs) OWRX_CUDA(cudaMalloc((void**)&g->d_rs, rows * S * sizeof(float)));
    g->tail_rows_cap = rows; g->tail_cap = cap;
    return OWRX_OK;
}

// Start of a feed / device block: drop the previous outputs (histories stay), reset the per-feed counters and
// provision every buffer for up to `rows` new FirDecimate outputs so that nothing reallocates while the
// streams overlap.
int group_begin_feed(owrx_bank* bank, Group* g, size_t rows, cudaStream_t st_fir, cudaStream_t st_tail, cudaStream_t st_serial, int parity)
{
    const int S = g->slots;
    int rc;
    g->cur = parity & 1;
    const size_t blocks = rows / (size_t)g->sq_len + 2;
    const size_t low = rows + (size_t)g->sq_len + 64;           // rows any low-rate stage can append in one feed
    if ((rc = g->s1.roll(g->s1.hist, st_fir)) != OWRX_OK) return rc;
    if (g->has_frac && (rc = g->s2.roll(g->s2.hist, st_tail)) != OWRX_OK) return rc;
    if ((rc = g->s3.roll(g->s3.hist, st_tail)) != OWRX_OK) return rc;
    if ((rc = g->f1.roll(g->f1.hist, st_tail)) != OWRX_OK) return rc;
    if (g->wfm) { g->f1b.roll(0, st_tail); if ((rc = g->f1p.roll(g->f1p.hist, st_tail)) != OWRX_OK) return rc; }
    g->f2.roll(0, st_tail);
    // f3 keeps the resampler's look-back (none without one); the Agc that wrote it and the copy are on the serial stream, and
    // the copy's destination may still be read by a split-phase drain
    if (g->f3.hist && g->f3.drained[g->f3.cur ^ 1]) OWRX_CUDA(cudaStreamWaitEvent(st_serial, g->f3.drained[g->f3.cur ^ 1], 0));
    if ((rc = g->f3.roll(g->f3.hist, st_serial)) != OWRX_OK) return rc;
    g->audio_af = g->f3.abs_end;
    g->rs_rows = 0;
    g->last_audio = g->last_demod = g->last_if = g->last_blocks = 0;
    g->dr_audio = g->dr_demod = g->dr_if = g->dr_blocks = 0;
    g->dr_final = false;
    g->sq_block_first = g->sq_block_abs;
    g->pass_audio = 0; g->feed_blocks = 0; g->tail_ran = false;
    const bool grow = g->s1.fill + rows > g->s1.cap_rows || (g->has_frac && g->s2.fill + low > g->s2.cap_rows) ||
                      g->s3.fill + low > g->s3.cap_rows || g->f1.fill + low > g->f1.cap_rows || low > g->f2.cap_rows ||
                      g->f3.fill + low > g->f3.cap_rows || (g->wfm && (low > g->f1b.cap_rows || g->f1p.fill + low > g->f1p.cap_rows)) ||
                      blocks > g->blocks_cap || (g->any_tail && tail_rows(g, low) > g->tail_rows_cap);
    if (grow) {
        OWRX_CUDA(cudaDeviceSynchronize());
        if ((rc = g->s1.ensure_new(rows, st_fir)) != OWRX_OK) return rc;
        if (g->has_frac && (rc = g->s2.ensure_new(low, st_tail)) != OWRX_OK) return rc;
        if ((rc = g->s3.ensure_new(low, st_tail)) != OWRX_OK) return rc;
        if ((rc = g->f1.ensure_new(low, st_tail)) != OWRX_OK) return rc;
        if (g->wfm && (rc = g->f1b.ensure_new(low, st_tail)) != OWRX_OK) return rc;
        if (g->wfm && (rc = g->f1p.ensure_new(low, st_tail)) != OWRX_OK) return rc;
        if ((rc = g->f2.ensure_new(low, st_tail)) != OWRX_OK) return rc;
        if ((rc = g->f3.ensure_new(low, st_tail)) != OWRX_OK) return rc;
        if (blocks > g->blocks_cap) {
            cudaFree(g->d_gate); cudaFree(g->d_power); cudaFree(g->d_dcmean); cudaFree(g->d_dcprev);
            g->d_gate = nullptr; g->d_power = nullptr; g->d_dcmean = nullptr; g->d_dcprev = nullptr; g->blocks_cap = 0;
            OWRX_CUDA(cudaMalloc((void**)&g->d_gate, blocks * (size_t)S));
            OWRX_CUDA(cudaMalloc((void**)&g->d_power, blocks * (size_t)S * sizeof(float)));
            OWRX_CUDA(cudaMalloc((void**)&g->d_dcmean, blocks * (size_t)S * sizeof(float)));
            OWRX_CUDA(cudaMalloc((void**)&g->d_dcprev, (size_t)S * sizeof(float)));
            g->blocks_cap = blocks;
        }
        if (g->any_tail && tail_rows(g, low) > g->tail_rows_cap && (rc = alloc_tail(g, tail_rows(g, low))) != OWRX_OK) return rc;
        OWRX_CUDA(cudaDeviceSynchronize());
    }
    if ((rc = apply_pending(bank, g, st_fir, st_tail, st_serial)) != OWRX_OK) return rc;
    if (g->any_tail) {
        // the audio tail's scratch follows any_tail and the resamplers, which apply_pending has just refreshed
        if (tail_rows(g, low) > g->tail_rows_cap || (g->any_rs && !g->d_rs)) {
            OWRX_CUDA(cudaDeviceSynchronize());
            if ((rc = alloc_tail(g, std::max(tail_rows(g, low), g->tail_rows_cap))) != OWRX_OK) return rc;
        }
        OWRX_CUDA(cudaMemsetAsync(g->d_tail_count, 0, (size_t)S * sizeof(int), st_serial));
    }
    // the tap staging follows the layouts apply_pending has just rebuilt; f1 and f3 append at most `low` rows per feed
    if ((rc = g->mpx.provision(low)) != OWRX_OK || (rc = g->atap.provision(low)) != OWRX_OK) return rc;
    return OWRX_OK;
}

Chan* get_chan(owrx_bank* bank, int chan)
{
    if (!bank || chan < 0 || (size_t)chan >= bank->chans.size()) return nullptr;
    return bank->chans[(size_t)chan].get();
}

// DRAIN_BYTES staging of n int16 rows and `cap` ADPCM bytes per slot: [int16 rows][ADPCM bytes per slot][byte count per slot]
size_t tail_bytes_at(size_t n, size_t slots) { return (n * slots * sizeof(int16_t) + 15) / 16 * 16; }
size_t tail_counts_at(size_t n, size_t slots, size_t cap) { return tail_bytes_at(n, slots) + (cap * slots + 15) / 16 * 16; }

// Lists what group g has that is not in the host queues yet: rows [dr_*, last_*) of its audio, demod, IF and S-meter power (as
// out_mask enables them) and, once the feed is complete (`final`), its client-audio bytes and multiplex tap.  Every item
// names, per slot, the client it belongs to now.  Marks the listed outputs delivered.
void drain_items(const owrx_bank* bank, Group* g, bool final, std::vector<DrainItem>& items)
{
    const int S = g->slots;
    std::vector<DrainTo> to((size_t)S, DrainTo{-1, 0, 0, 0});
    for (int s = 0; s < S; s++) {
        const int cid = g->slot_chan[(size_t)s];
        if (cid >= 0) to[(size_t)s] = DrainTo{cid, bank->chans[(size_t)cid]->gen, bank->chans[(size_t)cid]->audio_fmt, 0};
    }
    auto add = [&](DrainKind kind, size_t n, size_t bytes) -> DrainItem& {
        items.push_back(DrainItem{kind});
        DrainItem& it = items.back();
        it.g = g; it.n = n; it.slots = S; it.bytes = (bytes + 15) / 16 * 16; it.to = to;
        return it;
    };
    auto rows = [&](DrainKind kind, int bit, StageBuf& b, int width, size_t last, size_t& dr) {
        if ((bank->out_mask & bit) && last > dr) {
            DrainItem& it = add(kind, last - dr, (last - dr) * (size_t)S * width * sizeof(float));
            it.src = b.rows(b.fill - last + dr); it.buf = &b; it.width = width;
        }
        dr = last;
    };
    rows(DRAIN_AUDIO, OWRX_OUT_AUDIO, g->f3, 1, g->last_audio, g->dr_audio);
    rows(DRAIN_DEMOD, OWRX_OUT_DEMOD, g->f2, 1, g->last_demod, g->dr_demod);
    rows(DRAIN_IF, OWRX_OUT_IF, g->s3, 2, g->last_if, g->dr_if);
    if ((bank->out_mask & OWRX_OUT_POWER) && g->last_blocks > g->dr_blocks) {
        DrainItem& it = add(DRAIN_POWER, g->last_blocks - g->dr_blocks, (g->last_blocks - g->dr_blocks) * (size_t)S * sizeof(float));
        it.src = g->d_power + g->dr_blocks * (size_t)S;
        it.phase = g->sq_block_first + (long long)g->dr_blocks;
    }
    g->dr_blocks = g->last_blocks;
    if (!final || g->dr_final) return;
    g->dr_final = true;
    if (g->any_tail && g->tail_ran && g->last_audio) {
        // rows of the int16 scratch: the feed's audio rows, or more when a resampler produced more
        const size_t n = std::max(g->last_audio, g->rs_rows);
        DrainItem& it = add(DRAIN_BYTES, n, tail_counts_at(n, S, g->tail_cap) + (size_t)S * sizeof(int));
        it.cap = (size_t)g->tail_cap;
        for (int s = 0; s < S; s++) {
            // a resampled slot's count follows from its (L, M, origin), like the kernels' (the same RsCfg)
            const RsCfg& c = g->h_rs[(size_t)s];
            it.to[(size_t)s].n = c.L ? std::min(it.n, (size_t)(rs_outputs(c, g->f3.abs_end) - rs_outputs(c, g->audio_af))) : g->last_audio;
        }
    }
    for (DrainKind kind : {DRAIN_MPX, DRAIN_ATAP}) {
        TapStage& tap = kind == DRAIN_MPX ? g->mpx : g->atap;
        if (!tap.rows || tap.runs.empty()) continue;
        // packed as [F32 runs][S16 runs] of tap.rows each; a run goes to the client it was gathered for, in its format
        DrainItem& it = add(kind, tap.rows, tap.rows * (4 * (size_t)tap.nf + 2 * (size_t)tap.ns));
        it.tap = &tap;
        it.cap = tap.cap;
        it.to.clear();
        const size_t f32 = (size_t)tap.nf * it.n * 4;
        for (const TapRun& r : tap.runs)
            it.to.push_back(DrainTo{r.chan, r.gen, r.fmt, r.fmt == OWRX_MPX_F32 ? (size_t)r.run * it.n * 4 : f32 + (size_t)r.run * it.n * 2});
    }
}

// Stages `items` on `st`: one transpose per row output ([n][slots] rows -> [slots][n], so that a slot's samples are one
// contiguous run), then the D2H copies.  `split`: a split-phase drain, whose copies outlive the call; the next writer of a
// source buffer waits for the transpose that read it (StageBuf::drained), the next gather into a tap region for its copy.
int drain_enqueue(owrx_bank* bank, std::vector<DrainItem>& items, DrainStage& stage, cudaStream_t st, bool split)
{
    // the transposed items first, so that one copy moves them all
    size_t xp = 0;
    for (DrainItem& it : items) if (it.transposed()) { it.off = xp; xp += it.bytes; }
    size_t total = xp;
    for (DrainItem& it : items) if (!it.transposed()) { it.off = total; total += it.bytes; }
    if (!total) return OWRX_OK;
    int rc = stage.reserve(total, xp);
    if (rc != OWRX_OK) return rc;
    for (DrainItem& it : items) {
        Group* g = it.g;
        unsigned char* h = stage.h + it.off;
        const size_t S = (size_t)it.slots;
        if (it.transposed()) {
            const dim3 grid((unsigned)((S + 31) / 32), (unsigned)((it.n + 31) / 32));
            if (it.width == 1) transpose_kernel<float><<<grid, dim3(32, 8), 0, st>>>(it.src, it.slots, it.n, reinterpret_cast<float*>(stage.d + it.off));
            else transpose_kernel<float2><<<grid, dim3(32, 8), 0, st>>>(reinterpret_cast<const float2*>(it.src), it.slots, it.n,
                                                                         reinterpret_cast<float2*>(stage.d + it.off));
            OWRX_LAUNCH_CHECK();
            bank->stats.kernel_launches++;
            if (split && (rc = it.buf->mark_drained(st)) != OWRX_OK) return rc;
        } else if (it.kind == DRAIN_POWER) {
            OWRX_CUDA(cudaMemcpyAsync(h, it.src, it.n * S * sizeof(float), cudaMemcpyDeviceToHost, st));
        } else if (it.kind == DRAIN_BYTES) {
            OWRX_CUDA(cudaMemcpyAsync(h, g->d_tail_s16, it.n * S * sizeof(int16_t), cudaMemcpyDeviceToHost, st));
            OWRX_CUDA(cudaMemcpyAsync(h + tail_bytes_at(it.n, S), g->d_tail_bytes, it.cap * S, cudaMemcpyDeviceToHost, st));
            OWRX_CUDA(cudaMemcpyAsync(h + tail_counts_at(it.n, S, it.cap), g->d_tail_count, S * sizeof(int), cudaMemcpyDeviceToHost, st));
        } else {
            // a tap's runs, at most two copies
            const size_t n = it.n, nf = (size_t)it.tap->nf, ns = (size_t)it.tap->ns;
            const unsigned char* d = it.tap->d[g->cur];
            if (nf) OWRX_CUDA(cudaMemcpy2DAsync(h, n * 4, d, it.cap * 4, n * 4, nf, cudaMemcpyDeviceToHost, st));
            if (ns) OWRX_CUDA(cudaMemcpy2DAsync(h + nf * n * 4, n * 2, d + nf * it.cap * 4, it.cap * 2, n * 2, ns, cudaMemcpyDeviceToHost, st));
            if (split && (rc = it.tap->mark_drained(g->cur, st)) != OWRX_OK) return rc;
        }
    }
    if (xp) OWRX_CUDA(cudaMemcpyAsync(stage.h, stage.d, xp, cudaMemcpyDeviceToHost, st));
    return OWRX_OK;
}

// Pushes staged items into the per-channel queues.  A slot whose client has left, or whose id now belongs to a later client,
// gets nothing; nor does a tap run whose client has changed its tap format since.
void drain_deliver(owrx_bank* bank, const std::vector<DrainItem>& items, const unsigned char* stage)
{
    for (const DrainItem& it : items) {
        const unsigned char* h = stage + it.off;
        const float* f = reinterpret_cast<const float*>(h);
        for (size_t k = 0; k < it.to.size(); k++) {
            const DrainTo& t = it.to[k];
            Chan* ch = t.chan >= 0 && (size_t)t.chan < bank->chans.size() ? bank->chans[(size_t)t.chan].get() : nullptr;
            if (!ch || ch->gen != t.gen) continue;
            switch (it.kind) {
            case DRAIN_AUDIO: case DRAIN_DEMOD: case DRAIN_IF: {
                FQ& q = it.kind == DRAIN_AUDIO ? ch->q_audio : it.kind == DRAIN_DEMOD ? ch->q_demod : ch->q_if;
                q.push(f + k * it.n * it.width, it.n * it.width);
                break;
            }
            case DRAIN_POWER:
                // reportInterval = measurementsPerSec / readingsPerSec = 4 (selector.py:108-109,126)
                for (size_t b = 0; b < it.n; b++)
                    if ((it.phase + (long long)b) % 4 == 0) ch->q_power.push_back(f[b * it.slots + k]);
                break;
            case DRAIN_BYTES:
                if (t.fmt == OWRX_AUDIO_S16) {
                    const int16_t* h16 = reinterpret_cast<const int16_t*>(h);
                    const size_t o = ch->q_bytes.size();
                    ch->q_bytes.resize(o + t.n * 2);
                    int16_t* dst = reinterpret_cast<int16_t*>(ch->q_bytes.data() + o);
                    for (size_t i = 0; i < t.n; i++) dst[i] = h16[i * it.slots + k];
                } else if (t.fmt == OWRX_AUDIO_ADPCM) {
                    const unsigned char* hb = h + tail_bytes_at(it.n, it.slots) + k * it.cap;
                    ch->q_bytes.insert(ch->q_bytes.end(), hb, hb + reinterpret_cast<const int*>(h + tail_counts_at(it.n, it.slots, it.cap))[k]);
                }
                break;
            case DRAIN_MPX: case DRAIN_ATAP: {
                const bool mpx = it.kind == DRAIN_MPX;
                std::vector<unsigned char>& q = mpx ? ch->q_mpx : ch->q_atap;
                if ((mpx ? ch->mpx_fmt : ch->atap_fmt) == t.fmt) q.insert(q.end(), h + t.n, h + t.n + it.n * (t.fmt == OWRX_MPX_F32 ? 4 : 2));
                break;
            }
            }
        }
    }
}

// enqueue, wait, deliver with the synchronous staging on `st` (which already waits for the work that wrote the outputs)
int drain_now(owrx_bank* bank, std::vector<DrainItem>& items, cudaStream_t st)
{
    int rc = drain_enqueue(bank, items, bank->stage, st, false);
    if (rc != OWRX_OK) return rc;
    OWRX_CUDA(cudaStreamSynchronize(st));
    drain_deliver(bank, items, bank->stage.h);
    return OWRX_OK;
}

// every group's outputs of the feed or device block, complete
int drain_final(owrx_bank* bank, cudaStream_t st)
{
    std::vector<DrainItem> items;
    for (auto& g : bank->groups) if (g) drain_items(bank, g.get(), true, items);
    return drain_now(bank, items, st);
}

// `st` waits for everything owrx_bank_process_device has issued, on all three of its streams
int wait_device_path(owrx_bank* bank, cudaStream_t st)
{
    OWRX_CUDA(cudaStreamWaitEvent(st, bank->dev_done, 0));
    OWRX_CUDA(cudaStreamWaitEvent(st, bank->tail_done[0], 0));
    OWRX_CUDA(cudaStreamWaitEvent(st, bank->tail_done[1], 0));
    return OWRX_OK;
}

int pop_queue(FQ& q, float* out, size_t cap, size_t* n, size_t unit)
{
    *n = q.pop(out, cap * unit, unit) / unit;
    return OWRX_OK;
}

}  // namespace

extern "C" {

// deferred-drain mode (owrx_bank_set_deferred_drain): every call that reconfigures the bank first completes the pending feed
static int finish_pending(owrx_bank* bank);

int owrx_bank_create(int device, double input_rate, owrx_bank_t** out)
{
    if (!out) return fail(OWRX_E_INVALID, "out is NULL");
    *out = nullptr;
    if (!(input_rate > 0.0)) return fail(OWRX_E_INVALID, "input_rate must be positive");
    int sm = 0, rc = select_device(device, &sm);
    if (rc != OWRX_OK) return rc;
    owrx_bank* b = new (std::nothrow) owrx_bank();
    if (!b) return fail(OWRX_E_NOMEM, "out of host memory");
    b->device = device; b->sm_count = sm; b->input_rate = input_rate;
    if (const char* m = getenv("OWRX_FIR_MODE")) b->fir_mode = std::max(OWRX_FIR_AUTO, std::min(OWRX_FIR_FASTCONV_TC, atoi(m)));
    b->bp_mode = std::min(b->fir_mode, OWRX_FIR_FASTCONV);
    if (const char* m = getenv("OWRX_TAIL_FUSED")) b->tail_fused = atoi(m) != 0;
    if (const char* m = getenv("OWRX_FC_M")) b->fc_m = atoi(m);
    if (const char* f = getenv("OWRX_FC_TC_FMT")) b->fc_levels = !strcmp(f, "bf16x3") ? 3 : !strcmp(f, "f16x2") ? 2 : 0;
    if (const char* f = getenv("OWRX_FC_TC_FORM")) b->fc_tc_form = atoi(f);
    cudaError_t e = cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&b->copy_stream, cudaStreamNonBlocking);
    // The parallel low-rate stages are a chain of a dozen small dependent launches: on a high-priority stream their CTAs go
    // ahead of the bulk FIR passes of later blocks whenever an SM frees resources (C2 inside the three-stream pipeline: step
    // 0.33 -> 0.30 ms; the forward FFT pass stretches from 0.08 to 0.15 ms but is not the longest stage).  Bit 1 of
    // OWRX_TAIL_PRIORITY does the same for the serial Agc stream (no measurable effect: its CTAs already sit alone on
    // their SMs); 0 restores equal priorities.
    int prio_lo = 0, prio_hi = 0;
    if (e == cudaSuccess) e = cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    static const int tail_prio = getenv("OWRX_TAIL_PRIORITY") ? atoi(getenv("OWRX_TAIL_PRIORITY")) : 1;
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&b->side_stream, cudaStreamNonBlocking, (tail_prio & 1) ? prio_hi : prio_lo);
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&b->serial_stream, cudaStreamNonBlocking, (tail_prio & 2) ? prio_hi : prio_lo);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&b->drain_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->adrain_done, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&b->ctl_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->ptail_done[0], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->ptail_done[1], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreate(&b->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&b->ev1);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->fir_done, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->dev_done, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->tail_done[0], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&b->tail_done[1], cudaEventDisableTiming);
    if (e != cudaSuccess) { owrx_bank_destroy(b); return fail(OWRX_E_CUDA, "stream/event create: %s", cudaGetErrorString(e)); }
    *out = b;
    return OWRX_OK;
}

void owrx_bank_destroy(owrx_bank_t* bank)
{
    if (!bank) return;
    cudaSetDevice(bank->device);
    cudaDeviceSynchronize();
    for (auto& g : bank->groups) if (g) group_release(g.get());
    reap_groups(bank, true);
    if (bank->ctl_stream) cudaStreamDestroy(bank->ctl_stream);
    cudaFree(bank->d_iq[0]); cudaFree(bank->d_iq[1]); cudaFree(bank->d_raw);
    for (cudaEvent_t e : bank->chunk_events) cudaEventDestroy(e);
    for (cudaEvent_t e : bank->fir_events) cudaEventDestroy(e);
    for (cudaEvent_t e : bank->drain_events) cudaEventDestroy(e);
    if (bank->drain_stream) cudaStreamDestroy(bank->drain_stream);
    if (bank->adrain_done) cudaEventDestroy(bank->adrain_done);
    bank->stage.release();
    bank->adrain_stage.release();
    if (bank->fir_done) cudaEventDestroy(bank->fir_done);
    if (bank->dev_done) cudaEventDestroy(bank->dev_done);
    if (bank->tail_done[0]) cudaEventDestroy(bank->tail_done[0]);
    if (bank->tail_done[1]) cudaEventDestroy(bank->tail_done[1]);
    if (bank->copy_stream) cudaStreamDestroy(bank->copy_stream);
    if (bank->side_stream) cudaStreamDestroy(bank->side_stream);
    if (bank->serial_stream) cudaStreamDestroy(bank->serial_stream);
    if (bank->ptail_done[0]) cudaEventDestroy(bank->ptail_done[0]);
    if (bank->ptail_done[1]) cudaEventDestroy(bank->ptail_done[1]);
    if (bank->ev0) cudaEventDestroy(bank->ev0);
    if (bank->ev1) cudaEventDestroy(bank->ev1);
    for (auto& pe : bank->prof_events) { cudaEventDestroy(pe.first); cudaEventDestroy(pe.second); }
    for (auto& t : bank->rs_tabs) cudaFree(t.second.d);
    if (bank->stream) cudaStreamDestroy(bank->stream);
    delete bank;
}

static int add_channel_spec(owrx_bank_t* bank, const owrx_chan_spec_t& sp, int* chan)
{
    std::lock_guard<std::mutex> lk(bank->mu);
    OWRX_CUDA(cudaSetDevice(bank->device));
    if (bank->pending_final) { int rcp = finish_pending(bank); if (rcp != OWRX_OK) return rcp; }
    reap_groups(bank, false);
    int gi = find_group(bank, sp), rc;
    if (gi < 0 && (rc = group_create(bank, sp, &gi)) != OWRX_OK) return rc;
    Group* g = bank->groups[(size_t)gi].get();
    if (std::find(g->slot_chan.begin(), g->slot_chan.end(), -1) == g->slot_chan.end() && (rc = group_grow(bank, g)) != OWRX_OK) return rc;
    std::unique_ptr<Chan> ch(new Chan());
    // ids are handles like file descriptors: the lowest free one is handed out again
    size_t id = 0;
    while (id < bank->chans.size() && bank->chans[id]) id++;
    ch->id = (int)id;
    ch->gen = ++bank->chan_gen;
    ch->spec = sp;
    agc_defaults(ch->cfg, sp.wfm ? OWRX_DEMOD_WFM : OWRX_DEMOD_NONE, OWRX_AGC_SLOW);
    Chan* raw = ch.get();
    if (id == bank->chans.size()) bank->chans.push_back(std::move(ch));
    else bank->chans[id] = std::move(ch);
    if ((rc = place_channel(bank, raw, gi)) != OWRX_OK) return rc;
    *chan = raw->id;
    return OWRX_OK;
}

int owrx_bank_add_channel(owrx_bank_t* bank, double output_rate, int* chan)
{
    if (!bank || !chan) return fail(OWRX_E_INVALID, "NULL argument");
    if (!(output_rate > 0.0)) return fail(OWRX_E_INVALID, "output_rate must be positive");
    return add_channel_spec(bank, spec_from_rates(bank->input_rate, output_rate), chan);
}

int owrx_bank_add_channel_ex(owrx_bank_t* bank, const owrx_chan_spec_t* spec, int* chan)
{
    if (!bank || !chan || !spec) return fail(OWRX_E_INVALID, "NULL argument");
    return add_channel_spec(bank, *spec, chan);
}

int owrx_bank_remove_channel(owrx_bank_t* bank, int chan)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    std::lock_guard<std::mutex> lk(bank->mu);
    Chan* ch = get_chan(bank, chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    if (bank->pending_final) { cudaSetDevice(bank->device); int rcp = finish_pending(bank); if (rcp != OWRX_OK) return rcp; }
    if (ch->group >= 0) {
        Group* g = bank->groups[(size_t)ch->group].get();
        g->slot_chan[(size_t)ch->slot] = -1;
        ChanCfg idle{}; idle.kind = OWRX_DEMOD_NONE; idle.agc_ref = 0.8f; idle.agc_max = 1.f; idle.agc_thr = 0.8f;
        g->h_cfg[(size_t)ch->slot] = idle;
        g->h_bp_en[(size_t)ch->slot] = 0;
        g->h_tail_mode[(size_t)ch->slot] = 0;
        g->h_rs[(size_t)ch->slot] = RsCfg{};
        g->cfg_stale[0] = g->cfg_stale[1] = true;
        g->pend.erase(ch->slot);
        bool live = false;
        for (int cid : g->slot_chan) if (cid >= 0) live = true;
        if (!live) {
            OWRX_CUDA(cudaSetDevice(bank->device));
            int rcr = retire_group(bank, ch->group);
            if (rcr != OWRX_OK) return rcr;
        }
    }
    bank->chans[(size_t)chan].reset();
    return OWRX_OK;
}

int owrx_bank_channel_count(const owrx_bank_t* bank)
{
    if (!bank) return 0;
    int n = 0;
    for (auto& c : bank->chans) if (c) n++;
    return n;
}

int owrx_chan_set_shift_rate(owrx_bank_t* bank, int chan, double rate)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    std::lock_guard<std::mutex> lk(bank->mu);
    Chan* ch = get_chan(bank, chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    if (bank->pending_final) { cudaSetDevice(bank->device); int rcp = finish_pending(bank); if (rcp != OWRX_OK) return rcp; }
    ch->rate = rate;
    return OWRX_OK;
}

int owrx_chan_set_bandpass(owrx_bank_t* bank, int chan, double lo_rate, double hi_rate, int enabled)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    // the filter is designed before the mutex is taken: the DSP thread's next block never waits for a client's trigonometry
    std::vector<float2> designed;
    if (enabled) {
        int Tb = 0, bpP = 0;
        {
            std::lock_guard<std::mutex> lk(bank->mu);
            Chan* ch = get_chan(bank, chan);
            if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
            const Group* g = bank->groups[(size_t)ch->group].get();
            Tb = g->Tb; bpP = g->bpP;
        }
        design_bandpass_stage(designed, Tb, bpP, lo_rate, hi_rate);
    }
    std::lock_guard<std::mutex> lk(bank->mu);
    Chan* ch = get_chan(bank, chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    if (bank->pending_final) { cudaSetDevice(bank->device); int rcp = finish_pending(bank); if (rcp != OWRX_OK) return rcp; }
    OWRX_CUDA(cudaSetDevice(bank->device));
    ch->bp_enabled = enabled != 0; ch->bp_lo = lo_rate; ch->bp_hi = hi_rate;
    return upload_bandpass(bank, ch, &designed);                         // (re-designs under the mutex if the channel changed group meanwhile)
}

int owrx_chan_set_squelch_level(owrx_bank_t* bank, int chan, float level)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    std::lock_guard<std::mutex> lk(bank->mu);
    Chan* ch = get_chan(bank, chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    if (bank->pending_final) { cudaSetDevice(bank->device); int rcp = finish_pending(bank); if (rcp != OWRX_OK) return rcp; }
    ch->cfg.sq_level = level;
    Group* g = bank->groups[(size_t)ch->group].get();
    g->h_cfg[(size_t)ch->slot] = ch->cfg;
    g->cfg_stale[0] = g->cfg_stale[1] = true;
    return OWRX_OK;
}

int owrx_chan_set_demod(owrx_bank_t* bank, int chan, int kind, double audio_rate, double tau, int agc_profile)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    if (kind < OWRX_DEMOD_NFM || kind > OWRX_DEMOD_NONE) return fail(OWRX_E_INVALID, "unknown demodulator %d", kind);
    std::lock_guard<std::mutex> lk(bank->mu);
    Chan* ch = get_chan(bank, chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    if (bank->pending_final) { cudaSetDevice(bank->device); int rcp = finish_pending(bank); if (rcp != OWRX_OK) return rcp; }
    OWRX_CUDA(cudaSetDevice(bank->device));
    Group* g = bank->groups[(size_t)ch->group].get();
    const float level = ch->cfg.sq_level;
    agc_defaults(ch->cfg, kind, agc_profile);
    ch->cfg.sq_level = level;
    ch->agc_initial = agc_initial_gain(kind);
    const bool wfm = kind == OWRX_DEMOD_WFM;
    if (wfm && !(audio_rate > 0.0 && tau > 0.0)) return fail(OWRX_E_INVALID, "WFM needs audio_rate and tau");
    if (!wfm) { ch->mpx_fmt = OWRX_MPX_OFF; ch->q_mpx.clear(); }          // the multiplex tap is a WFm chain's
    if (kind == OWRX_DEMOD_NONE) { ch->atap_fmt = OWRX_MPX_OFF; ch->q_atap.clear(); }   // no demodulator: no audio to tap
    if (kind == OWRX_DEMOD_NONE && ch->rs_in) {                           // no audio: nothing to resample
        ch->rs_in = ch->rs_out = 0;
        ch->rs_dirty = true; g->rs_pending = true;
    }
    owrx_chan_spec_t sp = ch->spec;
    sp.wfm = wfm ? 1 : 0;
    if (wfm) {
        // WFm chain (analog.py:55-67): FractionalDecimator(FLOAT, IF rate / audio rate, prefilter=True) + WfmDeemphasis
        const double if_rate = bank->input_rate / sp.decimation / sp.fraction;
        sp.wfm_decimation = if_rate / audio_rate;
        sp.wfm_audio_rate = (int)audio_rate;
        sp.wfm_tau = tau;
    }
    if (!spec_equal(sp, g->spec)) {
        // move to the matching group (WFM channels keep their own lock-step group)
        int vrc = spec_validate(sp);
        if (vrc != OWRX_OK) return vrc;
        const int old_gi = ch->group, old_slot = ch->slot;
        g->slot_chan[(size_t)old_slot] = -1;
        {
            ChanCfg idle{}; idle.kind = OWRX_DEMOD_NONE; idle.agc_ref = 0.8f; idle.agc_max = 1.f; idle.agc_thr = 0.8f;
            g->h_cfg[(size_t)old_slot] = idle; g->h_bp_en[(size_t)old_slot] = 0; g->h_tail_mode[(size_t)old_slot] = 0;
            g->h_rs[(size_t)old_slot] = RsCfg{};
        }
        g->cfg_stale[0] = g->cfg_stale[1] = true;
        g->pend.erase(old_slot);
        bool live = false;
        for (int cid : g->slot_chan) if (cid >= 0) live = true;
        ch->spec = sp;
        if (!live) { int rcr = retire_group(bank, old_gi); if (rcr != OWRX_OK) return rcr; }
        int gi = find_group(bank, sp), rc;
        if (gi < 0 && (rc = group_create(bank, sp, &gi)) != OWRX_OK) return rc;
        Group* ng = bank->groups[(size_t)gi].get();
        if (std::find(ng->slot_chan.begin(), ng->slot_chan.end(), -1) == ng->slot_chan.end() && (rc = group_grow(bank, ng)) != OWRX_OK) return rc;
        if ((rc = place_channel(bank, ch, gi)) != OWRX_OK) return rc;
        return upload_bandpass(bank, ch);
    }
    // same group: new demodulator chain starts from fresh state (the reference rebuilds the modules) at the next block boundary
    add_patch(g, ch->slot, PATCH_DEMOD | PATCH_AGC_RESET, ch->agc_initial);
    g->h_cfg[(size_t)ch->slot] = ch->cfg;
    g->cfg_stale[0] = g->cfg_stale[1] = true;
    return OWRX_OK;
}

int owrx_chan_set_agc(owrx_bank_t* bank, int chan, int profile, float initial_gain, float max_gain)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    std::lock_guard<std::mutex> lk(bank->mu);
    Chan* ch = get_chan(bank, chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    if (bank->pending_final) { cudaSetDevice(bank->device); int rcp = finish_pending(bank); if (rcp != OWRX_OK) return rcp; }
    OWRX_CUDA(cudaSetDevice(bank->device));
    Group* g = bank->groups[(size_t)ch->group].get();
    ch->cfg.agc_decay = profile == OWRX_AGC_FAST ? 0.001f : 0.0001f;
    ch->cfg.agc_hang_time = profile == OWRX_AGC_FAST ? 200 : 600;
    if (max_gain > 0.f) ch->cfg.agc_max = max_gain;
    if (initial_gain > 0.f) {
        ch->agc_initial = initial_gain;
        add_patch(g, ch->slot, PATCH_AGC_GAIN, initial_gain);
    }
    g->h_cfg[(size_t)ch->slot] = ch->cfg;
    g->cfg_stale[0] = g->cfg_stale[1] = true;
    return OWRX_OK;
}

int owrx_chan_set_audio_format(owrx_bank_t* bank, int chan, int format)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    if (format != OWRX_AUDIO_F32 && format != OWRX_AUDIO_S16 && format != OWRX_AUDIO_ADPCM) return fail(OWRX_E_INVALID, "unknown audio format %d", format);
    std::lock_guard<std::mutex> lk(bank->mu);
    Chan* ch = get_chan(bank, chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    if (bank->pending_final) { cudaSetDevice(bank->device); int rcp = finish_pending(bank); if (rcp != OWRX_OK) return rcp; }
    OWRX_CUDA(cudaSetDevice(bank->device));
    Group* g = bank->groups[(size_t)ch->group].get();
    if (format != ch->audio_fmt) {
        // a new AdpcmEncoder starts from reset state and announces it with a SYNC block
        add_patch(g, ch->slot, PATCH_TAIL, 0.f);
        ch->q_bytes.clear();
    }
    ch->audio_fmt = format;
    g->h_tail_mode[(size_t)ch->slot] = format;
    g->cfg_stale[0] = g->cfg_stale[1] = true;
    return OWRX_OK;
}

int owrx_chan_set_audio_resampler(owrx_bank_t* bank, int chan, int input_rate, int output_rate)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    if (input_rate < 0 || output_rate < 0 || (input_rate == 0) != (output_rate == 0))
        return fail(OWRX_E_INVALID, "resampler rates must both be positive (or both 0): %d -> %d", input_rate, output_rate);
    const bool on = input_rate != output_rate;
    int L = 0, M = 0, K = 0;
    if (on && !design_audio_resampler(input_rate, output_rate, &L, &M, &K, nullptr))
        return fail(OWRX_E_INVALID, "resampler %d -> %d needs more than 65536 taps", input_rate, output_rate);
    std::lock_guard<std::mutex> lk(bank->mu);
    Chan* ch = get_chan(bank, chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    if (on && ch->cfg.kind == OWRX_DEMOD_NONE) return fail(OWRX_E_INVALID, "channel %d has no demodulator: it has no audio to resample", chan);
    if (bank->pending_final) { cudaSetDevice(bank->device); int rcp = finish_pending(bank); if (rcp != OWRX_OK) return rcp; }
    OWRX_CUDA(cudaSetDevice(bank->device));
    if (on && !bank->rs_tabs.count(std::make_pair(L, M))) {
        // first use of this ratio in the bank: design and upload its polyphase table (kept for the bank's lifetime)
        std::vector<float> tab;
        design_audio_resampler(input_rate, output_rate, &L, &M, &K, &tab);
        float* d = nullptr;
        OWRX_CUDA(cudaMalloc((void**)&d, tab.size() * sizeof(float)));
        OWRX_CUDA(cudaMemcpy(d, tab.data(), tab.size() * sizeof(float), cudaMemcpyHostToDevice));
        bank->rs_tabs[std::make_pair(L, M)] = owrx_bank::RsTab{d, K};
    }
    // a new Converter starts from empty history (taking effect at the next block boundary, like every setter)
    ch->rs_in = on ? input_rate : 0;
    ch->rs_out = on ? output_rate : 0;
    ch->rs_dirty = true;
    bank->groups[(size_t)ch->group]->rs_pending = true;
    return OWRX_OK;
}

int owrx_chan_read_bytes(owrx_bank_t* bank, int chan, void* out, size_t cap_bytes, size_t* n)
{
    if (!bank || !out || !n) return fail(OWRX_E_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(bank->mu);
    Chan* ch = get_chan(bank, chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    const size_t take = std::min(cap_bytes, ch->q_bytes.size());
    memcpy(out, ch->q_bytes.data(), take);
    ch->q_bytes.erase(ch->q_bytes.begin(), ch->q_bytes.begin() + (ptrdiff_t)take);
    *n = take;
    return OWRX_OK;
}

int owrx_chan_set_mpx(owrx_bank_t* bank, int chan, int format)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    if (format != OWRX_MPX_OFF && format != OWRX_MPX_F32 && format != OWRX_MPX_S16) return fail(OWRX_E_INVALID, "unknown multiplex format %d", format);
    std::lock_guard<std::mutex> lk(bank->mu);
    Chan* ch = get_chan(bank, chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    if (format != OWRX_MPX_OFF && !ch->spec.wfm) return fail(OWRX_E_INVALID, "channel %d is not a WFM channel: it has no multiplex tap", chan);
    if (bank->pending_final) { cudaSetDevice(bank->device); int rcp = finish_pending(bank); if (rcp != OWRX_OK) return rcp; }
    if (format != ch->mpx_fmt) {
        ch->q_mpx.clear();
        ch->mpx_fmt = format;                        // the group's tap layout is rebuilt at the next block boundary
    }
    return OWRX_OK;
}

// pops whole samples of a tap queue in format `fmt`
static void pop_tap(std::vector<unsigned char>& q, int fmt, void* out, size_t cap_bytes, size_t* n_bytes)
{
    const size_t unit = fmt == OWRX_MPX_S16 ? 2 : 4;
    size_t take = std::min(cap_bytes, q.size());
    take -= take % unit;
    memcpy(out, q.data(), take);
    q.erase(q.begin(), q.begin() + (ptrdiff_t)take);
    *n_bytes = take;
}

int owrx_chan_read_mpx(owrx_bank_t* bank, int chan, void* out, size_t cap_bytes, size_t* n_bytes)
{
    if (!bank || !out || !n_bytes) return fail(OWRX_E_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(bank->mu);
    Chan* ch = get_chan(bank, chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    pop_tap(ch->q_mpx, ch->mpx_fmt, out, cap_bytes, n_bytes);
    return OWRX_OK;
}

int owrx_chan_set_audio_tap(owrx_bank_t* bank, int chan, int format)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    if (format != OWRX_MPX_OFF && format != OWRX_MPX_F32 && format != OWRX_MPX_S16) return fail(OWRX_E_INVALID, "unknown audio tap format %d", format);
    std::lock_guard<std::mutex> lk(bank->mu);
    Chan* ch = get_chan(bank, chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    if (format != OWRX_MPX_OFF && ch->cfg.kind == OWRX_DEMOD_NONE) return fail(OWRX_E_INVALID, "channel %d has no demodulator: it has no audio to tap", chan);
    if (bank->pending_final) { cudaSetDevice(bank->device); int rcp = finish_pending(bank); if (rcp != OWRX_OK) return rcp; }
    if (format != ch->atap_fmt) {
        ch->q_atap.clear();
        ch->atap_fmt = format;                       // the group's tap layout is rebuilt at the next block boundary
    }
    return OWRX_OK;
}

int owrx_chan_read_audio_tap(owrx_bank_t* bank, int chan, void* out, size_t cap_bytes, size_t* n_bytes)
{
    if (!bank || !out || !n_bytes) return fail(OWRX_E_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(bank->mu);
    Chan* ch = get_chan(bank, chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    pop_tap(ch->q_atap, ch->atap_fmt, out, cap_bytes, n_bytes);
    return OWRX_OK;
}

int owrx_chan_read_message(owrx_bank_t* bank, int chan, int type_byte, void* out, size_t cap_bytes, size_t* n)
{
    if (!bank || !out || !n) return fail(OWRX_E_INVALID, "bad argument");
    if (type_byte != 0x02 && type_byte != 0x04) return fail(OWRX_E_INVALID, "message type must be 0x02 (audio) or 0x04 (HD audio)");
    std::lock_guard<std::mutex> lk(bank->mu);
    Chan* ch = get_chan(bank, chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    *n = 0;
    if (ch->q_bytes.empty() || cap_bytes < 2) return OWRX_OK;
    const size_t take = std::min(cap_bytes - 1, ch->q_bytes.size());
    uint8_t* o = (uint8_t*)out;
    o[0] = (uint8_t)type_byte;                                 // write_dsp_data / write_hd_audio (owrx/connection.py:477-481)
    memcpy(o + 1, ch->q_bytes.data(), take);
    ch->q_bytes.erase(ch->q_bytes.begin(), ch->q_bytes.begin() + (ptrdiff_t)take);
    *n = take + 1;
    return OWRX_OK;
}

int owrx_bank_set_outputs(owrx_bank_t* bank, int mask)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    std::lock_guard<std::mutex> lk(bank->mu);
    if (bank->pending_final) { cudaSetDevice(bank->device); int rcp = finish_pending(bank); if (rcp != OWRX_OK) return rcp; }
    bank->out_mask = mask;
    return OWRX_OK;
}

// deferred-drain mode: move the last outputs of the previous feed into the host queues (waits for that feed's kernels)
static int finish_pending(owrx_bank* bank)
{
    if (!bank->pending_final) return OWRX_OK;
    int rc = drain_final(bank, bank->stream);
    if (rc != OWRX_OK) return rc;
    bank->pending_final = false;
    return OWRX_OK;
}

// Host path.  The block is uploaded in chunks on a copy stream; the K3 pass of chunk c runs while chunk
// c+1 is still crossing PCIe.  The low-rate stages run once over everything the chunks produced.
int owrx_bank_feed(owrx_bank_t* bank, const float* iq, size_t n_samples)
{
    return owrx_bank_feed_fmt(bank, iq, n_samples, OWRX_IQ_CF32, 1.0f);
}

int owrx_bank_feed_fmt(owrx_bank_t* bank, const void* iq_raw, size_t n_samples, int format, float gain)
{
    if (!bank || (!iq_raw && n_samples)) return fail(OWRX_E_INVALID, "NULL argument");
    const size_t in_bytes = iq_format_bytes(format);
    if (!in_bytes) return fail(OWRX_E_INVALID, "unknown IQ format %d", format);
    const float* iq = static_cast<const float*>(iq_raw);             // OWRX_IQ_CF32 view
    std::lock_guard<std::mutex> lk(bank->mu);
    OWRX_CUDA(cudaSetDevice(bank->device));
    cudaStream_t st = bank->stream;
    static const bool trace = getenv("OWRX_TRACE") != nullptr;
    const auto T0 = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (trace) fprintf(stderr, "[owrx feed] %-18s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - T0).count());
    };
    reap_groups(bank, false);
    bool any = false;
    for (auto& g : bank->groups) if (g) any = true;
    if (!any) return OWRX_OK;                         // nobody listening: samples are dropped like an unread ring
    if (n_samples) (host_is_pinned(iq_raw) ? bank->stats.h2d_pinned_bytes : bank->stats.h2d_pageable_bytes) += n_samples * in_bytes;
    const size_t need = bank->iq_fill + n_samples;
    int rc;
    if (need > bank->iq_cap || (format != OWRX_IQ_CF32 && n_samples * in_bytes > bank->raw_cap)) {
        if ((rc = finish_pending(bank)) != OWRX_OK) return rc;       // reallocation below synchronises: nothing to overlap with
    }
    if (need > bank->iq_cap) {
        const size_t cap = std::max(need, bank->iq_cap * 2);
        for (int b = 0; b < 2; b++) {
            float2* nb = nullptr;
            OWRX_CUDA(cudaMalloc((void**)&nb, cap * sizeof(float2)));
            if (b == bank->iq_cur && bank->iq_fill)
                OWRX_CUDA(cudaMemcpyAsync(nb, bank->d_iq[b], bank->iq_fill * sizeof(float2), cudaMemcpyDeviceToDevice, st));
            OWRX_CUDA(cudaStreamSynchronize(st));
            cudaFree(bank->d_iq[b]);
            bank->d_iq[b] = nb;
        }
        bank->iq_cap = cap;
    }
    float2* buf = bank->d_iq[bank->iq_cur];
    if (format != OWRX_IQ_CF32 && n_samples * in_bytes > bank->raw_cap) {
        OWRX_CUDA(cudaStreamSynchronize(bank->copy_stream));
        cudaFree(bank->d_raw); bank->d_raw = nullptr; bank->raw_cap = 0;
        OWRX_CUDA(cudaMalloc((void**)&bank->d_raw, n_samples * in_bytes));
        bank->raw_cap = n_samples * in_bytes;
    }
    OWRX_CUDA(cudaEventRecord(bank->ev0, st));
    // chunks of 2 M samples: the work left after the last H2D chunk (its FIR, low-rate stages and drain) stays short while a
    // chunk still spans 11+ overlap-save blocks; small feeds are a single chunk
    // (raw formats: the same 16 MB of PCIe traffic per chunk, i.e. 4 M int16 / 8 M uint8 samples)
    static const size_t chunk_f32 = (size_t)1 << (getenv("OWRX_FEED_CHUNK_LOG2") ? std::max(16, std::min(26, atoi(getenv("OWRX_FEED_CHUNK_LOG2")))) : 21);
    const size_t chunk = chunk_f32 * (sizeof(float2) / in_bytes);
    const size_t n_chunks = std::max<size_t>(1, (n_samples + chunk - 1) / chunk);
    while (bank->chunk_events.size() < n_chunks) {
        cudaEvent_t e;
        OWRX_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        bank->chunk_events.push_back(e);
    }
    // The uploads need no ordering against earlier device work: they fill [iq_fill, iq_fill + n) of the current buffer, the
    // previous feed's carry copy (on `st`) fills [0, iq_fill) of the same buffer, and the last kernels that READ this buffer
    // belong to the feed before the previous one, which has been synchronised (finish_pending / the synchronous return) before
    // this call.  So this feed's chunks queue right behind the previous feed's on the copy stream: PCIe never idles.
    for (size_t c = 0; c < n_chunks; c++) {
        const size_t o = c * chunk, len = std::min(chunk, n_samples - o);
        if (len && format == OWRX_IQ_CF32) {
            OWRX_CUDA(cudaMemcpyAsync(buf + bank->iq_fill + o, iq + 2 * o, len * sizeof(float2), cudaMemcpyHostToDevice, bank->copy_stream));
        } else if (len) {
            // raw samples cross PCIe as they are; Convert (+ Gain) runs on the copy stream behind each chunk's upload
            unsigned char* d_raw = bank->d_raw + o * in_bytes;
            OWRX_CUDA(cudaMemcpyAsync(d_raw, static_cast<const unsigned char*>(iq_raw) + o * in_bytes, len * in_bytes, cudaMemcpyHostToDevice,
                                      bank->copy_stream));
            int rcc = iq_convert_launch(format, d_raw, buf + bank->iq_fill + o, len, gain, bank->copy_stream);
            if (rcc != OWRX_OK) return rcc;
            bank->stats.kernel_launches++;
        }
        OWRX_CUDA(cudaEventRecord(bank->chunk_events[c], bank->copy_stream));
    }
    // deferred drain: the previous feed's last outputs go to the host queues now, while this feed's chunks cross PCIe
    if ((rc = finish_pending(bank)) != OWRX_OK) return rc;
    const size_t fill0 = bank->iq_fill;
    // with several chunks the low-rate stages of chunk c run on the side stream beside the K3 pass of chunk c+1
    const bool overlap = n_chunks > 1;
    cudaStream_t tails = overlap ? bank->side_stream : st;
    bank->reserve_sm = overlap;
    if (overlap) {
        OWRX_CUDA(cudaEventRecord(bank->fir_done, st));
        OWRX_CUDA(cudaStreamWaitEvent(tails, bank->fir_done, 0));
    }
    for (auto& gp : bank->groups) {
        Group* g = gp.get();
        if (!g) continue;
        const size_t rows = (fill0 + n_samples - g->in_off) / (size_t)g->D + 1;
        if ((rc = group_begin_feed(bank, g, rows, st, tails, tails, (int)(bank->feeds & 1))) != OWRX_OK) return rc;
    }
    while (bank->drain_events.size() < n_chunks) {
        cudaEvent_t e;
        OWRX_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        bank->drain_events.push_back(e);
    }
    std::vector<DrainItem> chunk_items;               // outputs of the previous chunk, drained while the GPU works on the next
    while (bank->fir_events.size() < n_chunks) {
        cudaEvent_t e;
        OWRX_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        bank->fir_events.push_back(e);
    }
    for (size_t c = 0; c < n_chunks; c++) {
        OWRX_CUDA(cudaStreamWaitEvent(st, bank->chunk_events[c], 0));
        const size_t avail = fill0 + std::min(n_samples, (c + 1) * chunk);
        for (auto& gp : bank->groups) {
            Group* g = gp.get();
            if (!g) continue;
            size_t consumed = 0;
            if ((rc = group_fir(bank, g, buf + g->in_off, avail - g->in_off, &consumed, st)) != OWRX_OK) return rc;
            g->in_off += consumed;
            int live = 0;
            for (int cid : g->slot_chan) if (cid >= 0) live++;
            bank->stats.channel_samples += (uint64_t)consumed * (uint64_t)live;
        }
        if (overlap) {
            OWRX_CUDA(cudaEventRecord(bank->fir_events[c], st));
            OWRX_CUDA(cudaStreamWaitEvent(tails, bank->fir_events[c], 0));
        }
        for (auto& gp : bank->groups) {
            Group* g = gp.get();
            if (!g) continue;
            if ((rc = group_tail(bank, g, tails)) != OWRX_OK) return rc;
            if ((rc = group_tail_serial(bank, g, tails)) != OWRX_OK) return rc;
        }
        if (overlap) {
            // outputs of chunk c are complete once `tails` gets here; while the GPU works on chunk c+1 the host copies the
            // outputs of chunk c-1 into the per-channel queues (drain stream: waits for that chunk only)
            OWRX_CUDA(cudaEventRecord(bank->drain_events[c], tails));
            // (deferred drain: the host does not wait inside a feed at all — every output of the block moves at the start of
            // the next feed, so that feed's uploads queue right behind this one's and PCIe never idles)
            if (!bank->deferred) {
                if (!chunk_items.empty()) {
                    OWRX_CUDA(cudaStreamWaitEvent(bank->drain_stream, bank->drain_events[c - 1], 0));
                    if ((rc = drain_now(bank, chunk_items, bank->drain_stream)) != OWRX_OK) return rc;
                    chunk_items.clear();
                }
                // the last chunk's outputs go with the feed's final drain
                if (c + 1 < n_chunks)
                    for (auto& gp : bank->groups) if (gp) drain_items(bank, gp.get(), false, chunk_items);
            }
        }
    }
    bank->reserve_sm = false;
    // drop consumed wideband samples: the carry moves to the other buffer right behind the last FirDecimate pass on `st`
    bank->iq_fill += n_samples;
    size_t min_off = bank->iq_fill;
    for (auto& gp : bank->groups) if (gp) min_off = std::min(min_off, gp->in_off);
    if (min_off > 0) {
        const size_t tail = bank->iq_fill - min_off;
        if (tail) OWRX_CUDA(cudaMemcpyAsync(bank->d_iq[bank->iq_cur ^ 1], buf + min_off, tail * sizeof(float2), cudaMemcpyDeviceToDevice, st));
        bank->iq_cur ^= 1;
        bank->iq_fill = tail;
        for (auto& gp : bank->groups) if (gp) gp->in_off -= min_off;
    }
    if (overlap) {
        OWRX_CUDA(cudaEventRecord(bank->fir_done, tails));
        OWRX_CUDA(cudaStreamWaitEvent(st, bank->fir_done, 0));
    }
    OWRX_CUDA(cudaEventRecord(bank->ev1, st));
    lap("launched");
    bank->stats.input_samples += n_samples;
    bank->feeds++;
    if (bank->deferred) {
        bank->pending_final = true;                   // drained by the next feed (behind its uploads) or owrx_bank_flush
        return OWRX_OK;
    }
    if (trace) { cudaStreamSynchronize(st); lap("gpu done"); }
    if ((rc = drain_final(bank, st)) != OWRX_OK) return rc;
    lap("drained");
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, bank->ev0, bank->ev1) == cudaSuccess) bank->stats.device_ms += ms;
    return OWRX_OK;
}

int owrx_bank_set_deferred_drain(owrx_bank_t* bank, int enable)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    std::lock_guard<std::mutex> lk(bank->mu);
    OWRX_CUDA(cudaSetDevice(bank->device));
    int rc = finish_pending(bank);
    bank->deferred = enable != 0;
    return rc;
}

int owrx_bank_flush(owrx_bank_t* bank)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    std::lock_guard<std::mutex> lk(bank->mu);
    OWRX_CUDA(cudaSetDevice(bank->device));
    return finish_pending(bank);
}

// Device-resident path.  With owrx_bank_set_pipelined(bank, 1) every stage after FirDecimate of block i runs on the
// bank's side stream beside the Shift + FirDecimate pass of block i+1 on the caller's stream; owrx_bank_join makes a
// stream wait for everything issued so far.
int owrx_bank_process_device(owrx_bank_t* bank, const void* iq_dev, size_t n_samples, void* stream)
{
    if (!bank || !iq_dev) return fail(OWRX_E_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(bank->mu);
    if (bank->pending_final) { cudaSetDevice(bank->device); int rcp = finish_pending(bank); if (rcp != OWRX_OK) return rcp; }
    OWRX_CUDA(cudaSetDevice(bank->device));
    cudaStream_t sa = stream ? (cudaStream_t)stream : bank->stream;
    cudaStream_t sb = bank->pipelined ? bank->side_stream : sa;
    cudaStream_t sc = bank->pipelined ? bank->serial_stream : sa;
    const int par = (int)(bank->calls & 1);
    reap_groups(bank, false);
    int rc = OWRX_OK;
    if (bank->pipelined) {
        // s1 ping-pong: this block's FirDecimate writes the buffer the parallel stages of two blocks ago were reading
        OWRX_CUDA(cudaStreamWaitEvent(sa, bank->ptail_done[par], 0));
        // f2 ping-pong: this block's parallel stages write the buffer the Agc of two blocks ago was reading
        OWRX_CUDA(cudaStreamWaitEvent(sb, bank->tail_done[par], 0));
    }
    bank->reserve_sm = bank->pipelined;
    for (auto& gp : bank->groups) {
        Group* g = gp.get();
        if (!g) continue;
        size_t consumed = 0;
        // previous block's outputs are dropped; histories stay
        // pipelined: every stage after FirDecimate (rolls of their history buffers included) lives on the side stream
        if ((rc = group_begin_feed(bank, g, n_samples / (size_t)g->D + 1, sa, sb, sc, par)) != OWRX_OK) return rc;
        // the output buffers this block writes (the rolls above have just selected them) may still be read by a split-phase
        // drain of an earlier block that used the same buffer: both low-rate streams wait for that transpose (none: no-op)
        for (const StageBuf* sbuf : {&g->f3, &g->f2, &g->s3}) {
            if ((rc = sbuf->wait_drained(sb)) != OWRX_OK) return rc;
            if (sc != sb && (rc = sbuf->wait_drained(sc)) != OWRX_OK) return rc;
        }
        // groups consume whole decimation steps: a group that got further than the slowest one in the previous block starts
        // `dev_lead` samples into this one (the caller presents [carry | new] from owrx_bank_last_consumed on)
        const size_t lead = std::min(g->dev_lead, n_samples);
        if ((rc = group_fir(bank, g, (const float2*)iq_dev + lead, n_samples - lead, &consumed, sa)) != OWRX_OK) return rc;
        g->dev_lead = lead + consumed;               // rebased on the slowest group below
        int live = 0;
        for (int cid : g->slot_chan) if (cid >= 0) live++;
        bank->stats.channel_samples += (uint64_t)consumed * (uint64_t)live;
    }
    {
        size_t cmin = n_samples;
        for (auto& gp : bank->groups) if (gp) cmin = std::min(cmin, gp->dev_lead);
        for (auto& gp : bank->groups) if (gp) gp->dev_lead -= cmin;
        bank->last_consumed = cmin;
    }
    if (bank->pipelined) {
        OWRX_CUDA(cudaEventRecord(bank->fir_done, sa));
        OWRX_CUDA(cudaStreamWaitEvent(sb, bank->fir_done, 0));
    }
    if ((rc = prof_mark(bank, OWRX_PROF_TAIL, sb, true)) != OWRX_OK) return rc;
    for (auto& gp : bank->groups) {
        Group* g = gp.get();
        if (!g) continue;
        if ((rc = group_tail(bank, g, sb)) != OWRX_OK) return rc;
    }
    if ((rc = prof_mark(bank, OWRX_PROF_TAIL, sb, false)) != OWRX_OK) return rc;
    // three-deep pipeline: FirDecimate of block i+2 (sa) | parallel low-rate stages of block i+1 (sb) | the sample-serial
    // Agc / audio tail of block i (sc).  Ping-pong stage buffers keep consecutive blocks apart; a buffer is reused two
    // blocks later: s1 after ptail_done[par] (awaited by sa), f2 after tail_done[par] (awaited by sb).
    if (bank->pipelined) {
        OWRX_CUDA(cudaEventRecord(bank->ptail_done[par], sb));
        OWRX_CUDA(cudaStreamWaitEvent(sc, bank->ptail_done[par], 0));
    }
    for (auto& gp : bank->groups) {
        Group* g = gp.get();
        if (g && (rc = group_tail_serial(bank, g, sc)) != OWRX_OK) return rc;
    }
    bank->reserve_sm = false;
    if (bank->pipelined) OWRX_CUDA(cudaEventRecord(bank->tail_done[par], sc));   // awaited by the call after next
    OWRX_CUDA(cudaEventRecord(bank->dev_done, sa));
    bank->calls++;
    bank->stats.input_samples += n_samples;
    return rc;
}

// Device path + host outputs: copy what the last owrx_bank_process_device call produced into the per-channel
// host queues (the same queues owrx_bank_feed fills), so owrx_chan_read_* can pop it.
int owrx_bank_drain(owrx_bank_t* bank)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    std::lock_guard<std::mutex> lk(bank->mu);
    if (bank->pending_final) { cudaSetDevice(bank->device); int rcp = finish_pending(bank); if (rcp != OWRX_OK) return rcp; }
    OWRX_CUDA(cudaSetDevice(bank->device));
    int rc = wait_device_path(bank, bank->stream);
    return rc != OWRX_OK ? rc : drain_final(bank, bank->stream);
}

// Split-phase drain (streaming hosts of the device path): _begin enqueues, on the drain stream and with staging of its own, the
// transposes and D2H copies of what the last owrx_bank_process_device call produced, behind that block's kernels; the caller
// may issue the NEXT block before _end, which waits for the copies and hands the samples to the per-channel queues.  The stage
// buffers are double-buffered, so the next block does not touch what is being drained; whichever later block writes such a
// buffer again waits for the transpose that read it (StageBuf::drained), and the next gather into a tap region for its copy
// (TapStage::drained).  S-meter power reports and client-audio bytes are read from scratch the next block overwrites: with
// either enabled, _begin completes the drain at once.
int owrx_bank_drain_begin(owrx_bank_t* bank)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    std::lock_guard<std::mutex> lk(bank->mu);
    if (bank->adrain_pending) return fail(OWRX_E_INVALID, "owrx_bank_drain_begin: the previous split-phase drain has not been ended");
    OWRX_CUDA(cudaSetDevice(bank->device));
    if (bank->pending_final) { int rcp = finish_pending(bank); if (rcp != OWRX_OK) return rcp; }
    if (bank->calls == 0) return OWRX_OK;
    std::vector<DrainItem> items;
    for (auto& g : bank->groups) if (g) drain_items(bank, g.get(), true, items);
    bool now = (bank->out_mask & OWRX_OUT_POWER) != 0;
    for (const DrainItem& it : items) if (it.kind == DRAIN_BYTES) now = true;
    int rc;
    if (now) {
        if ((rc = wait_device_path(bank, bank->stream)) != OWRX_OK) return rc;
        return drain_now(bank, items, bank->stream);
    }
    if (items.empty()) return OWRX_OK;
    cudaStream_t ds = bank->drain_stream;
    if ((rc = wait_device_path(bank, ds)) != OWRX_OK || (rc = drain_enqueue(bank, items, bank->adrain_stage, ds, true)) != OWRX_OK)
        return rc;
    OWRX_CUDA(cudaEventRecord(bank->adrain_done, ds));
    bank->adrain_items = std::move(items);
    bank->adrain_pending = true;
    return OWRX_OK;
}

int owrx_bank_drain_end(owrx_bank_t* bank)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    std::lock_guard<std::mutex> lk(bank->mu);
    if (!bank->adrain_pending) return OWRX_OK;
    OWRX_CUDA(cudaSetDevice(bank->device));
    OWRX_CUDA(cudaEventSynchronize(bank->adrain_done));
    bank->adrain_pending = false;
    drain_deliver(bank, bank->adrain_items, bank->adrain_stage.h);
    bank->adrain_items.clear();
    return OWRX_OK;
}

int owrx_bank_set_pipelined(owrx_bank_t* bank, int enable)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    std::lock_guard<std::mutex> lk(bank->mu);
    OWRX_CUDA(cudaSetDevice(bank->device));
    OWRX_CUDA(cudaDeviceSynchronize());
    bank->pipelined = enable != 0;
    return OWRX_OK;
}

int owrx_bank_join(owrx_bank_t* bank, void* stream)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    std::lock_guard<std::mutex> lk(bank->mu);
    OWRX_CUDA(cudaSetDevice(bank->device));
    cudaStream_t sa = stream ? (cudaStream_t)stream : bank->stream;
    OWRX_CUDA(cudaStreamWaitEvent(sa, bank->tail_done[0], 0));
    OWRX_CUDA(cudaStreamWaitEvent(sa, bank->tail_done[1], 0));
    return OWRX_OK;
}

int owrx_bank_last_consumed(const owrx_bank_t* bank, size_t* n_samples)
{
    if (!bank || !n_samples) return fail(OWRX_E_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(const_cast<owrx_bank_t*>(bank)->mu);
    *n_samples = bank->last_consumed;
    return OWRX_OK;
}

int owrx_bank_last_audio_count(const owrx_bank_t* bank, int chan, size_t* n)
{
    if (!bank || !n) return fail(OWRX_E_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(const_cast<owrx_bank_t*>(bank)->mu);
    Chan* ch = get_chan(const_cast<owrx_bank_t*>(bank), chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    *n = bank->groups[(size_t)ch->group]->last_audio;
    return OWRX_OK;
}

int owrx_bank_last_audio_device(const owrx_bank_t* bank, int chan, const float** base, size_t* stride, size_t* slot)
{
    if (!bank || !base || !stride || !slot) return fail(OWRX_E_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(const_cast<owrx_bank_t*>(bank)->mu);
    Chan* ch = get_chan(const_cast<owrx_bank_t*>(bank), chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    const Group* g = bank->groups[(size_t)ch->group].get();
    *base = g->f3.rows(g->f3.fill - g->last_audio);
    *stride = (size_t)g->slots;
    *slot = (size_t)ch->slot;
    return OWRX_OK;
}

int owrx_chan_read_audio(owrx_bank_t* bank, int chan, float* out, size_t cap_samples, size_t* n)
{
    if (!bank || !out || !n) return fail(OWRX_E_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(bank->mu);
    Chan* ch = get_chan(bank, chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    return pop_queue(ch->q_audio, out, cap_samples, n, 1);
}

int owrx_bank_read_audio_all(owrx_bank_t* bank, const int* chans, int n_chans, float* out, size_t cap_samples, size_t* counts)
{
    if (!bank || !chans || n_chans < 0 || !out || !counts) return fail(OWRX_E_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(bank->mu);
    for (int i = 0; i < n_chans; i++)
        if (!get_chan(bank, chans[i])) return fail(OWRX_E_INVALID, "unknown channel %d", chans[i]);
    for (int i = 0; i < n_chans; i++) {
        Chan* ch = get_chan(bank, chans[i]);
        int rc = pop_queue(ch->q_audio, out + (size_t)i * cap_samples, cap_samples, &counts[i], 1);
        if (rc != OWRX_OK) return rc;
    }
    return OWRX_OK;
}

int owrx_chan_read_demod(owrx_bank_t* bank, int chan, float* out, size_t cap_samples, size_t* n)
{
    if (!bank || !out || !n) return fail(OWRX_E_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(bank->mu);
    Chan* ch = get_chan(bank, chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    return pop_queue(ch->q_demod, out, cap_samples, n, 1);
}

int owrx_chan_read_if(owrx_bank_t* bank, int chan, float* out_iq, size_t cap_samples, size_t* n)
{
    if (!bank || !out_iq || !n) return fail(OWRX_E_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(bank->mu);
    Chan* ch = get_chan(bank, chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    return pop_queue(ch->q_if, out_iq, cap_samples, n, 2);
}

int owrx_chan_read_power(owrx_bank_t* bank, int chan, float* out, size_t cap, size_t* n)
{
    if (!bank || !out || !n) return fail(OWRX_E_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(bank->mu);
    Chan* ch = get_chan(bank, chan);
    if (!ch) return fail(OWRX_E_INVALID, "no such channel %d", chan);
    return pop_queue(ch->q_power, out, cap, n, 1);
}

int owrx_bank_profile(owrx_bank_t* bank, int enable)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    std::lock_guard<std::mutex> lk(bank->mu);
    bank->profile = enable != 0;
    return OWRX_OK;
}

static int prof_collect(owrx_bank_t* bank)
{
    for (size_t i = 0; i < bank->prof_used; i++) {
        OWRX_CUDA(cudaEventSynchronize(bank->prof_events[i].second));
        float ms = 0.f;
        OWRX_CUDA(cudaEventElapsedTime(&ms, bank->prof_events[i].first, bank->prof_events[i].second));
        const int tag = bank->prof_tags[i];
        bank->prof_ms[tag] += ms;
        bank->prof_launches[tag]++;
    }
    bank->prof_used = 0;
    return OWRX_OK;
}

int owrx_bank_profile_read(owrx_bank_t* bank, double* k3_ms, uint64_t* k3_launches, int reset)
{
    if (!bank || !k3_ms || !k3_launches) return fail(OWRX_E_INVALID, "NULL argument");
    double ms[OWRX_PROF_KINDS];
    uint64_t n[OWRX_PROF_KINDS];
    int rc = owrx_bank_profile_read_ex(bank, ms, n, reset);
    if (rc != OWRX_OK) return rc;
    // the dominant kernel of whichever form ran: direct K3, or the fast-convolution contraction
    const int k = n[OWRX_PROF_FC_CONTRACT] ? OWRX_PROF_FC_CONTRACT : OWRX_PROF_K3_DIRECT;
    *k3_ms = ms[k];
    *k3_launches = n[k];
    return OWRX_OK;
}

int owrx_bank_profile_read_ex(owrx_bank_t* bank, double* ms, uint64_t* launches, int reset)
{
    if (!bank || !ms || !launches) return fail(OWRX_E_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(bank->mu);
    OWRX_CUDA(cudaSetDevice(bank->device));
    int rc = prof_collect(bank);
    if (rc != OWRX_OK) return rc;
    for (int k = 0; k < OWRX_PROF_KINDS; k++) {
        ms[k] = bank->prof_ms[k];
        launches[k] = bank->prof_launches[k];
        if (reset) { bank->prof_ms[k] = 0.0; bank->prof_launches[k] = 0; }
    }
    return OWRX_OK;
}

int owrx_bank_set_fir_mode(owrx_bank_t* bank, int mode)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    if (mode < OWRX_FIR_AUTO || mode > OWRX_FIR_FASTCONV_TC) return fail(OWRX_E_INVALID, "unknown FIR mode %d", mode);
    std::lock_guard<std::mutex> lk(bank->mu);
    bank->fir_mode = mode;
    bank->bp_mode = mode;
    return OWRX_OK;
}

int owrx_bank_fir_form(const owrx_bank_t* bank)
{
    if (!bank) return fail(OWRX_E_INVALID, "NULL bank");
    return bank->fir_form_used;
}

int owrx_bank_get_stats(const owrx_bank_t* bank, owrx_bank_stats_t* st)
{
    if (!bank || !st) return fail(OWRX_E_INVALID, "bad argument");
    *st = bank->stats;
    return OWRX_OK;
}

}  // extern "C"
