/*
 * owrx_b200.h — C ABI of libowrx_b200.so: the B200-native (sm_100a) DSP hot path of OpenWebRX+.
 *
 * This is the drop-in boundary.  The reference reaches this arithmetic through the CPython
 * extension `pycsdr` (un-vendored: luarvique/pycsdr@master wrapping luarvique/csdr@master; pinned
 * only as python3-csdr >= 0.18.36 in debian/control:22).  Each entry point below names the pycsdr
 * module(s) / reference call site it replaces.  The repo's `pycsdr/` package binds these symbols
 * with ctypes so that the reference's unmodified csdr.chain classes run on top (INTEGRATION.md).
 *
 * Conventions: plain C types only; every function returns 0 on success or a negative OWRX_E_* code
 * (owrx_last_error() gives a thread-local message); no exceptions cross the ABI; output buffers are
 * caller-owned; objects are internally synchronised (setters may race with feed/read).
 * IQ is interleaved float32 (re,im) = pycsdr Format.COMPLEX_FLOAT.  There is NO CPU fallback: every
 * create call fails with OWRX_E_CUDA when no sm_100-class device is usable.
 */
#ifndef OWRX_B200_H
#define OWRX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OWRX_OK            0
#define OWRX_E_INVALID    -1   /* bad argument            -> ValueError in the Python shim */
#define OWRX_E_CUDA       -2   /* CUDA runtime failure    -> RuntimeError                  */
#define OWRX_E_NOMEM      -3   /* allocation failure      -> MemoryError                   */
#define OWRX_E_OVERFLOW   -4   /* caller buffer too small -> BufferError                   */
#define OWRX_E_STATE      -5   /* object stopped / wrong state                             */

const char* owrx_last_error(void);
const char* owrx_version(void);
/* number of kernels this library has launched in this process (bench.py "gpu_launches") */
uint64_t owrx_launch_count(void);
int owrx_device_count(int* n);

/* Page-locked host memory for the IQ ingress ring (SURVEY 8f-4 / a19: the reference's TcpSource writes the connector's TCP
 * stream into the source Buffer, owrx/source/__init__.py:307-330; here that Buffer's storage is a cudaHostAlloc'd ring, so
 * recv() lands where the copy engine reads and no pageable bounce copy remains between the socket and HBM).
 * Portable across devices.  owrx_host_is_pinned: 1 if `p` lies in page-locked memory known to CUDA, 0 if not. */
int owrx_pinned_alloc(size_t bytes, void** out);
void owrx_pinned_free(void* p);
int owrx_host_is_pinned(const void* p);

/* Wideband IQ ingress formats (SURVEY 8f-4).  Sources that do not deliver complex float32 are converted by the reference on
 * the CPU — Chain([Convert(Format.COMPLEX_SHORT, Format.COMPLEX_FLOAT), Gain(Format.COMPLEX_FLOAT, 5.0)]),
 * owrx/source/fifi_sdr.py:27-28 via owrx/source/direct.py:59-71; owrx_*_feed_fmt takes the raw samples (interleaved I, Q)
 * and does that Convert (+ Gain) on the GPU:  CS16: x / 32767;  CU8: x / 127.5 - 1;  then * gain. */
#define OWRX_IQ_CF32 0   /* complex float32, 8 bytes per sample (what owrx_wf_feed / owrx_bank_feed take) */
#define OWRX_IQ_CS16 1   /* complex int16 little-endian, 4 bytes per sample */
#define OWRX_IQ_CU8  2   /* complex uint8 offset binary (rtl_sdr raw), 2 bytes per sample */

/* Multi-GPU IQ hop (SURVEY 8e; the cross-GPU form of every client reading the one source ring, owrx/dsp.py:835-837,
 * owrx/source/__init__.py:307-330): copies n_bytes from src_dev (this GPU) to multicast_dst, an NVSwitch multicast (NVLS)
 * address that maps the same offset of a buffer on every GPU of the group — one pass of multimem.st stores replicates the
 * block into all of them.  The multicast mapping is created by the host (e.g. torch.distributed symmetric memory); the
 * caller orders a cross-GPU barrier after this call on `stream` before the block is read.  16-byte aligned pointers and size. */
int owrx_iq_multicast_store(const void* src_dev, void* multicast_dst, size_t n_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Waterfall — replaces the pycsdr chain  Fft -> LogPower|LogAveragePower -> FftSwap -> [FftAdpcm]
 * built by FftChain (csdr/chain/fft.py:25-49) and driven by SpectrumThread (owrx/fft.py:40-73).
 * ---------------------------------------------------------------------------------------------- */
typedef struct owrx_wf owrx_wf_t;

#define OWRX_COMPRESSION_NONE  0   /* float32 dB lines, 4*N bytes   (FftSwap output)            */
#define OWRX_COMPRESSION_ADPCM 1   /* IMA-ADPCM lines, (N+10)/2 B   (FftAdpcm, csdr/chain/fft.py:44) */

/* Fft(size=, every_n_samples=) + LogAveragePower(add_db=, fft_size=, avg_number=) [avg==0: LogPower(add_db=)]
 * + FftSwap(fft_size=) + optional FftAdpcm(fft_size=).  fft_size: power of two, 256..65536. */
int owrx_wf_create(int device, int fft_size, int every_n_samples, int avg_number, float add_db,
                   int compression, owrx_wf_t** out);
void owrx_wf_destroy(owrx_wf_t* wf);
int owrx_wf_feed_fmt(owrx_wf_t* wf, const void* iq, size_t n_samples, int format, float gain);   /* owrx_wf_feed for OWRX_IQ_* input */
/* Websocket framing of the outputs (SURVEY 8f-2; owrx/connection.py:473-481): one message = a 1-byte type prefix + payload.
 * owrx_wf_read_message pops ONE waterfall line as 0x01 + line (write_spectrum_data); owrx_chan_read_message pops the
 * queued client-audio bytes (owrx_chan_set_audio_format S16 / ADPCM) as type_byte + data with type_byte 0x02
 * (write_dsp_data) or 0x04 (write_hd_audio).  *n = 0 when nothing is queued.  The S-meter message is JSON built by the
 * host from owrx_chan_read_power (write_s_meter_level, :483-489). */
int owrx_wf_read_message(owrx_wf_t* wf, void* out, size_t cap_bytes, size_t* n_bytes);
int owrx_wf_set_every_n_samples(owrx_wf_t* wf, int every_n_samples);   /* Fft.setEveryNSamples, csdr/chain/fft.py:55 */
int owrx_wf_set_avg_number(owrx_wf_t* wf, int avg_number);             /* FftAverager.setFftAverages, csdr/chain/fft.py:12-16 */
int owrx_wf_set_compression(owrx_wf_t* wf, int compression);           /* FftChain.setCompression, csdr/chain/fft.py:87-96 */
/* Spectral-subtraction noise filter on the averaged line power (BASELINE config 4).  NOT a reference module: OpenWebRX+
 * has no waterfall noise filter (its NoiseFilter is audio-only, csdr/chain/clientaudio.py:13-14) — spec-defined stage after
 * power averaging (SURVEY 8d C4), off by default.  Per bin, across lines:
 *   N = first line ? P : min(P, N * (1 + growth));   P' = max(P - alpha * N, beta * P);   dB = 10 log10(P') + corrections */
int owrx_wf_set_noise_filter(owrx_wf_t* wf, int enable, float alpha, float beta, float growth);
size_t owrx_wf_line_bytes(const owrx_wf_t* wf);
/* host-path ingress bytes by source memory kind (see owrx_bank_stats_t) */
int owrx_wf_get_h2d_bytes(const owrx_wf_t* wf, uint64_t* pinned_bytes, uint64_t* pageable_bytes);

/* Streaming host path (what the pycsdr shim calls): append n_samples of interleaved IQ from HOST
 * memory; every completed line is computed on the GPU and queued. */
int owrx_wf_feed(owrx_wf_t* wf, const float* iq, size_t n_samples);
/* Pop up to cap_bytes of whole queued lines into out; *n_bytes = bytes written (multiple of line_bytes). */
int owrx_wf_read(owrx_wf_t* wf, void* out, size_t cap_bytes, size_t* n_bytes);

/* Device-resident batch path: iq_dev holds n_samples complex float32 on the object's device.
 * Computes every whole line of that record (line l uses frames l*avg..l*avg+avg-1, frame f starts at
 * sample f*every_n) into out_dev (device; line_bytes each).  db_dev / s16_dev may be NULL; when given
 * they receive the swapped float32 dB lines (N each) / the quantised int16 lines (N+10 each).
 * stream: a cudaStream_t; NULL selects the object's own non-blocking stream (so the legacy default
 * stream cannot be named here: pass a created stream to order against other work).  Asynchronous. */
int owrx_wf_process_device(owrx_wf_t* wf, const void* iq_dev, size_t n_samples, void* out_dev,
                           size_t out_cap_bytes, void* db_dev, void* s16_dev, size_t* n_lines, void* stream);
/* Pipelined device path: the FftAdpcm encoder of batch i (latency-bound: one warp per 32 lines) runs on a
 * high-priority side stream beside the FFT pass of batch i+1.  owrx_wf_join makes `stream` wait for it. */
int owrx_wf_set_pipelined(owrx_wf_t* wf, int enable);
int owrx_wf_join(owrx_wf_t* wf, void* stream);
/* number of whole lines a record of n_samples yields with the current parameters */
size_t owrx_wf_lines_for(const owrx_wf_t* wf, size_t n_samples);

/* Stand-alone FftAdpcm encoder stage on the GPU: s16_dev = n_lines x (fft_size+10) int16 (already
 * quantised and padded), out_dev = n_lines x (fft_size+10)/2 bytes.  State resets per line
 * (SURVEY A.5; decoder: htdocs/openwebrx.js:1124-1128). */
int owrx_fft_adpcm_encode_device(int device, const void* s16_dev, int fft_size, size_t n_lines, void* out_dev, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Channel bank — replaces, for every client attached to one wideband source, the pycsdr chain
 *   Shift -> FirDecimate -> [FractionalDecimator] -> [Bandpass] -> Squelch      (Selector,
 *   csdr/chain/selector.py:89-214) followed by the analog demodulator chain
 *   AmDemod/DcBlock/Agc | FmDemod/Limit/NfmDeemphasis/Agc | FmDemod/Limit/FractionalDecimator/
 *   WfmDeemphasis | RealPart/Agc   (csdr/chain/analog.py:11-127),
 * batched: all channels of a bank share ONE pass over the wideband IQ block (owrx/dsp.py:835-837
 * attaches one reader per client to the same source ring in the reference).
 * ---------------------------------------------------------------------------------------------- */
typedef struct owrx_bank owrx_bank_t;

#define OWRX_DEMOD_NFM  0   /* NFm: csdr/chain/analog.py:34-52  */
#define OWRX_DEMOD_AM   1   /* Am:  csdr/chain/analog.py:11-21  */
#define OWRX_DEMOD_SSB  2   /* Ssb: csdr/chain/analog.py:119-127 */
#define OWRX_DEMOD_WFM  3   /* WFm: csdr/chain/analog.py:55-116 */
#define OWRX_DEMOD_NONE 4   /* selector output only (IF samples) */

#define OWRX_AGC_SLOW 0
#define OWRX_AGC_FAST 1

int owrx_bank_create(int device, double input_rate, owrx_bank_t** out);
void owrx_bank_destroy(owrx_bank_t* bank);

/* Threading and ordering of the control calls below (the reference calls the setters from websocket threads while the DSP
 * thread pumps the chain: csdr/chain/selector.py:132-166, owrx/dsp.py:96-148,835-839).  Every owrx_bank_add_channel* /
 * owrx_bank_remove_channel / owrx_chan_set_* call is thread-safe against the feed calls and only RECORDS the change: it takes
 * effect at the next block boundary (the next owrx_bank_feed* / owrx_bank_process_device), applied on the device in stream
 * order, so blocks already in flight are not touched and no call synchronises the device (the one exception: adding the 65th,
 * 129th, ... client of a parameter class re-lays that class's tables).  A new or re-moded client starts from fresh module state
 * (empty filter histories, reset Agc / codec), as the reference's freshly built pycsdr modules do; a retune keeps the NCO phase
 * continuous.  Channel ids are handles: the lowest free id is handed out again after owrx_bank_remove_channel. */

/* Selector(inputRate, outputRate): csdr/chain/selector.py:89-113 (Decimator math :21-26,37-51). */
int owrx_bank_add_channel(owrx_bank_t* bank, double output_rate, int* chan);

/* The same channel described by the exact arguments the reference's chain classes pass to the
 * pycsdr module constructors (what the pycsdr shim sees; SURVEY Appendix D.2):
 *   FirDecimate(decimation, transition, cutoff)                    csdr/chain/selector.py:29
 *   FractionalDecimator(Format.COMPLEX_FLOAT, fraction)            csdr/chain/selector.py:33   (1.0 = absent)
 *   Bandpass(transition=bp_transition, use_fft=True)               csdr/chain/selector.py:115-117
 *   Squelch(Format.COMPLEX_FLOAT, length=squelch_length, decimation=5, hangLength=2*length, ...)  :119-130
 *   NfmDeemphasis(deemph_rate)                                     csdr/chain/analog.py:43
 *   FractionalDecimator(Format.FLOAT, wfm_decimation, prefilter=True), WfmDeemphasis(wfm_audio_rate, wfm_tau)
 *                                                                  csdr/chain/analog.py:66-67  (wfm != 0 only) */
typedef struct {
    int    decimation;
    double transition;
    double cutoff;
    double fraction;
    double bp_transition;
    int    squelch_length;
    int    deemph_rate;
    int    wfm;
    double wfm_decimation;
    int    wfm_audio_rate;
    double wfm_tau;
} owrx_chan_spec_t;
int owrx_bank_add_channel_ex(owrx_bank_t* bank, const owrx_chan_spec_t* spec, int* chan);
/* Agc.setProfile / setInitialGain / setMaxGain (csdr/chain/analog.py:13-15,37-39,121-122); gains <= 0 keep the current value */
int owrx_chan_set_agc(owrx_bank_t* bank, int chan, int profile, float initial_gain, float max_gain);
int owrx_bank_remove_channel(owrx_bank_t* bank, int chan);
int owrx_bank_channel_count(const owrx_bank_t* bank);
/* Shift.setRate(rate), rate = -offset/inputRate: csdr/chain/selector.py:138-140 */
int owrx_chan_set_shift_rate(owrx_bank_t* bank, int chan, double rate);
/* Bandpass.setBandpass(lo, hi) in units of the selector output rate; enabled=0 removes the stage:
 * csdr/chain/selector.py:149-166 */
int owrx_chan_set_bandpass(owrx_bank_t* bank, int chan, double lo_rate, double hi_rate, int enabled);
/* Squelch.setSquelchLevel(linear): csdr/chain/selector.py:145-147; default 0 = always open */
int owrx_chan_set_squelch_level(owrx_bank_t* bank, int chan, float level);
/* demodulator chain selection (DspManager.setDemodulator, owrx/dsp.py:654-680).
 * audio_rate/tau only for WFM; agc_profile OWRX_AGC_*; initial_gain/max_gain <= 0 pick the
 * reference's per-mode values (analog.py:15,39). */
int owrx_chan_set_demod(owrx_bank_t* bank, int chan, int kind, double audio_rate, double tau, int agc_profile);

/* Streaming host path: one wideband block from HOST memory, shared by every channel. */
int owrx_bank_feed(owrx_bank_t* bank, const float* iq, size_t n_samples);
/* Streaming mode.  By default owrx_bank_feed returns when the block's outputs are in the host queues.  With deferred drain
 * enabled a feed only enqueues its work (uploads, kernels) and returns; the block's outputs reach the queues at the start of
 * the NEXT feed — after that feed's uploads have been queued behind this one's, so PCIe never idles and the kernel tail,
 * D2H and queue hand-over of block i run under the upload of block i+1 — or when owrx_bank_flush is called.  Outputs,
 * state and order are identical to the synchronous mode (tests/test_gpu_selector.py::test_deferred_drain_...).
 * The host buffer passed to a feed must stay valid until the next feed / flush returns.  Calls that reconfigure the bank
 * (add / remove channel, owrx_chan_set_*) complete a pending feed first. */
int owrx_bank_set_deferred_drain(owrx_bank_t* bank, int enable);
int owrx_bank_flush(owrx_bank_t* bank);
/* the same for raw OWRX_IQ_CS16 / OWRX_IQ_CU8 samples (Convert + Gain on the GPU, half / a quarter of the PCIe bytes) */
int owrx_bank_feed_fmt(owrx_bank_t* bank, const void* iq, size_t n_samples, int format, float gain);
/* Pop queued outputs of one channel (float32 audio after AGC / pre-AGC demod / complex IF). */
int owrx_chan_read_audio(owrx_bank_t* bank, int chan, float* out, size_t cap_samples, size_t* n);
/* the same pop for many channels in one call (what a fan-out thread serving every websocket of a source does,
 * owrx/dsp.py:863-870 per client): channel chans[i] -> out[i * cap_samples ...], counts[i] samples */
int owrx_bank_read_audio_all(owrx_bank_t* bank, const int* chans, int n_chans, float* out, size_t cap_samples, size_t* counts);
int owrx_chan_read_demod(owrx_bank_t* bank, int chan, float* out, size_t cap_samples, size_t* n);
int owrx_chan_read_if(owrx_bank_t* bank, int chan, float* out_iq, size_t cap_samples, size_t* n);
int owrx_chan_read_power(owrx_bank_t* bank, int chan, float* out, size_t cap, size_t* n);
/* Client audio tail (SURVEY 8f-1), run on the GPU after the AGC:
 *   OWRX_AUDIO_F32   none (float32 audio via owrx_chan_read_audio)
 *   OWRX_AUDIO_S16   Convert(Format.FLOAT, Format.SHORT)                      csdr/chain/clientaudio.py:12
 *   OWRX_AUDIO_ADPCM Convert + AdpcmEncoder(sync=True)                        csdr/chain/clientaudio.py:34
 * S16 / ADPCM bytes are popped with owrx_chan_read_bytes (little-endian int16, or the SYNC-framed stream
 * the browser decodes: htdocs/lib/AudioEngine.js:449-491). */
#define OWRX_AUDIO_F32   0
#define OWRX_AUDIO_S16   1
#define OWRX_AUDIO_ADPCM 2
int owrx_chan_set_audio_format(owrx_bank_t* bank, int chan, int format);
/* Client-audio resampler.  When the client's audio rate differs from the demodulator's, the reference's Converter is
 * AudioResampler(inputRate, clientRate) -> Limit -> Convert(FLOAT, SHORT) [-> AdpcmEncoder(sync=True)]
 * (csdr/chain/clientaudio.py:6-19,34).  owrx_chan_set_audio_resampler puts AudioResampler + Limit in front of this channel's
 * S16 / ADPCM bytes; owrx_chan_read_audio / _demod and the multiplex tap stay at the demodulator rate.  The resampler is
 * SPEC-DEFINED (the reference's libsamplerate is not reproduced, see DESIGN.md): with out/in = L/M reduced, a polyphase
 * Kaiser-windowed sinc (96 dB stop band, cutoff 0.45 * min(in, out)) evaluated causally, so that after n input samples exactly
 * ceil(n * L / M) output samples exist; then Limit clamps to +-1.  Rates are positive integers; 0, 0 or equal rates remove
 * it.  OWRX_E_INVALID for a ratio needing more than 65536 taps or a channel without a demodulator (OWRX_DEMOD_NONE).  Like
 * every setter it takes effect at the next block boundary; setting or changing it starts it from empty history and leaves
 * the selector, demodulator and Agc state alone.  The ratio is per channel: a channel keeps its group. */
int owrx_chan_set_audio_resampler(owrx_bank_t* bank, int chan, int input_rate, int output_rate);
int owrx_chan_read_bytes(owrx_bank_t* bank, int chan, void* out, size_t cap_bytes, size_t* n);
/* the same bytes as one websocket message: type_byte (0x02 audio / 0x04 HD audio) + data; see owrx_wf_read_message */
int owrx_chan_read_message(owrx_bank_t* bank, int chan, int type_byte, void* out, size_t cap_bytes, size_t* n);
/* which optional outputs are materialised for the host (bitmask of OWRX_OUT_*; default AUDIO) */
#define OWRX_OUT_AUDIO 1
#define OWRX_OUT_DEMOD 2
#define OWRX_OUT_IF    4
#define OWRX_OUT_POWER 8
int owrx_bank_set_outputs(owrx_bank_t* bank, int mask);
/* WFM multiplex tap.  The reference's WFm chain writes its Limit output (FmDemod + Limit at the IF rate, before the audio
 * FractionalDecimator) into a tap buffer of its own, metaTapBuffer (csdr/chain/analog.py:62,73-76); the RDS path reads it
 * through Convert(Format.FLOAT, Format.SHORT) into redsea.  owrx_chan_set_mpx delivers that signal per channel:
 *   OWRX_MPX_F32  the limited discriminator output, float32 (what metaTapBuffer carries)
 *   OWRX_MPX_S16  the same after Convert(FLOAT, SHORT): int16 little-endian, x * 32767 truncated toward zero
 * WFM channels only (OWRX_E_INVALID otherwise).  Like every setter it takes effect at the next block boundary; a format change
 * discards queued samples of the old format, and re-moding the channel away from WFM turns the tap off.  Every drain path
 * (owrx_bank_feed*, deferred drain, owrx_bank_drain, owrx_bank_drain_begin / _end) queues the samples, in order;
 * owrx_chan_read_mpx pops up to cap_bytes of whole samples.  A channel id handed out again never receives samples of the
 * client that held it before. */
#define OWRX_MPX_OFF 0   /* tap formats: the multiplex tap and the audio tap below use this one set of codes */
#define OWRX_MPX_F32 1
#define OWRX_MPX_S16 2
int owrx_chan_set_mpx(owrx_bank_t* bank, int chan, int format);
int owrx_chan_read_mpx(owrx_bank_t* bank, int chan, void* out, size_t cap_bytes, size_t* n_bytes);
/* Demodulated-audio tap.  The reference's secondary demodulators (the digital-mode decoders: FT8 and the other WSJT modes, JS8,
 * packet, ...) read the Buffer the primary demodulator's last stage writes (Agc, or WfmDeemphasis for WFM), beside the
 * client-audio Converter; a WSJT-style decoder reads it through Convert(Format.FLOAT, Format.SHORT).  owrx_chan_set_audio_tap
 * delivers that signal per channel, at the DEMODULATOR rate (before any client-audio resampler, whatever the client-audio
 * format and whether OWRX_OUT_AUDIO is set; squelch-closed blocks come out as zeros, as the audio does), in the tap formats:
 *   OWRX_MPX_F32  float32, the samples owrx_chan_read_audio pops
 *   OWRX_MPX_S16  the same after Convert(FLOAT, SHORT): int16 little-endian, x * 32767 truncated toward zero, clamped to
 *                 [-32768, 32767]
 * OWRX_E_INVALID for a channel without a demodulator (OWRX_DEMOD_NONE); re-moding a channel to none turns the tap off, a
 * change between demodulators keeps it.  Like every setter it takes effect at the next block boundary; a format change
 * discards queued samples of the old format.  Every drain path (owrx_bank_feed*, deferred drain, owrx_bank_drain,
 * owrx_bank_drain_begin / _end) queues the samples, in order; the split-phase drain delivers them asynchronously, like the
 * multiplex tap.  owrx_chan_read_audio_tap pops up to cap_bytes of whole samples.  A channel id handed out again never
 * receives samples of the client that held it before. */
int owrx_chan_set_audio_tap(owrx_bank_t* bank, int chan, int format);
int owrx_chan_read_audio_tap(owrx_bank_t* bank, int chan, void* out, size_t cap_bytes, size_t* n_bytes);

/* Device-resident batch path (bench / embedding): process one wideband block that already lives
 * in device memory; outputs stay on the device and are NOT queued for the host.
 * Stream contract — [carry | new]: FirDecimate consumes whole decimation steps, so a call uses only the first
 * ((n - T) / D + 1) * D samples of the block (T taps, D decimation; nothing if n < T) and keeps NO copy of the rest.  A caller
 * that streams consecutive blocks presents the next block starting at sample owrx_bank_last_consumed() of this one (the
 * unconsumed tail followed by the new samples); the NCO phase and every stage history carry over exactly as in
 * owrx_bank_feed, which does this carry internally.  With several decimation classes in one bank the reported count is the
 * slowest group's; groups that got further skip their lead in the next block. */
int owrx_bank_process_device(owrx_bank_t* bank, const void* iq_dev, size_t n_samples, void* stream);
/* samples of the last owrx_bank_process_device block that every channel is done with (see the stream contract above) */
int owrx_bank_last_consumed(const owrx_bank_t* bank, size_t* n_samples);
/* Pipelined device path: the low-rate stages of block i run on the bank's side stream while the K3 pass of
 * block i+1 runs on the caller's stream.  owrx_bank_join makes `stream` wait for everything issued so far. */
int owrx_bank_set_pipelined(owrx_bank_t* bank, int enable);
int owrx_bank_join(owrx_bank_t* bank, void* stream);
/* Copy the outputs of the last owrx_bank_process_device call into the per-channel host queues (D2H), so that
 * owrx_chan_read_* pops them exactly as after owrx_bank_feed.  Synchronous. */
int owrx_bank_drain(owrx_bank_t* bank);
/* Split-phase form for hosts that stream blocks through the device path: _begin enqueues the D2H of the last
 * owrx_bank_process_device block behind that block's kernels and returns; the caller may issue the NEXT
 * owrx_bank_process_device before _end, which waits for the copies and fills the queues exactly as owrx_bank_drain would
 * have.  One drain in flight at a time (_begin before the previous _end is OWRX_E_INVALID); _end without _begin is a
 * no-op.  When S-meter power reports (OWRX_OUT_POWER) or a client-audio format are enabled, _begin drains synchronously.
 * The multiplex and audio taps (owrx_chan_set_mpx, owrx_chan_set_audio_tap) go asynchronously like the other outputs.  Audio, demod and IF follow the tap's
 * rule: a channel id handed out again between _begin and _end never receives samples of the client that held it before. */
int owrx_bank_drain_begin(owrx_bank_t* bank);
int owrx_bank_drain_end(owrx_bank_t* bank);
/* samples of audio produced per channel by the last owrx_bank_process_device call */
int owrx_bank_last_audio_count(const owrx_bank_t* bank, int chan, size_t* n);
/* device pointer + layout of the last block's audio: element (k, slot) at base[k*stride + slot] */
int owrx_bank_last_audio_device(const owrx_bank_t* bank, int chan, const float** base, size_t* stride, size_t* slot);

/* per-bank statistics since creation */
typedef struct {
    uint64_t input_samples;     /* wideband samples consumed                 */
    uint64_t channel_samples;   /* sum over channels of wideband samples     */
    uint64_t kernel_launches;
    double   device_ms;         /* CUDA-event time of the host-path feeds    */
    uint64_t h2d_pinned_bytes;   /* host-path feeds whose source was page-locked memory (DMA straight from the ring)   */
    uint64_t h2d_pageable_bytes; /* ... and whose source was pageable memory (the driver stages it through a bounce buffer) */
} owrx_bank_stats_t;
int owrx_bank_get_stats(const owrx_bank_t* bank, owrx_bank_stats_t* st);

/* Optional per-kernel timing of the dominant kernel (K3: NCO mix + FIR decimation): when enabled a
 * CUDA event pair brackets every K3 launch on the launching stream; owrx_bank_profile_read waits for
 * the recorded events and returns the accumulated device time and launch count. */
int owrx_bank_profile(owrx_bank_t* bank, int enable);
int owrx_bank_profile_read(owrx_bank_t* bank, double* k3_ms, uint64_t* k3_launches, int reset);
/* per kernel kind: ms[OWRX_PROF_KINDS], launches[OWRX_PROF_KINDS] */
#define OWRX_PROF_K3_DIRECT   0   /* fir_decimate_kernel: direct-form NCO mix + polyphase FIR                 */
#define OWRX_PROF_FC_FORWARD  1   /* fc_forward_kernel: shared per-branch forward FFTs                        */
#define OWRX_PROF_FC_CONTRACT 2   /* fc_contract_kernel: per-channel spectral contraction over the branches   */
#define OWRX_PROF_FC_INVERSE  3   /* fc_inverse_kernel: per-channel inverse FFT + post-rotation               */
#define OWRX_PROF_TAIL        4   /* every parallel stage between FirDecimate and the Agc (one bracket per block)  */
#define OWRX_PROF_AGC         5   /* agc_kernel: the sample-serial Agc                                        */
#define OWRX_PROF_RESAMPLE    6   /* audio_resample_kernel: the client-audio resampler                        */
#define OWRX_PROF_TAP         7   /* tap_gather_kernel: the multiplex and audio taps' gathers                 */
#define OWRX_PROF_KINDS       8
int owrx_bank_profile_read_ex(owrx_bank_t* bank, double* ms, uint64_t* launches, int reset);

/* How Shift + FirDecimate (csdr/chain/selector.py:29,95) is evaluated.  All forms compute the same sums
 * (float32 rounding differs at the 1e-6 level):
 *   OWRX_FIR_DIRECT    direct-form polyphase FIR, 2T/D FMA per input sample per channel (K3)
 *   OWRX_FIR_FASTCONV  polyphase fast convolution: one shared forward FFT pass + a per-channel spectral contraction,
 *                      ~4.5 FMA per input sample per channel (K3F); needs decimation >= 8
 *   OWRX_FIR_FASTCONV_TC  the same fast convolution with the spectral contraction on the tensor cores (tcgen05): every
 *                      float32 operand is carried as three bf16 terms and six partial products are accumulated in FP32
 *   OWRX_FIR_AUTO      (default) direct for feeds that yield < 64 outputs per channel, else fast convolution — on the
 *                      tensor cores when a pass holds enough overlap-save blocks (> ~21 at 64 slots, > ~18 at 128), on the FP32 pipe below that */
#define OWRX_FIR_AUTO        0
#define OWRX_FIR_DIRECT      1
#define OWRX_FIR_FASTCONV    2
#define OWRX_FIR_FASTCONV_TC 3
int owrx_bank_set_fir_mode(owrx_bank_t* bank, int mode);
/* the form the latest Shift + FirDecimate pass used (OWRX_FIR_DIRECT / _FASTCONV / _FASTCONV_TC; 0 before any pass) */
int owrx_bank_fir_form(const owrx_bank_t* bank);

#ifdef __cplusplus
}
#endif
#endif
