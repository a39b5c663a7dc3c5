// selector_kernels.cuh — K3/K4/K5: batched Selector front end + analog demodulators on sm_100a.
//
// Replaces, for all channels of one decimator group at once, the per-client pycsdr chains
//   Shift -> FirDecimate -> [FractionalDecimator] -> [Bandpass] -> Squelch   (csdr/chain/selector.py:89-130)
//   -> AmDemod/DcBlock | FmDemod/Limit/NfmDeemphasis | RealPart | FmDemod/Limit/FractionalDecimator/
//      WfmDeemphasis -> Agc                                                    (csdr/chain/analog.py:11-127)
// Arithmetic spec: SURVEY.md Appendix A.6-A.11.
//
// Data layout: every low-rate stream is "channel-minor": element (time i, slot s) lives at
// base[i * slots + s], so a warp's 32 lanes = 32 adjacent channel slots -> fully coalesced, and the
// sample-serial recurrences (AGC, IIR, squelch hang) run one channel per lane.
#pragma once
#include "common.cuh"
#include "adpcm.cuh"

namespace owrx {

// ------------------------------------------------------------------------------------------------
// K3: NCO mix + polyphase FIR decimation, direct form, FP32-FMA bound.
//   y_c[k] = sum_{t<T} x[kD+t] * e^{j 2 pi (ph_c + rate_c (kD+t+1))} * h[t]
// Polyphase view (SURVEY Appendix E2): t = pD + r.  A thread owns CN=2 channels (lane <-> channel
// pair) and 28 rolling accumulators per channel (one per polyphase branch p = output k = j-p of the
// input block j it is streaming).  Each rotated sample is used for 28 branch FMAs x 2 (re,im); the
// 28 taps h[pD+r] of one r come from shared memory as 7 broadcast LDS.128.  Warps split the r-range
// of a block; their partial sums meet in shared memory once per block.
// ------------------------------------------------------------------------------------------------
constexpr int K3_NW = 12;        // warps per CTA (3 per scheduler)
constexpr int K3_CN = 2;         // channels per lane
constexpr int K3_PP = 28;        // polyphase branches per pass (padded, multiple of 4)
constexpr int K3_RBMAX = 896;    // max samples of one block (r-range) staged per CTA
constexpr int K3_CG = 32 * K3_CN;   // channels per CTA

struct K3Params {
    const float2* iq;        // sample 0 of output 0 of this launch
    long long n_lim;         // samples readable from iq
    const float* taps;       // [nseg][D][28]: taps[(ts*D + r)*28 + p'] = h[(ts*28+p')*D + r] (0 beyond T)
    const double* ch_rate;   // per group slot: Shift rate (turns / sample)
    const double* ch_phase;  // per group slot: phase (turns) at iq[-1]
    const float2* ch_w;      // per group slot: e^{j 2 pi rate}
    float2* partial;         // [nparts = nseg*nrs][n_k][slots]: complete outputs and range-tail partial sums
    float2* side;            // [nparts][n_ranges][27][slots]: range-head partial sums (outputs owned by the previous range)
    int D, nseg, nrs, RB, JB, n_blocks, n_k, slots;
};

__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gsrc)
{
    unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(d), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::); }

// K3 itself lives in its own translation unit (k3_fir.cu): it is compiled with `-Xptxas -O1`, because the
// default ptxas scheduler rotates its FFMA2 loop and pays ~24 register copies per sample for it.
int launch_fir_decimate(const K3Params& p, dim3 grid, size_t smem, cudaStream_t st);

#ifndef OWRX_K3_ONLY

// K3b: sum the tap-segment / r-split partials and the range-head partial sums into the FirDecimate
// output stream s1[k][slot].
__global__ void __launch_bounds__(256)
fir_reduce_kernel(const float2* __restrict__ partial, const float2* __restrict__ side, int nparts, int n_ranges, int JB, int n_k,
                  int slots, float2* __restrict__ out)
{
    const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t total = (size_t)n_k * slots;
    if (gid >= total) return;
    const int k = (int)(gid / slots), s = (int)(gid % slots);
    float2 acc = make_float2(0.f, 0.f);
    for (int q = 0; q < nparts; q++) {
        const float2 v = partial[(size_t)q * total + gid];
        acc.x += v.x; acc.y += v.y;
    }
    // is k one of the 27 outputs just below a range start?  range = ceil-ish((k + 27) / JB)
    const int range = (k + (K3_PP - 1)) / JB;
    const int h = k - (range * JB - (K3_PP - 1));
    if (range >= 1 && range < n_ranges && h >= 0 && h < K3_PP - 1) {
        for (int q = 0; q < nparts; q++) {
            const float2 v = side[(((size_t)q * n_ranges + range) * (K3_PP - 1) + h) * slots + s];
            acc.x += v.x; acc.y += v.y;
        }
    }
    out[gid] = acc;
}

// ------------------------------------------------------------------------------------------------
// 12-point Lagrange coefficients (SURVEY A.8): nodes x_i = i-5 relative to ih, evaluated at -d.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void lagrange12(float d, float* c)
{
    const float xe = -d;
#pragma unroll
    for (int i = 0; i < 12; i++) {
        float num = 1.0f, den = 1.0f;
#pragma unroll
        for (int j = 0; j < 12; j++)
            if (j != i) { num *= xe - (float)(j - 5); den *= (float)(i - j); }
        c[i] = num / den;
    }
}

// FractionalDecimator(Format.COMPLEX_FLOAT, rate): out[m] for m_abs = m0 + m, where = 5 + m_abs*rate.
// in: rows of `in_slots` complex, row 0 = absolute index in_abs0; slot map gives the column.
__global__ void __launch_bounds__(128)
fracdec_cf_kernel(const float2* __restrict__ in, long long in_abs0, int in_slots, const int* __restrict__ slot_map,
                  double rate, long long m0, int n_out, int slots, float2* __restrict__ out)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    const int m = blockIdx.y * blockDim.y + threadIdx.y;
    if (s >= slots || m >= n_out) return;
    const double where = 5.0 + (double)(m0 + m) * rate;
    const double ihd = ceil(where);
    float c[12];
    lagrange12((float)(ihd - where), c);
    const int col = slot_map ? slot_map[s] : s;
    const float2* x = in + ((long long)ihd - 5 - in_abs0) * in_slots + col;
    float re = 0.f, im = 0.f;
#pragma unroll
    for (int i = 0; i < 12; i++) {
        const float2 v = x[(size_t)i * in_slots];
        re += c[i] * v.x; im += c[i] * v.y;
    }
    out[(size_t)m * slots + s] = make_float2(re, im);
}

// Bandpass: y[i] = sum_t h_s[t] x[i-t] (causal, zero history = zero rows before the stream start) — the linear
// convolution the reference's FFT overlap-add computes (SURVEY A.9).  taps: [T][slots] complex, per channel;
// enabled[s]==0 passes the sample through.  Register-blocked direct form: a thread owns BP_RB consecutive outputs
// of one channel (lane <-> channel, so tap and sample loads are coalesced) and slides a 2*BP_RB-1 sample window
// through registers: per BP_RB taps it loads BP_RB taps + BP_RB samples and issues 4*BP_RB^2 FMAs.
constexpr int BP_RB = 8;
// packed FP32 helpers (fma.rn.f32x2 -> FFMA2; a (x, x) pair assembles to the scalar-broadcast operand form)
typedef unsigned long long bp_f32x2;
__device__ __forceinline__ bp_f32x2 bp_pk2(float lo, float hi)
{
    bp_f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void bp_upk2(bp_f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ void bp_ffma2(bp_f32x2& c, bp_f32x2 a, bp_f32x2 b) { asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(c) : "l"(a), "l"(b)); }

__global__ void __launch_bounds__(128)
bandpass_kernel(const float2* __restrict__ in, int in_slots, const int* __restrict__ slot_map,
                const float2* __restrict__ taps, const int* __restrict__ enabled, int T, int n_out, int slots,
                float2* __restrict__ out)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    const int i0 = (blockIdx.y * blockDim.y + threadIdx.y) * BP_RB;
    if (s >= slots || i0 >= n_out) return;
    const int col = slot_map ? slot_map[s] : s;
    const float2* x = in + col;                          // x[i * in_slots] is sample i of this channel (row 0 = output 0)
    if (!enabled[s]) {
#pragma unroll
        for (int j = 0; j < BP_RB; j++)
            if (i0 + j < n_out) out[(size_t)(i0 + j) * slots + s] = x[(ptrdiff_t)(i0 + j) * in_slots];
        return;
    }
    // acc = (re, im) of an output: acc += h.re * (v.x, v.y) + h.im * (-v.y, v.x)
    bp_f32x2 acc[BP_RB];
#pragma unroll
    for (int j = 0; j < BP_RB; j++) acc[j] = 0ull;
    // window xw[k] = x[b - (BP_RB-1) + k], b = i0 - t0 (xn = the same samples as (-y, x)); only indices up to
    // i0+BP_RB-1 ever carry weight, and rows past the last valid output are never read: clamp the row index (their
    // accumulators are discarded)
    const int last = n_out - 1;
    bp_f32x2 xw[2 * BP_RB - 1], xn[2 * BP_RB - 1];
#pragma unroll
    for (int k = 0; k < 2 * BP_RB - 1; k++) {
        const float2 v = x[(ptrdiff_t)min(i0 - (BP_RB - 1) + k, last) * in_slots];
        xw[k] = bp_pk2(v.x, v.y);
        xn[k] = bp_pk2(-v.y, v.x);
    }
    for (int t0 = 0; t0 < T; t0 += BP_RB) {
        float2 h[BP_RB];
#pragma unroll
        for (int u = 0; u < BP_RB; u++) h[u] = t0 + u < T ? taps[(size_t)(t0 + u) * slots + s] : make_float2(0.f, 0.f);
#pragma unroll
        for (int u = 0; u < BP_RB; u++) {
            const bp_f32x2 hr = bp_pk2(h[u].x, h[u].x), hi = bp_pk2(h[u].y, h[u].y);
#pragma unroll
            for (int j = 0; j < BP_RB; j++) bp_ffma2(acc[j], hr, xw[BP_RB - 1 + j - u]);
#pragma unroll
            for (int j = 0; j < BP_RB; j++) bp_ffma2(acc[j], hi, xn[BP_RB - 1 + j - u]);
        }
        // slide the window BP_RB samples into the past
#pragma unroll
        for (int k = 2 * BP_RB - 2; k >= BP_RB; k--) { xw[k] = xw[k - BP_RB]; xn[k] = xn[k - BP_RB]; }
        const int b = i0 - t0 - BP_RB;
#pragma unroll
        for (int k = 0; k < BP_RB; k++) {
            const float2 v = x[(ptrdiff_t)(b - (BP_RB - 1) + k) * in_slots];
            xw[k] = bp_pk2(v.x, v.y);
            xn[k] = bp_pk2(-v.y, v.x);
        }
    }
#pragma unroll
    for (int j = 0; j < BP_RB; j++) {
        float re, im;
        bp_upk2(acc[j], re, im);
        if (i0 + j < n_out) out[(size_t)(i0 + j) * slots + s] = make_float2(re, im);
    }
}

// per-channel serial state
struct ChanState {
    float2 fm_last;     // FmDemod: previous (gated) sample
    float dc_last;      // DcBlock: previous block mean
    float iir;          // WfmDeemphasis y[n-1]
    float agc_gain;
    int agc_hang;
    int sq_hang;        // squelch hang counter (blocks)
    int pad;
};

struct ChanCfg {
    int kind;           // OWRX_DEMOD_*
    float sq_level;     // linear power threshold (0 = open)
    float agc_ref, agc_attack, agc_decay, agc_max;
    int agc_hang_time;
    int active;
    float agc_thr;      // largest float a with fl(a / agc_ref) <= 1: "err > 1" <=> abs(v)*gain > agc_thr, exactly
    int mpx;            // WFM multiplex tap: OWRX_MPX_OFF / _F32 / _S16 (tap_gather_kernel)
    int mpx_run;        // index of this slot's run among the group's tapped slots of the same format
};

// Per-slot client-audio resampler (audio_resample_kernel), a per-parity table beside ChanCfg (kept apart so that ChanCfg, which
// the Agc loads whole, keeps its size and alignment): ratio L/M reduced (L = 0: none), K taps per phase, the polyphase table
// tab[p * K + j] = h[p + j * L], and the absolute audio row that is its input 0 (rows before it read as zero).
struct RsCfg {
    int L, M, K, pad;
    long long origin;
    const float* tab;
};

// outputs a resampled slot has produced once the absolute audio row `a` is reached: ceil((a - origin) * L / M)
__host__ __device__ __forceinline__ long long rs_outputs(const RsCfg& c, long long a)
{
    const long long m = a - c.origin;
    return m > 0 ? (m * c.L + c.M - 1) / c.M : 0;
}

// Squelch (SURVEY A.10).  Block power = mean |x|^2 over every `decim`-th sample.  CTA = (32 slots, one block): eight
// warps stage |x|^2 of the block's decimated samples in shared memory (row loads of 32 adjacent slots), then warp 0
// adds them in sample order (the oracle's summation order) from shared memory.  The gate (threshold + hang counter,
// sequential over blocks) is a second tiny kernel.
constexpr int SQ_MAXROWS = 96;           // decimated samples staged per pass (12 KB: fits beside a resident contraction CTA)
__global__ void __launch_bounds__(256)
squelch_power_kernel(const float2* __restrict__ in, int slots, int n_blocks, int length, int decim, float* __restrict__ power)
{
    __shared__ float tile[SQ_MAXROWS][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int s = blockIdx.x * 32 + lane;
    const int b = blockIdx.y;
    const float2* x = in + (size_t)b * length * slots + s;
    const int cnt = (length + decim - 1) / decim;
    float p = 0.f;
    for (int j0 = 0; j0 < cnt; j0 += SQ_MAXROWS) {
        const int nj = min(SQ_MAXROWS, cnt - j0);
        for (int j = w; j < nj; j += 8) {
            const float2 v = x[(size_t)((j0 + j) * decim) * slots];
            tile[j][lane] = v.x * v.x + v.y * v.y;
        }
        __syncthreads();
        if (w == 0) {
#pragma unroll 8
            for (int j = 0; j < nj; j++) p += tile[j][lane];
        }
        __syncthreads();
    }
    if (w == 0) power[(size_t)b * slots + s] = p / (float)cnt;
}

__global__ void __launch_bounds__(128)
squelch_gate_kernel(const float* __restrict__ power, int slots, int n_blocks, int hang_blocks, const ChanCfg* __restrict__ cfg,
                    ChanState* __restrict__ st, unsigned char* __restrict__ gate)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= slots) return;
    const float level = cfg[s].sq_level;
    int hang = st[s].sq_hang;
    for (int b = 0; b < n_blocks; b++) {
        const float p = power[(size_t)b * slots + s];
        int open = 0;
        if (p >= level) { open = 1; hang = hang_blocks; }
        else if (hang > 0) { open = 1; hang--; }
        gate[(size_t)b * slots + s] = (unsigned char)open;
    }
    st[s].sq_hang = hang;
}

// Demodulator front: gated IF -> AmDemod | FmDemod+Limit | RealPart  (SURVEY A.11).
// One thread per (sample, slot).  FM needs the previous gated sample: previous row, or the carried
// state for the first row.  The last row's gated sample is written back by the i == n-1 threads.
__global__ void __launch_bounds__(128)
demod_front_kernel(const float2* __restrict__ in, int slots, int n, int length, const unsigned char* __restrict__ gate,
                   const ChanCfg* __restrict__ cfg, ChanState* __restrict__ st, float* __restrict__ out)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = blockIdx.y * blockDim.y + threadIdx.y;
    if (s >= slots || i >= n) return;
    const int kind = cfg[s].kind;
    float2 x = in[(size_t)i * slots + s];
    if (!gate[(size_t)(i / length) * slots + s]) x = make_float2(0.f, 0.f);
    float y = 0.f;
    if (kind == OWRX_DEMOD_NFM || kind == OWRX_DEMOD_WFM) {
        float2 pv;
        if (i == 0) pv = st[s].fm_last;
        else {
            pv = in[(size_t)(i - 1) * slots + s];
            if (!gate[(size_t)((i - 1) / length) * slots + s]) pv = make_float2(0.f, 0.f);
        }
        const float K = 0.340447550238101026565118445432744920253753662109375f;
        const float num = x.x * (x.y - pv.y) - x.y * (x.x - pv.x);
        const float den = x.x * x.x + x.y * x.y;
        y = den != 0.f ? K * num / den : 0.f;
        y = fminf(1.f, fmaxf(-1.f, y));                       // Limit
    } else if (kind == OWRX_DEMOD_AM) {
        y = sqrtf(x.x * x.x + x.y * x.y);
    } else if (kind == OWRX_DEMOD_SSB) {
        y = x.x;
    }
    out[(size_t)i * slots + s] = y;
}

__global__ void __launch_bounds__(128)
demod_front_commit_kernel(const float2* __restrict__ in, int slots, int n, int length,
                          const unsigned char* __restrict__ gate, ChanState* __restrict__ st)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= slots || n <= 0) return;
    float2 x = in[(size_t)(n - 1) * slots + s];
    if (!gate[(size_t)((n - 1) / length) * slots + s]) x = make_float2(0.f, 0.f);
    st[s].fm_last = x;
}

// ------------------------------------------------------------------------------------------------
// tail_front_kernel — Squelch (block power + gate), the demodulator front and the DcBlock block means in ONE launch
// (squelch_power / squelch_gate / demod_front / demod_front_commit / dc_mean above, kept as the reference evaluation).
// CTA = (32 slots, squelch block b, row split z).  The gate is a sequential scan over blocks, but its hang counter is at most
// `hang_blocks` = 2 (hangLength = 2 x blockLength, csdr/chain/selector.py:124), so the gate of block b is a LOCAL function:
//     open_b = p_b >= L  or  p_{b-1} >= L  or  p_{b-2} >= L           (b >= 2; the carried counter replaces missing blocks)
// and a CTA evaluates the few block powers it needs itself (each in the oracle's summation order) instead of waiting for a
// scan kernel.  FmDemod's first row needs the last GATED sample of block b-1, i.e. that block's gate: one more power.
// In the common case — every slot of blocks b and b-1 above its level — two powers decide everything.
// The state the next feed starts from (hang counter, FmDemod's last sample) is stashed by the last block's CTA and
// committed by tail_back_kernel, which runs after every reader of the old state.
// ------------------------------------------------------------------------------------------------
struct TailStash {
    float2 fm_last;
    int sq_hang;
    int pad;
};
constexpr int TF_ROWS = 1024;            // rows of a block one CTA transforms

__device__ __forceinline__ float tf_block_power(const float2* __restrict__ x, int slots, int length, int decim, int lane, int w,
                                                float (*tile)[32])
{
    // mean |x|^2 over every decim-th sample, added in sample order by warp 0 (the oracle's order); all 8 warps stage
    const int cnt = (length + decim - 1) / decim;
    float p = 0.f;
    for (int j0 = 0; j0 < cnt; j0 += SQ_MAXROWS) {
        const int nj = min(SQ_MAXROWS, cnt - j0);
        for (int j = w; j < nj; j += 8) {
            const float2 v = x[(size_t)((j0 + j) * decim) * slots];
            tile[j][lane] = v.x * v.x + v.y * v.y;
        }
        __syncthreads();
        if (w == 0) {
#pragma unroll 8
            for (int j = 0; j < nj; j++) p += tile[j][lane];
        }
        __syncthreads();
    }
    return p / (float)cnt;                   // valid in warp 0
}

__global__ void __launch_bounds__(256)
tail_front_kernel(const float2* __restrict__ in, int slots, int n_blocks, int length, int decim, int hang_blocks,
                  const ChanCfg* __restrict__ cfg, const ChanState* __restrict__ st, float* __restrict__ power,
                  unsigned char* __restrict__ gate_out, float* __restrict__ f1, float* __restrict__ dc_mean,
                  float* __restrict__ dc_prev, TailStash* __restrict__ stash)
{
    __shared__ float tile[2][SQ_MAXROWS][32];
    __shared__ float s_p[4][32];             // powers of blocks b, b-1, b-2, b-3
    __shared__ unsigned char s_gate[2][32];  // gate of block b, b-1
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int s = blockIdx.x * 32 + lane;
    const int b = blockIdx.y, z = blockIdx.z;
    const ChanCfg c = cfg[s];
    const float level = c.sq_level;
    const int h0 = st[s].sq_hang;
    const bool last_cta = b == n_blocks - 1 && z == gridDim.z - 1;
    // ---- block powers: b and b-1 always, b-2 and b-3 only if some slot is below its level in b or b-1
    const float2* xb = in + (size_t)b * length * slots + s;
    {
        const float p0 = tf_block_power(xb, slots, length, decim, lane, w, tile[0]);
        if (w == 0) s_p[0][lane] = p0;
        const float p1 = b >= 1 ? tf_block_power(xb - (size_t)length * slots, slots, length, decim, lane, w, tile[0]) : 0.f;
        if (w == 0) s_p[1][lane] = p1;
    }
    __syncthreads();
    const bool below = s_p[0][lane] < level || (b >= 1 && s_p[1][lane] < level);
    if (__syncthreads_or(below)) {
        const float p2 = b >= 2 ? tf_block_power(xb - (size_t)2 * length * slots, slots, length, decim, lane, w, tile[0]) : 0.f;
        const float p3 = b >= 3 ? tf_block_power(xb - (size_t)3 * length * slots, slots, length, decim, lane, w, tile[0]) : 0.f;
        if (w == 0) { s_p[2][lane] = p2; s_p[3][lane] = p3; }
    } else if (w == 0) {
        s_p[2][lane] = level; s_p[3][lane] = level;          // never looked at: everything is open
    }
    __syncthreads();
    if (w == 0) {
        // hang counter entering block j: h_j = p_{j-1} >= L ? H : (p_{j-2} >= L ? H - 1 : ...) for H = hang_blocks = 2; blocks
        // before the pass come from the carried counter h0
        auto hang_before = [&](int j) -> int {                // j = b or b - 1 (>= 0)
            const int d = b - j;                              // s_p index of block j
            if (j == 0) return h0;
            const bool o1 = s_p[d + 1][lane] >= level;        // block j - 1
            if (o1) return hang_blocks;
            if (j == 1) return max(h0 - 1, 0);
            const bool o2 = s_p[d + 2][lane] >= level;        // block j - 2
            if (hang_blocks >= 2 && o2) return hang_blocks - 1;
            if (j == 2) return max(h0 - 2, 0);
            return 0;
        };
        const int hb = hang_before(b);
        const bool open_b = s_p[0][lane] >= level || hb > 0;
        s_gate[0][lane] = open_b ? 1 : 0;
        bool open_prev = true;
        if (b >= 1) open_prev = s_p[1][lane] >= level || hang_before(b - 1) > 0;
        s_gate[1][lane] = open_prev ? 1 : 0;
        if (z == 0) {
            power[(size_t)b * slots + s] = s_p[0][lane];
            gate_out[(size_t)b * slots + s] = open_b ? 1 : 0;
        }
        if (last_cta) stash[s].sq_hang = s_p[0][lane] >= level ? hang_blocks : max(hb - 1, 0);
    }
    __syncthreads();
    const bool open_b = s_gate[0][lane] != 0, open_prev = s_gate[1][lane] != 0;
    // ---- demodulator front over this CTA's rows of the block, in tiles of SQ_MAXROWS rows.  DcBlock's block mean (AM) is
    // the in-order sum of the gated envelope over the WHOLE block: the z = 0 CTA also walks the rows other CTAs transform,
    // every warp stages its rows' envelopes in a shared tile, and warp 0 adds tile t in sample order (the oracle's order)
    // while the other warps already work on tile t + 1 (two tile buffers, one barrier per tile).
    const bool am = c.kind == OWRX_DEMOD_AM;
    const bool do_dc = __syncthreads_or(am) && z == 0;
    const int r0 = z * TF_ROWS, r1 = min(length, r0 + TF_ROWS);
    const int t_begin = do_dc ? 0 : r0, t_end = do_dc ? length : r1;
    const int kind = c.kind;
    float acc = 0.f;
    int buf = 0;
    for (int t0 = t_begin; t0 < t_end; t0 += SQ_MAXROWS, buf ^= 1) {
        const int nt = min(SQ_MAXROWS, t_end - t0);
        // a warp takes TF_WR consecutive rows of the tile and fetches them (and the row before) in one go: one memory latency per
        // tile and warp instead of one per row (54 CTAs cannot hide latency by occupancy)
        constexpr int TF_WR = SQ_MAXROWS / 8;
        const int j0 = w * TF_WR;
        float2 xr[TF_WR + 1];                               // xr[k + 1] = row t0 + j0 + k, xr[0] = the row before (gated)
#pragma unroll
        for (int k = 0; k <= TF_WR; k++) {
            const int i = t0 + j0 + k - 1;
            float2 v = make_float2(0.f, 0.f);
            if (k == 0) {
                if (i >= 0) { if (open_b) v = xb[(size_t)i * slots]; }
                else if (b > 0) { if (open_prev) v = xb[-(ptrdiff_t)slots]; }
                else v = st[s].fm_last;
            } else if (j0 + k - 1 < nt && open_b) {
                v = xb[(size_t)i * slots];
            }
            xr[k] = v;
        }
#pragma unroll
        for (int k = 0; k < TF_WR; k++) {
            const int j = j0 + k, i = t0 + j;
            if (j >= nt) break;
            const float2 x = xr[k + 1], pv = xr[k];
            float y = 0.f;
            if (kind == OWRX_DEMOD_NFM || kind == OWRX_DEMOD_WFM) {
                const float K = 0.340447550238101026565118445432744920253753662109375f;
                const float num = x.x * (x.y - pv.y) - x.y * (x.x - pv.x);
                const float den = x.x * x.x + x.y * x.y;
                y = den != 0.f ? K * num / den : 0.f;
                y = fminf(1.f, fmaxf(-1.f, y));                       // Limit
            } else if (kind == OWRX_DEMOD_AM) {
                y = sqrtf(x.x * x.x + x.y * x.y);
            } else if (kind == OWRX_DEMOD_SSB) {
                y = x.x;
            }
            if (do_dc) tile[buf][j][lane] = am ? y : 0.f;
            if (i >= r0 && i < r1) {
                f1[((size_t)b * length + i) * slots + s] = y;
                if (last_cta && i == length - 1) stash[s].fm_last = x;
            }
        }
        if (do_dc) {
            __syncthreads();
            if (w == 0) {
#pragma unroll 8
                for (int j = 0; j < nt; j++) acc += tile[buf][j][lane];
            }
        }
    }
    if (z == 0 && w == 0) {
        dc_mean[(size_t)b * slots + s] = am ? acc / (float)length : 0.f;
        if (b == 0) dc_prev[s] = am ? st[s].dc_last : 0.f;
    }
}

// the state hand-over of the fused tail: runs as part of tail_back_kernel's first CTAs, after every reader of the old state
__device__ __forceinline__ void tail_commit(int s, int n_blocks, const ChanCfg* cfg, const float* dc_mean, int slots,
                                            const TailStash* stash, ChanState* st)
{
    st[s].sq_hang = stash[s].sq_hang;
    st[s].fm_last = stash[s].fm_last;
    if (cfg[s].kind == OWRX_DEMOD_AM) st[s].dc_last = dc_mean[(size_t)(n_blocks - 1) * slots + s];
}

__global__ void __launch_bounds__(128)
tail_commit_kernel(int slots, int n_blocks, const ChanCfg* __restrict__ cfg, const float* __restrict__ dc_mean,
                   const TailStash* __restrict__ stash, ChanState* __restrict__ st)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < slots && n_blocks > 0) tail_commit(s, n_blocks, cfg, dc_mean, slots, stash, st);
}

// Demodulator back (12 kHz-class groups): NFM -> NfmDeemphasis FIR; AM -> DcBlock (block = squelch
// block); SSB -> copy.  in points at the row of output 0 and has >= T-1 + 2*DB_RB rows of history before it.
// A thread owns DB_RB consecutive outputs of one channel; the FIR slides a 2*DB_RB-1 sample window through
// registers (taps in ascending order, like the oracle): DB_RB loads per DB_RB^2 FMAs.
constexpr int DB_RB = 8;
__global__ void __launch_bounds__(128)
demod_back_kernel(const float* __restrict__ in, int slots, int n, int length, const float* __restrict__ deemph, int T,
                  const ChanCfg* __restrict__ cfg, const float* __restrict__ dc_mean, const float* __restrict__ dc_prev,
                  float* __restrict__ out)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    const int i0 = (blockIdx.y * blockDim.y + threadIdx.y) * DB_RB;
    if (s >= slots || i0 >= n) return;
    const int kind = cfg[s].kind;
    const float* x = in + s;
    float y[DB_RB];
    if (kind == OWRX_DEMOD_NFM) {
#pragma unroll
        for (int j = 0; j < DB_RB; j++) y[j] = 0.f;
        // xw[d + DB_RB - 1] = x[i0 - t0 + d], d in (-DB_RB, DB_RB); rows past the last output are clamped (never weighted
        // into a stored output)
        const int last = n - 1;
        float xw[2 * DB_RB - 1];
#pragma unroll
        for (int k = 0; k < 2 * DB_RB - 1; k++) xw[k] = x[(ptrdiff_t)min(i0 - (DB_RB - 1) + k, last) * slots];
        for (int t0 = 0; t0 < T; t0 += DB_RB) {
            float h[DB_RB];
#pragma unroll
            for (int u = 0; u < DB_RB; u++) h[u] = t0 + u < T ? __ldg(deemph + t0 + u) : 0.f;
#pragma unroll
            for (int u = 0; u < DB_RB; u++)
#pragma unroll
                for (int j = 0; j < DB_RB; j++) y[j] = fmaf(h[u], xw[DB_RB - 1 + j - u], y[j]);
#pragma unroll
            for (int k = 2 * DB_RB - 2; k >= DB_RB; k--) xw[k] = xw[k - DB_RB];
            const int b = i0 - t0 - DB_RB;
#pragma unroll
            for (int k = 0; k < DB_RB; k++) xw[k] = x[(ptrdiff_t)(b - (DB_RB - 1) + k) * slots];
        }
    } else if (kind == OWRX_DEMOD_AM) {
#pragma unroll
        for (int j = 0; j < DB_RB; j++) {
            const int i = min(i0 + j, n - 1);
            const int b = i / length, ib = i % length;
            const float last = b == 0 ? dc_prev[s] : dc_mean[(size_t)(b - 1) * slots + s];
            const float avg = dc_mean[(size_t)b * slots + s];
            y[j] = x[(size_t)i * slots] - (last + (avg - last) * ((float)ib / (float)length));
        }
    } else {
#pragma unroll
        for (int j = 0; j < DB_RB; j++) y[j] = x[(size_t)min(i0 + j, n - 1) * slots];
    }
#pragma unroll
    for (int j = 0; j < DB_RB; j++)
        if (i0 + j < n) out[(size_t)(i0 + j) * slots + s] = y[j];
}

// DcBlock block means.  CTA = (32 slots, one block): eight warps stage the block's samples in shared memory, warp 0
// adds them in sample order (sequential float sum like the oracle).
constexpr int DC_ROWS = 96;             // 2 x 12 KB: fits beside a resident contraction CTA
__global__ void __launch_bounds__(256)
dc_mean_kernel(const float* __restrict__ in, int slots, int n_blocks, int length, const ChanCfg* __restrict__ cfg,
               ChanState* __restrict__ st, float* __restrict__ dc_mean, float* __restrict__ dc_prev)
{
    __shared__ float tile[2][DC_ROWS][32];             // double-buffered: warps 1-7 fetch tile t+1 while warp 0 adds tile t
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int s = blockIdx.x * 32 + lane;
    const int b = blockIdx.y;
    const bool am = cfg[s].kind == OWRX_DEMOD_AM;
    if (!__syncthreads_or(am)) {                       // no AM channel among these 32 slots
        if (w == 0) { if (b == 0) dc_prev[s] = 0.f; dc_mean[(size_t)b * slots + s] = 0.f; }
        return;
    }
    const float* x = in + (size_t)b * length * slots + s;
    float acc = 0.f;
    const int nt = (length + DC_ROWS - 1) / DC_ROWS;
    for (int i = w; i < min(DC_ROWS, length); i += 8) tile[0][i][lane] = x[(size_t)i * slots];
    __syncthreads();
    for (int t = 0; t < nt; t++) {
        const int i0 = t * DC_ROWS, ni = min(DC_ROWS, length - i0);
        if (w == 0) {
#pragma unroll 8
            for (int i = 0; i < ni; i++) acc += tile[t & 1][i][lane];
        } else if (t + 1 < nt) {
            const int n1 = min(DC_ROWS, length - i0 - DC_ROWS);
            for (int i = w - 1; i < n1; i += 7) tile[(t + 1) & 1][i][lane] = x[(size_t)(i0 + DC_ROWS + i) * slots];
        }
        __syncthreads();
    }
    if (w == 0) {
        dc_mean[(size_t)b * slots + s] = am ? acc / (float)length : 0.f;
        if (b == 0) dc_prev[s] = am ? st[s].dc_last : 0.f;
    }
}

__global__ void __launch_bounds__(128)
dc_commit_kernel(int slots, int n_blocks, const ChanCfg* __restrict__ cfg, const float* __restrict__ dc_mean,
                 ChanState* __restrict__ st)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= slots || n_blocks <= 0) return;
    if (cfg[s].kind == OWRX_DEMOD_AM) st[s].dc_last = dc_mean[(size_t)(n_blocks - 1) * slots + s];
}

// Forward-looking real FIR with taps shared by all channels: v[i] = sum_t x[i+t] pre[t] — the prefilter of
// FractionalDecimator(FLOAT, prefilter=True) evaluated once per input index instead of 12 times per output.
// Register-blocked like bandpass_kernel; rows past `last_row` are never weighted by a non-zero tap and are clamped.
__global__ void __launch_bounds__(128)
fir_fwd_f_kernel(const float* __restrict__ in, int slots, int n_out, int last_row, const float* __restrict__ pre, int T,
                 float* __restrict__ out)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    const int i0 = (blockIdx.y * blockDim.y + threadIdx.y) * BP_RB;
    if (s >= slots || i0 >= n_out) return;
    const float* x = in + s;
    float acc[BP_RB];
#pragma unroll
    for (int j = 0; j < BP_RB; j++) acc[j] = 0.f;
    float xw[2 * BP_RB - 1];                            // xw[k] = x[i0 + t0 + k]
#pragma unroll
    for (int k = 0; k < 2 * BP_RB - 1; k++) xw[k] = x[(size_t)min(i0 + k, last_row) * slots];
    for (int t0 = 0; t0 < T; t0 += BP_RB) {
        float h[BP_RB];
#pragma unroll
        for (int u = 0; u < BP_RB; u++) h[u] = t0 + u < T ? __ldg(pre + t0 + u) : 0.f;
#pragma unroll
        for (int u = 0; u < BP_RB; u++)
#pragma unroll
            for (int j = 0; j < BP_RB; j++) acc[j] = fmaf(h[u], xw[j + u], acc[j]);
#pragma unroll
        for (int k = 0; k < BP_RB - 1; k++) xw[k] = xw[k + BP_RB];
#pragma unroll
        for (int k = BP_RB - 1; k < 2 * BP_RB - 1; k++) xw[k] = x[(size_t)min(i0 + t0 + BP_RB + k, last_row) * slots];
    }
#pragma unroll
    for (int j = 0; j < BP_RB; j++)
        if (i0 + j < n_out) out[(size_t)(i0 + j) * slots + s] = acc[j];
}

// WFM: FractionalDecimator(Format.FLOAT, rate, prefilter=True): 12-point Lagrange over the
// forward-looking prefiltered signal v[idx] = sum_t x[idx+t] pre[t]  (SURVEY A.8).
__global__ void __launch_bounds__(128)
fracdec_f_kernel(const float* __restrict__ in, long long in_abs0, int slots, double rate, long long m0, int n_out,
                 const float* __restrict__ pre, int Tpre, float* __restrict__ out)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    const int m = blockIdx.y * blockDim.y + threadIdx.y;
    if (s >= slots || m >= n_out) return;
    const double where = 5.0 + (double)(m0 + m) * rate;
    const double ihd = ceil(where);
    float c[12];
    lagrange12((float)(ihd - where), c);
    const float* x = in + ((long long)ihd - 5 - in_abs0) * slots + s;
    float acc = 0.f;
#pragma unroll 1
    for (int i = 0; i < 12; i++) {
        float v;
        if (Tpre > 0) {
            v = 0.f;
            for (int t = 0; t < Tpre; t++) v += x[(size_t)(i + t) * slots] * pre[t];
        } else {
            v = x[(size_t)i * slots];        // input already prefiltered (fir_fwd_f_kernel)
        }
        acc += c[i] * v;
    }
    out[(size_t)m * slots + s] = acc;
}

// Sample-serial recurrences run one channel per lane.  A lane's samples sit `slots` floats apart, so a
// warp-wide access to one time step is coalesced.  The input is streamed through a per-warp shared
// memory ring with cp.async, SER_STAGES-1 tiles of SER_TT time steps ahead of the dependent chain, so
// the only latency left on the chain is the arithmetic itself.  Each lane only ever reads the column
// it loaded itself: no barrier is needed.
constexpr int SER_TT = 16;
constexpr int SER_STAGES = 6;

__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc)
{
    unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(d), "l"(gsrc));
}
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

struct SerialFeed {
    float (*ring)[SER_TT][32];
    const float* in;
    int slots, n, s, lane, nt;
    __device__ void issue(int tile) const
    {
        if (tile < nt) {
#pragma unroll
            for (int t = 0; t < SER_TT; t++) {
                const int i = tile * SER_TT + t;
                if (i < n) cp_async4(&ring[tile % SER_STAGES][t][lane], in + (size_t)i * slots + s);
            }
        }
        cp_async_commit();
    }
};

// WfmDeemphasis one-pole IIR y[n] = alpha x[n] + (1-alpha) y[n-1] (SURVEY A.11).  A linear recurrence: one WARP owns a
// channel and advances 256 samples per step.  Each lane runs its 8 consecutive samples from a zero state, the lane
// end-states are combined by a warp scan of the affine maps y -> om^8 y + s (5 shuffles), and the lane re-runs its 8
// samples from its true entry state.  Same recurrence formula per sample; only the entry states are associated
// differently (float32 rounding at the 1e-7 level against the sequential order).  Tile staging as in agc_kernel below.
constexpr int IIR_E = 8;           // consecutive samples per lane
constexpr int IIR_CH = 8;          // channels (= warps) per CTA
constexpr int IIR_TL = 32 * IIR_E; // samples per warp step (= threads per CTA)
__global__ void __launch_bounds__(IIR_TL)
wfm_deemph_kernel(const float* __restrict__ in, int slots, int n, float alpha, ChanState* __restrict__ st,
                  float* __restrict__ out)
{
    __shared__ __align__(16) float xin[2][IIR_CH][IIR_TL + 4];
    __shared__ __align__(16) float xout[IIR_CH][IIR_TL + 4];
    if (n <= 0) return;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int s0 = blockIdx.x * IIR_CH, s = s0 + w;
    const float om = 1.0f - alpha;
    float om_pow[6];                                   // om^(8 * 2^k)
    {
        float p = om;
#pragma unroll
        for (int k = 0; k < 3; k++) p *= p;            // om^8
#pragma unroll
        for (int k = 0; k < 6; k++) { om_pow[k] = p; p *= p; }
    }
    float y = st[s].iir;                               // state entering the current step (warp-uniform)
    const int nt = (n + IIR_TL - 1) / IIR_TL;
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    auto fetch = [&](int tile, float4& lo, float4& hi) {
        const int t = tile * IIR_TL + tid;
        if (t < n) {
            const float4* p = reinterpret_cast<const float4*>(in + (size_t)t * slots + s0);
            lo = __ldg(p); hi = __ldg(p + 1);
        } else {
            lo = zero4; hi = zero4;
        }
    };
    auto stage = [&](int buf, const float4& lo, const float4& hi) {
        xin[buf][0][tid] = lo.x; xin[buf][1][tid] = lo.y; xin[buf][2][tid] = lo.z; xin[buf][3][tid] = lo.w;
        xin[buf][4][tid] = hi.x; xin[buf][5][tid] = hi.y; xin[buf][6][tid] = hi.z; xin[buf][7][tid] = hi.w;
    };
    float4 lo, hi;
    fetch(0, lo, hi);
    stage(0, lo, hi);
    __syncthreads();
    for (int tile = 0; tile < nt; tile++) {
        const int buf = tile & 1;
        if (tile + 1 < nt) fetch(tile + 1, lo, hi);
        float v[IIR_E];
        {
            const float4* xv = reinterpret_cast<const float4*>(&xin[buf][w][IIR_E * lane]);
            const float4 a = xv[0], b = xv[1];
            v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
        }
        // lane-local response from a zero state
        float sl = 0.f;
#pragma unroll
        for (int e = 0; e < IIR_E; e++) sl = alpha * v[e] + om * sl;
        // inclusive scan of (A, B): state after lane l = A_l * y_entry + B_l, A = om^(8 (l+1))
        float B = sl;
#pragma unroll
        for (int k = 0; k < 5; k++) {
            const float prev = __shfl_up_sync(0xffffffffu, B, 1 << k);
            if (lane >= (1 << k)) B = om_pow[k] * prev + B;
        }
        // A_l = om^(8 (l+1)) by binary powers
        float A = 1.f;
#pragma unroll
        for (int k = 0; k < 5; k++)
            if ((lane + 1) & (1 << k)) A *= om_pow[k];
        if (lane == 31) A = om_pow[5];
        const float endstate = A * y + B;              // state after this lane's 8 samples
        float yin = __shfl_up_sync(0xffffffffu, endstate, 1);
        if (lane == 0) yin = y;
        // true outputs of this lane
        float yo[IIR_E];
#pragma unroll
        for (int e = 0; e < IIR_E; e++) { yin = alpha * v[e] + om * yin; yo[e] = yin; }
        {
            float4* ov = reinterpret_cast<float4*>(&xout[w][IIR_E * lane]);
            ov[0] = make_float4(yo[0], yo[1], yo[2], yo[3]);
            ov[1] = make_float4(yo[4], yo[5], yo[6], yo[7]);
        }
        // the next step's entry state: the state after the last VALID sample of this tile
        const int valid = min(IIR_TL, n - tile * IIR_TL);
        const int ll = (valid - 1) / IIR_E, le = (valid - 1) % IIR_E;
        float cand = yo[IIR_E - 1];
#pragma unroll
        for (int e = 0; e < IIR_E - 1; e++) cand = le == e ? yo[e] : cand;
        y = __shfl_sync(0xffffffffu, cand, ll);
        __syncthreads();
        const int t = tile * IIR_TL + tid;
        if (t < n) {
            float4* p = reinterpret_cast<float4*>(out + (size_t)t * slots + s0);
            p[0] = make_float4(xout[0][tid], xout[1][tid], xout[2][tid], xout[3][tid]);
            p[1] = make_float4(xout[4][tid], xout[5][tid], xout[6][tid], xout[7][tid]);
        }
        if (tile + 1 < nt) stage(buf ^ 1, lo, hi);
        __syncthreads();
    }
    if (lane == 0) st[s].iir = y;
}

// Agc (SPEC-DEFINED, SURVEY A.11): per non-zero sample, |v|*gain/ref > 1 -> gain *= 1-attack, hang = hang_time;
// else hang > 0 -> hang--; else gain *= 1+decay; gain clamped to [0, max]; out = clamp(v*gain, +-1).
//
// The recurrence is sample-serial, but BETWEEN attack events the state does not depend on the data, only on the
// count of non-zero samples: the gain is constant during the hang and then follows the iterated product
// U[k] = fl(U[k-1]*up).  One WARP owns a channel and evaluates 128 consecutive samples at a time (4 per lane):
//   * ballots give every lane how many hang decrements / rising steps precede it,
//   * the warp runs the R <= 128 rising steps of the tile as ONE FMUL chain (the only serial work: one instruction per
//     rising sample; the [0, max] clamp commutes with the monotone chain: min(fl(min(u,M)*up), M) == min(fl(u*up), M)),
//   * every lane tests its own sample for an attack against the speculative "no attack" gain; the first attack
//     found (ballot + ffs) is applied and the lanes after it are re-evaluated from the new state.
// Bit-identical to the sample-by-sample recurrence (tests/test_gpu_selector.py::test_agc_bit_exact_on_own_demod).
constexpr int AGC_CH = 8;          // channels (= warps) per CTA: one 32-byte sector per time row
constexpr int AGC_TL = 256;        // samples staged per step (= threads per CTA)

constexpr int AGC_E = 4;           // consecutive samples per lane: a warp step covers 128 samples

struct AgcWarp {
    float gain, dn, up, thr, gmax;
    int hang, hang_time;
    // v[e] = sample 4*lane + e of the step; returns the outputs in place.  U: per-warp scratch of 132 floats.
    // The same step when every one of the 128 samples is non-zero (the usual case: audio is exactly 0 only behind a closed
    // squelch).  The "how many live / rising samples precede me" counts of the general path are then plain index
    // arithmetic — sample j of the step (pending from j0) has j - j0 live samples before it, is a rising step iff
    // j - j0 >= hang, and has max(j - j0 - hang, 0) rising steps before it — so the eight ballots per pass go away, and the
    // chain values are stored four at a time.  Ud[k + 3] = U[k] (so that k = 1, 5, 9, ... are 16-byte aligned).
    __device__ __forceinline__ void step_dense(float (&v)[AGC_E], int lane, float* Ud)
    {
        const unsigned full = 0xffffffffu;
        float o[AGC_E];
        int j0 = 0;
        while (true) {
            const int R = max(32 * AGC_E - j0 - hang, 0);                   // rising steps among the pending samples
            float u = gain;
            Ud[3] = u;
            // the chain of R <= 128 dependent FMULs is the only sample-serial work of the step: straight-line groups of four
            // (4 FMUL + one 16-byte store, each group under one warp-uniform predicate computed up front), no loop-carried
            // counter or branch between the multiplies
#pragma unroll
            for (int c = 0; c < 32 * AGC_E / 4; c++) {
                if (4 * c + 4 <= R) {
                    const float a = u * up, b = a * up, cc = b * up, d = cc * up;
                    *reinterpret_cast<float4*>(&Ud[4 * c + 4]) = make_float4(a, b, cc, d);
                    u = d;
                }
            }
            for (int k = (R & ~3) + 1; k <= R; k++) {
                u *= up;
                Ud[k + 3] = u;
            }
            __syncwarp();
            float gb[AGC_E], ga[AGC_E];
            unsigned att = 0, pend = 0;
#pragma unroll
            for (int e = 0; e < AGC_E; e++) {
                const int d = AGC_E * lane + e - j0;                        // live samples before this one (if pending)
                const int rb = max(d - hang, 0);
                const int is_rise = d >= hang ? 1 : 0;
                const int idx = max(rb, 0);
                gb[e] = fminf(Ud[idx + 3], gmax);
                ga[e] = fminf(Ud[idx + is_rise + 3], gmax);
                const bool p = d >= 0;
                pend |= (p ? 1u : 0u) << e;
                att |= (p && fabsf(v[e]) * gb[e] > thr ? 1u : 0u) << e;
            }
            __syncwarp();
            const unsigned am = __ballot_sync(full, att != 0u);
            if (am == 0u) {
#pragma unroll
                for (int e = 0; e < AGC_E; e++)
                    if ((pend >> e) & 1u) o[e] = fminf(1.f, fmaxf(-1.f, v[e] * ga[e]));
                gain = fminf(u, gmax);
                hang = max(hang - (32 * AGC_E - j0), 0);
                break;
            }
            const int L = __ffs(am) - 1;
            const int ef = __ffs(att) - 1;
            const float gsel = ef == 0 ? gb[0] : (ef == 1 ? gb[1] : (ef == 2 ? gb[2] : gb[3]));
            const int e_first = __shfl_sync(full, ef, L);
            const float gnew = fmaxf(fminf(__shfl_sync(full, gsel, L) * dn, gmax), 0.f);
            const int jf = AGC_E * L + e_first;
#pragma unroll
            for (int e = 0; e < AGC_E; e++) {
                const int j = AGC_E * lane + e;
                if (((pend >> e) & 1u) && j < jf) o[e] = fminf(1.f, fmaxf(-1.f, v[e] * ga[e]));
                if (j == jf) o[e] = fminf(1.f, fmaxf(-1.f, v[e] * gnew));
            }
            gain = gnew;
            hang = hang_time;
            j0 = jf + 1;
            if (j0 >= 32 * AGC_E) break;
        }
#pragma unroll
        for (int e = 0; e < AGC_E; e++) v[e] = o[e];
    }

    __device__ __forceinline__ void step(float (&v)[AGC_E], int lane, volatile float* U)
    {
        const unsigned full = 0xffffffffu, lt = (1u << lane) - 1u;
        unsigned nzbits = 0;
#pragma unroll
        for (int e = 0; e < AGC_E; e++) nzbits |= (v[e] != 0.f ? 1u : 0u) << e;
        if (__all_sync(full, nzbits == 0xfu)) {
            step_dense(v, lane, const_cast<float*>(U));
            return;
        }
        float o[AGC_E];
#pragma unroll
        for (int e = 0; e < AGC_E; e++) o[e] = v[e];
        int j0 = 0;                                        // first sample of the step not yet committed
        while (true) {
            // samples >= j0 still to do: this lane's bits e with 4*lane + e >= j0
            const int sh = min(max(j0 - AGC_E * lane, 0), AGC_E);
            const unsigned act = (0xfu << sh) & 0xfu;
            const unsigned live = nzbits & act;
            unsigned m[AGC_E];
#pragma unroll
            for (int e = 0; e < AGC_E; e++) m[e] = __ballot_sync(full, (live >> e) & 1u);
            int base = 0, n_live = 0;
#pragma unroll
            for (int e = 0; e < AGC_E; e++) { base += __popc(m[e] & lt); n_live += __popc(m[e]); }
            // rising steps: live samples once the hang counter has run out
            unsigned rise = 0;
#pragma unroll
            for (int e = 0; e < AGC_E; e++) {
                const int before = base + __popc(live & ((1u << e) - 1u));
                rise |= (((live >> e) & 1u) && before >= hang ? 1u : 0u) << e;
            }
            int rbase = 0, R = 0;
#pragma unroll
            for (int e = 0; e < AGC_E; e++) {
                const unsigned r = __ballot_sync(full, (rise >> e) & 1u);
                rbase += __popc(r & lt);
                R += __popc(r);
            }
            // U[k] = k rising steps applied to the entry gain: the only sample-serial work (FMUL + STS per step)
            float u = gain;
            U[0] = u;
#pragma unroll 8
            for (int k = 1; k <= R; k++) {
                u *= up;
                U[k] = u;
            }
            __syncwarp();
            float gb[AGC_E], ga[AGC_E];
            unsigned att = 0;
#pragma unroll
            for (int e = 0; e < AGC_E; e++) {
                const int rb = rbase + __popc(rise & ((1u << e) - 1u));
                gb[e] = fminf(U[rb], gmax);                                 // gain sample e is compared with
                ga[e] = fminf(U[rb + ((rise >> e) & 1u)], gmax);            // gain applied to its output (no attack)
                att |= (((live >> e) & 1u) && fabsf(v[e]) * gb[e] > thr ? 1u : 0u) << e;   // == (|v|*gain/ref > 1), exactly
            }
            __syncwarp();
            const unsigned am = __ballot_sync(full, att != 0u);
            if (am == 0u) {
#pragma unroll
                for (int e = 0; e < AGC_E; e++)
                    if ((act >> e) & 1u) o[e] = fminf(1.f, fmaxf(-1.f, v[e] * ga[e]));
                gain = fminf(u, gmax);
                hang = max(hang - n_live, 0);
                break;
            }
            const int L = __ffs(am) - 1;
            const int ef = __ffs(att) - 1;                                   // this lane's first attacking sample (if any)
            const float gsel = ef == 0 ? gb[0] : (ef == 1 ? gb[1] : (ef == 2 ? gb[2] : gb[3]));
            const int e_first = __shfl_sync(full, ef, L);
            const float gnew = fmaxf(fminf(__shfl_sync(full, gsel, L) * dn, gmax), 0.f);
            const int jf = AGC_E * L + e_first;
#pragma unroll
            for (int e = 0; e < AGC_E; e++) {
                const int j = AGC_E * lane + e;
                if (((act >> e) & 1u) && j < jf) o[e] = fminf(1.f, fmaxf(-1.f, v[e] * ga[e]));
                if (j == jf) o[e] = fminf(1.f, fmaxf(-1.f, v[e] * gnew));
            }
            gain = gnew;
            hang = hang_time;
            j0 = jf + 1;
            if (j0 >= 32 * AGC_E) break;
        }
#pragma unroll
        for (int e = 0; e < AGC_E; e++) v[e] = o[e];
    }
};

// CTA = 8 adjacent channel slots (slots is a multiple of 64).  All 256 threads move [256 samples][8 slots] tiles between
// global memory (32-byte rows: whole sectors) and shared memory, register-prefetched one tile ahead; warp w then runs
// channel w's recurrence over the tile, 128 samples at a time.
__global__ void __launch_bounds__(AGC_TL)
agc_kernel(const float* __restrict__ in, int slots, int n, const ChanCfg* __restrict__ cfg, ChanState* __restrict__ st,
           float* __restrict__ out)
{
    __shared__ __align__(16) float xin[2][AGC_CH][AGC_TL];
    __shared__ __align__(16) float xout[AGC_CH][AGC_TL];
    __shared__ __align__(16) float U_all[AGC_CH][32 * AGC_E + 8];
    if (n <= 0) return;
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int s0 = blockIdx.x * AGC_CH, s = s0 + w;
    const ChanCfg c = cfg[s];
    const bool bypass = c.kind == OWRX_DEMOD_WFM || c.kind == OWRX_DEMOD_NONE;     // no Agc in these chains: pass through
    AgcWarp a{st[s].agc_gain, 1.f - c.agc_attack, 1.f + c.agc_decay, c.agc_thr, c.agc_max, st[s].agc_hang, c.agc_hang_time};
    a.gain = fmaxf(fminf(a.gain, a.gmax), 0.f);
    volatile float* U = U_all[w];
    const int nt = (n + AGC_TL - 1) / AGC_TL;
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    auto fetch = [&](int tile, float4& lo, float4& hi) {
        const int t = tile * AGC_TL + tid;
        if (t < n) {
            const float4* p = reinterpret_cast<const float4*>(in + (size_t)t * slots + s0);
            lo = __ldg(p); hi = __ldg(p + 1);
        } else {
            lo = zero4; hi = zero4;                        // zeros change neither state nor outputs
        }
    };
    auto stage = [&](int buf, const float4& lo, const float4& hi) {
        xin[buf][0][tid] = lo.x; xin[buf][1][tid] = lo.y; xin[buf][2][tid] = lo.z; xin[buf][3][tid] = lo.w;
        xin[buf][4][tid] = hi.x; xin[buf][5][tid] = hi.y; xin[buf][6][tid] = hi.z; xin[buf][7][tid] = hi.w;
    };
    float4 lo, hi;
    fetch(0, lo, hi);
    stage(0, lo, hi);
    __syncthreads();
    for (int tile = 0; tile < nt; tile++) {
        const int buf = tile & 1;
        if (tile + 1 < nt) fetch(tile + 1, lo, hi);
#pragma unroll 1
        for (int k = 0; k < AGC_TL / (32 * AGC_E); k++) {
            const float4 x4 = *reinterpret_cast<const float4*>(&xin[buf][w][k * 32 * AGC_E + AGC_E * lane]);
            float v[AGC_E] = {x4.x, x4.y, x4.z, x4.w};
            if (!bypass) a.step(v, lane, U);
            *reinterpret_cast<float4*>(&xout[w][k * 32 * AGC_E + AGC_E * lane]) = make_float4(v[0], v[1], v[2], v[3]);
        }
        __syncthreads();                                   // xout complete, xin[buf] consumed
        const int t = tile * AGC_TL + tid;
        if (t < n) {
            float4* p = reinterpret_cast<float4*>(out + (size_t)t * slots + s0);
            p[0] = make_float4(xout[0][tid], xout[1][tid], xout[2][tid], xout[3][tid]);
            p[1] = make_float4(xout[4][tid], xout[5][tid], xout[6][tid], xout[7][tid]);
        }
        if (tile + 1 < nt) stage(buf ^ 1, lo, hi);
        __syncthreads();                                   // next tile staged, xout free
    }
    if (lane == 0 && !bypass) {
        st[s].agc_gain = a.gain;
        st[s].agc_hang = a.hang;
    }
}

// [n][slots] -> [slots][n] (output drain: one contiguous run per channel for the host)
template <typename T>
__global__ void __launch_bounds__(256) transpose_kernel(const T* __restrict__ in, int slots, size_t n, T* __restrict__ out)
{
    __shared__ T tile[32][33];
    const int s0 = blockIdx.x * 32;
    const size_t i0 = (size_t)blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += 8) {
        const size_t i = i0 + r;
        const int sl = s0 + threadIdx.x;
        if (i < n && sl < slots) tile[r][threadIdx.x] = in[i * slots + sl];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int sl = s0 + r;
        const size_t i = i0 + threadIdx.x;
        if (i < n && sl < slots) out[(size_t)sl * n + i] = tile[threadIdx.x][r];
    }
}

// ------------------------------------------------------------------------------------------------
// Client-audio resampler: AudioResampler(in, out) -> Limit (csdr/chain/clientaudio.py:6-19), in front of the audio tail.
// SPEC-DEFINED (the reference's libsamplerate is not in the tree): L/M = out/in reduced, polyphase Kaiser-windowed sinc of
// K taps per phase (designed on the host, RsCfg::tab), causal
//   y[k] = sum_{j<K} x[floor(kM/L) - j] * h[kM - floor(kM/L) L + jL],   x[n < 0] = 0,
// with n counted from RsCfg::origin; after n inputs exactly ceil(nL/M) outputs exist, whatever the pass sizes.
// The ratio is per slot.  x: the group's audio rows (f3), row r holds absolute row x_abs0 + r and the K - 1 rows before this
// pass are kept as history.  Output k of a slot goes to row k - (outputs before the feed) of `out`, so that the audio tail
// finds the pass's outputs where it writes their int16 samples.  Slots without a resampler, or whose audio stays float
// (mode 0), are skipped.  lane = slot; each warp walks RS_T consecutive outputs of its 32 slots; float32 accumulation.
// ------------------------------------------------------------------------------------------------
constexpr int RS_T = 8;
constexpr int RS_WARPS = 4;
__global__ void __launch_bounds__(32 * RS_WARPS)
audio_resample_kernel(const float* __restrict__ x, long long x_abs0, int slots, const RsCfg* __restrict__ cfg,
                      const int* __restrict__ mode, long long a0, int n, long long af, float* __restrict__ out)
{
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int s = blockIdx.x * 32 + lane;
    if (s >= slots || !mode[s]) return;
    const RsCfg c = cfg[s];
    if (!c.L) return;
    const long long kf = rs_outputs(c, af), k1 = rs_outputs(c, a0 + n);
    const long long step = (long long)gridDim.y * RS_WARPS * RS_T;
    for (long long kb = rs_outputs(c, a0) + ((long long)blockIdx.y * RS_WARPS + w) * RS_T; kb < k1; kb += step) {
        const long long ke = kb + RS_T < k1 ? kb + RS_T : k1;
        for (long long k = kb; k < ke; k++) {
            const long long nmax = k * c.M / c.L;                        // newest input of output k (origin-relative)
            const float* h = c.tab + (k * c.M - nmax * c.L) * c.K;
            const float* xp = x + (c.origin + nmax - x_abs0) * slots + s;
            const int jn = nmax + 1 < c.K ? (int)nmax + 1 : c.K;         // inputs before the origin are zero
            float acc = 0.f;
            for (int j = 0; j < jn; j++) acc = fmaf(__ldg(xp - (ptrdiff_t)j * slots), __ldg(h + j), acc);
            out[(k - kf) * slots + s] = fminf(fmaxf(acc, -1.0f), 1.0f);   // Limit
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Client audio tail (SURVEY 8f-1): Convert(FLOAT -> SHORT) [+ AdpcmEncoder(sync=True)], reference
// csdr/chain/clientaudio.py:12,34.  Wire format pinned by the browser decoder
// (htdocs/lib/AudioEngine.js:449-491): "SYNC", int16 LE step index, int16 LE predictor, then 1001
// data bytes, low nibble first.  One channel per thread; the codec state is sample-serial.
// ------------------------------------------------------------------------------------------------
struct TailState {
    int index, pred, since_sync, have_lo, lo;
};

// mode[s]: 0 = float only, 1 = int16, 2 = int16 + ADPCM with SYNC framing.
// One CTA of four warps per 32 channels, specialised: the codec state is sample-serial per channel (lane = channel) and a lone
// warp issues one instruction every ~2.8 cycles, so everything that is NOT the quantiser recurrence is taken off the encoder
// warp's instruction stream:
//   warps 1..3  fetch tiles of AT_R rows (coalesced 128-byte rows), do Convert(FLOAT, SHORT), store the int16 rows, leave the
//               integers in shared memory; warp 1 also moves the finished tiles' bytes to global memory, one contiguous run
//               per channel;
//   warp 0      only runs ima_encode over the staged integers and drops bytes into shared memory.
// Two tile buffers, named barriers full[b] / empty[b] between the roles.  History: one dependent global load per sample
// (first version) 11.6 ms per C2 block of 20 141 samples per channel; cp.async staging in a single warp 3.1 ms; this form
// see profiles/r2_adpcm_notes.md.
constexpr int AT_R = 32;
constexpr int AT_OB = 36;
__device__ __forceinline__ void at_bar_sync(int id) { asm volatile("barrier.sync %0, 128;" ::"r"(id) : "memory"); }
__device__ __forceinline__ void at_bar_arrive(int id) { asm volatile("barrier.arrive %0, 128;" ::"r"(id) : "memory"); }

__global__ void __launch_bounds__(128)
audio_tail_kernel(const float* __restrict__ in, int slots, int n, const int* __restrict__ mode, TailState* __restrict__ ts,
                  int16_t* __restrict__ s16_out, unsigned char* __restrict__ bytes_out, int* __restrict__ count_out, int cap,
                  const float* __restrict__ rs, const RsCfg* __restrict__ rcfg, long long a0, long long af)
{
    __shared__ uint4 succ[IMA_TABLE_ENTRIES];
    __shared__ int qt[2][AT_R][32];                  // converted samples of a tile
    __shared__ unsigned char obuf[2][32][AT_OB];     // a tile's output bytes per channel (<= AT_R / 2 data + 8 SYNC), padded rows
    __shared__ int onb[2][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    ima_build_table(succ, threadIdx.x, 128);
    const int s = blockIdx.x * 32 + lane;
    const bool live = s < slots;
    const int sc = live ? s : slots - 1;
    const int md = live ? mode[sc] : 0;
    if (__syncthreads_and(md == 0)) return;          // (also publishes the table)
    // this pass's rows of the slot: the n new audio rows, written at feed row a0 - af; or, for a resampled slot
    // (rcfg != nullptr, L != 0), the resampler's outputs of this pass, read from and written at feed output row k0 - kf
    int ns = n;
    long long row0 = a0 - af;
    if (rcfg && rcfg[sc].L) {
        const RsCfg c = rcfg[sc];
        const long long kf = rs_outputs(c, af), k0 = rs_outputs(c, a0);
        ns = (int)(rs_outputs(c, a0 + n) - k0);
        row0 = k0 - kf;
        in = rs + row0 * slots;
    }
    s16_out += row0 * slots;
    const int n_tiles = (__reduce_max_sync(0xffffffffu, ns) + AT_R - 1) / AT_R;     // the same lanes in every warp
    constexpr int FULL = 1, EMPTY = 3;               // barrier ids FULL + b, EMPTY + b
    if (w == 0) {
        // ---------------------------------------------------------------- encoder
        TailState t = ts[sc];
        ImaState cs = ima_state(t.index, t.pred);
        for (int tl = 0; tl < n_tiles; tl++) {
            const int b = tl & 1, valid = min(AT_R, ns - tl * AT_R);
            at_bar_sync(FULL + b);
            int nb = 0;
            if (md == 2) {
                unsigned char* ob = obuf[b][lane];
                const int* q = &qt[b][0][lane];
                auto sync_block = [&]() {
                    if (t.since_sync == 1001) {
                        ob[nb++] = 'S'; ob[nb++] = 'Y'; ob[nb++] = 'N'; ob[nb++] = 'C';
                        ob[nb++] = (unsigned char)(cs.index & 0xff); ob[nb++] = (unsigned char)((cs.index >> 8) & 0xff);
                        ob[nb++] = (unsigned char)(cs.pred & 0xff);  ob[nb++] = (unsigned char)((cs.pred >> 8) & 0xff);
                        t.since_sync = 0;
                    }
                };
                int k = 0;
                if (t.have_lo && valid > 0) {                                    // an odd sample left over from the previous tile
                    const unsigned hi = ima_encode(q[0], cs, succ);
                    ob[nb++] = (unsigned char)((unsigned)t.lo | (hi << 4));
                    t.have_lo = 0; t.since_sync++;
                    k = 1;
                }
#pragma unroll 2
                for (; k + 1 < valid; k += 2) {                                  // whole bytes: low nibble first
                    sync_block();
                    const unsigned lo = ima_encode(q[k * 32], cs, succ);
                    const unsigned hi = ima_encode(q[(k + 1) * 32], cs, succ);
                    ob[nb++] = (unsigned char)(lo | (hi << 4));
                    t.since_sync++;
                }
                if (k < valid) {
                    sync_block();
                    t.lo = (int)ima_encode(q[k * 32], cs, succ);
                    t.have_lo = 1;
                }
            }
            onb[b][lane] = nb;
            at_bar_arrive(EMPTY + b);
        }
        if (live && md != 0) {
            t.index = cs.index; t.pred = cs.pred;
            ts[s] = t;
        }
    } else {
        // ---------------------------------------------------------------- loaders / converters / flusher
        unsigned char* o = bytes_out + (size_t)sc * cap;
        int cnt = count_out[sc];       // append behind earlier passes of the same feed (host zeroes it per feed); warp 1 keeps it
        auto flush = [&](int b) {
            if (w != 1) return;
            const int nb = onb[b][lane];
            if (__any_sync(0xffffffffu, nb > 0)) {
                const unsigned long long dst = (unsigned long long)(o + cnt);
                for (int l = 0; l < 32; l++) {
                    const int nl = __shfl_sync(0xffffffffu, nb, l);
                    if (nl == 0) continue;
                    unsigned char* d = (unsigned char*)__shfl_sync(0xffffffffu, dst, l);
                    if (lane < nl) d[lane] = obuf[b][l][lane];
                }
                cnt += nb;
            }
        };
        for (int tl = 0; tl < n_tiles; tl++) {
            const int b = tl & 1, r0 = tl * AT_R, valid = min(AT_R, ns - r0);
            if (tl >= 2) { at_bar_sync(EMPTY + b); flush(b); }
            float v[(AT_R + 2) / 3];
#pragma unroll
            for (int j = 0; j < (AT_R + 2) / 3; j++) {
                const int k = (w - 1) + 3 * j;
                v[j] = k < valid ? in[(size_t)(r0 + k) * slots + sc] : 0.f;
            }
#pragma unroll
            for (int j = 0; j < (AT_R + 2) / 3; j++) {
                const int k = (w - 1) + 3 * j;
                if (k < valid) {
                    const float x = v[j] * 32767.0f;                             // Convert(FLOAT, SHORT), SURVEY A.12
                    const int q = x > 32767.0f ? 32767 : (x < -32768.0f ? -32768 : __float2int_rz(x));
                    qt[b][k][lane] = q;
                    if (md != 0) s16_out[(size_t)(r0 + k) * slots + sc] = (int16_t)q;
                }
            }
            at_bar_arrive(FULL + b);
        }
        for (int tl = max(0, n_tiles - 2); tl < n_tiles; tl++) {
            const int b = tl & 1;
            at_bar_sync(EMPTY + b);
            flush(b);
        }
        if (w == 1 && live && md != 0) count_out[s] = cnt;
    }
}

// ------------------------------------------------------------------------------------------------
// Per-channel taps: a second reader of a Buffer that the fused chain keeps on the device.  One gather kernel serves both:
//  - the WFM multiplex tap (csdr/chain/analog.py:62,73-76): the WFm chain writes its Limit output into a tap buffer that the
//    audio path and the RDS path (Convert(FLOAT, SHORT) -> redsea) both read.  Here that signal is f1, channel-minor at the IF
//    rate; a slot's (format, run) is ChanCfg::mpx / mpx_run (MpxTapSel).
//  - the demodulated-audio tap: the Buffer the last demodulator stage writes (Agc, or WfmDeemphasis for WFM), which a
//    secondary demodulator (Convert(FLOAT, SHORT) -> a digital-mode decoder) reads beside the client-audio Converter.  Here
//    that signal is f3 at the demodulator rate; a slot's (format, run) comes from a per-parity table beside ChanCfg
//    (AudioTapSel), so that ChanCfg, which the Agc loads whole, keeps its layout.
// The kernel copies the new rows of the tapped slots only, one contiguous run per channel in a staging region, so the D2H
// moves just the tapped bytes (C5: 128 slots; copying all of f1 would be 512 B per IF sample):
//   F32 runs first, run k at byte k * cap * 4;  then S16 runs, run k at byte n_f32 * cap * 4 + k * cap * 2
// (cap is a multiple of 8: every run starts on 16 bytes).  This launch's rows land at rows [r0, r0 + n) of the runs.
// CTA = 32 slots x tiles of MG_R destination rows: warps read 32-slot row segments (128-byte rows) into shared memory, then each
// tapped slot's column leaves as 16-byte stores (F32: 4 rows per lane, all 32 lanes; S16: 8 rows per lane, 16 lanes), read from
// shared memory in a per-lane rotated row order so that neither phase has bank conflicts.
// S16 is Convert(FLOAT, SHORT) exactly as the client audio tail does it (SURVEY A.12).
// ------------------------------------------------------------------------------------------------
constexpr int MG_R = 128;
struct TapFmt {
    int fmt;            // OWRX_MPX_OFF / _F32 / _S16
    int run;            // index of this slot's run among the group's tapped slots of the same format
};
struct MpxTapSel {
    const ChanCfg* __restrict__ cfg;
    __device__ __forceinline__ TapFmt operator()(int s) const { return TapFmt{cfg[s].mpx, cfg[s].mpx_run}; }
};
struct AudioTapSel {
    const TapFmt* __restrict__ tab;
    __device__ __forceinline__ TapFmt operator()(int s) const { return tab[s]; }
};

template <typename Sel>
__global__ void __launch_bounds__(256)
tap_gather_kernel(const float* __restrict__ in, int slots, int n, Sel sel, long long r0, long long cap, int n_f32,
                  unsigned char* __restrict__ out)
{
    __shared__ float tile[MG_R][33];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int s0 = blockIdx.x * 32, s = s0 + lane;
    const unsigned tapped = __ballot_sync(0xffffffffu, s < slots && sel(s).fmt != OWRX_MPX_OFF);
    if (!tapped) return;                                         // the same ballot in every warp: the whole CTA leaves
    const long long t_first = r0 / MG_R, t_end = (r0 + n + MG_R - 1) / MG_R;
    for (long long t = t_first + blockIdx.y; t < t_end; t += gridDim.y) {
        const long long d0 = t * MG_R;                           // destination row of tile row 0
        for (int j = w; j < MG_R; j += 8) {
            const long long i = d0 + j - r0;
            tile[j][lane] = (i >= 0 && i < n && s < slots) ? in[i * slots + s] : 0.f;
        }
        __syncthreads();
        for (int l = w; l < 32; l += 8) {
            if (!((tapped >> l) & 1u)) continue;
            const TapFmt c = sel(s0 + l);
            if (c.fmt == OWRX_MPX_F32) {
                const long long d = d0 + 4 * lane;
                float* o = reinterpret_cast<float*>(out + (size_t)c.run * cap * 4) + d;
                // rows 4*lane + k sit 4*lane banks apart: each group of 8 lanes starts at another k (rot), so the 32 lanes of a read
                // hit 32 different banks; the selects put the values back in row order
                const int rot = lane >> 3;
                float a[4], v[4];
#pragma unroll
                for (int kk = 0; kk < 4; kk++) a[kk] = tile[4 * lane + ((kk + rot) & 3)][l];
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const int i = (k - rot) & 3;
                    v[k] = i == 0 ? a[0] : (i == 1 ? a[1] : (i == 2 ? a[2] : a[3]));
                }
                if (d >= r0 && d + 4 <= r0 + n) {
                    *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
                } else {
#pragma unroll
                    for (int k = 0; k < 4; k++)
                        if (d + k >= r0 && d + k < r0 + n) o[k] = v[k];
                }
            } else if (lane < 16) {
                const long long d = d0 + 8 * lane;
                int16_t* o = reinterpret_cast<int16_t*>(out + (size_t)n_f32 * cap * 4 + (size_t)c.run * cap * 2) + d;
                // the same bank rotation over 8 rows (lanes 0, 4, 8, 12 share banks without it); each converted sample goes straight
                // to its 16-bit place in the two 64-bit halves of the 16-byte store
                const int rot = 2 * (lane >> 2);
                unsigned long long lo = 0ull, hi = 0ull;
#pragma unroll
                for (int kk = 0; kk < 8; kk++) {
                    const int k = (kk + rot) & 7;
                    const float x = tile[8 * lane + k][l] * 32767.0f;                   // Convert(FLOAT, SHORT), SURVEY A.12
                    const int q = x > 32767.0f ? 32767 : (x < -32768.0f ? -32768 : __float2int_rz(x));
                    const unsigned long long b = (unsigned long long)(uint16_t)q << (16 * (k & 3));
                    if (k < 4) lo |= b; else hi |= b;
                }
                if (d >= r0 && d + 8 <= r0 + n) {
                    *reinterpret_cast<uint4*>(o) = make_uint4((unsigned)lo, (unsigned)(lo >> 32), (unsigned)hi, (unsigned)(hi >> 32));
                } else {
                    for (int k = 0; k < 8; k++)
                        if (d + k >= r0 && d + k < r0 + n) o[k] = (int16_t)(uint16_t)((k < 4 ? lo : hi) >> (16 * (k & 3)));
                }
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// Control path (csdr/chain/selector.py:132-166: setFrequencyOffset / setBandpass / setSquelchLevel from websocket threads;
// owrx/dsp.py:96-148: demodulator swaps): nothing a client does may stall the device.  Host setters only record what
// changed; at the next block boundary the changes reach the device as stream-ordered work on the stream that owns the
// state they touch — per-slot state patches (slot_patch_kernel), staged band-pass columns (bp_scatter_kernel), and the
// per-slot tables, which are double-buffered by block parity so that a block still in flight keeps reading its own copy.
// ------------------------------------------------------------------------------------------------
enum : int {
    PATCH_DEMOD = 1,       // fresh demodulator modules: FmDemod's last sample, DcBlock's mean, the de-emphasis IIR
    PATCH_AGC_RESET = 2,   // fresh Agc: gain = agc_gain, hang counter 0
    PATCH_TAIL = 4,        // fresh AdpcmEncoder(sync=True): reset codec, SYNC block first
    PATCH_SQUELCH = 8,     // fresh Squelch: hang counter 0
    PATCH_HISTORY = 16,    // fresh modules everywhere: the slot's column of every stage history is zeroed (host: memset2D)
    PATCH_AGC_GAIN = 32,   // Agc.setInitialGain on a live Agc: gain only
};
struct SlotPatch {
    int slot, flags;
    float agc_gain;
    int pad;
};

__global__ void __launch_bounds__(128)
slot_patch_kernel(const SlotPatch* __restrict__ patches, int n, int mask, ChanState* __restrict__ st, TailState* __restrict__ tail)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const SlotPatch p = patches[i];
    const int f = p.flags & mask, s = p.slot;
    if (f & PATCH_DEMOD) { st[s].fm_last = make_float2(0.f, 0.f); st[s].dc_last = 0.f; st[s].iir = 0.f; }
    if (f & PATCH_SQUELCH) st[s].sq_hang = 0;
    if (f & PATCH_AGC_RESET) { st[s].agc_gain = p.agc_gain; st[s].agc_hang = 0; }
    else if (f & PATCH_AGC_GAIN) st[s].agc_gain = p.agc_gain;
    if (f & PATCH_TAIL) tail[s] = TailState{0, 0, 1001, 0, 0};
}

// staged band-pass columns -> the per-slot tables: stage[i] = Tb taps followed by nH partition-spectrum entries of slot slots[i]
__global__ void __launch_bounds__(256)
bp_scatter_kernel(const float2* __restrict__ stage, const int* __restrict__ slots_list, int Tb, int nH, int S,
                  float2* __restrict__ d_bp, float2* __restrict__ d_bp_H)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    const int i = blockIdx.y;
    if (e >= Tb + nH) return;
    const int slot = slots_list[i];
    const float2 v = stage[(size_t)i * (Tb + nH) + e];
    if (e < Tb) d_bp[(size_t)e * S + slot] = v;
    else d_bp_H[(size_t)(e - Tb) * S + slot] = v;
}

#endif  // OWRX_K3_ONLY

}  // namespace owrx
