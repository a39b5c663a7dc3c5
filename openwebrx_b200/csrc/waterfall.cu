// waterfall.cu — K1/K2: the waterfall FftChain on sm_100a.
//
// Replaces the pycsdr worker chain built by FftChain (reference csdr/chain/fft.py:25-49):
//   Fft(size, every_n_samples) -> LogAveragePower(add_db, fft_size, avg_number) | LogPower(add_db)
//   -> FftSwap(fft_size) -> [FftAdpcm(fft_size)]
// Arithmetic spec: SURVEY.md Appendix A.2-A.5.
//
// Kernels (all hand-written, no cuFFT):
//   wf_fft_kernel<LOG2M>    shared-memory Stockham FFT of M < 4096 points (radix 16,16,R3) with the
//                           Hamming window fused into the load and |X|^2 accumulated over the avg
//                           frames of a line; one CTA per (line, frame-subset).
//   wf_fft2_kernel          the same for 4096 points on packed FP32, two frames per pass.
//   wf_big_kernel<R0>       the four-step FFT of N = R0 x 4096 points (8192 ... 65536), one cluster
//                           of R0 CTAs per frame pair.
//   wf_finalize_kernel      sums the frame-subset partials, 10*log10 + add_db - 10*log10(avg),
//                           half-swap on store, x100 -> int16 truncation + 10-sample pad.
//   wf_adpcm_kernel         IMA-ADPCM, state reset per line, low nibble first.
#include "common.cuh"
#include "fft_small.cuh"
#include "ingress.cuh"
#include "adpcm.cuh"

#include <algorithm>
#include <cmath>
#include <deque>
#include <mutex>
#include <vector>

namespace owrx {

__device__ __forceinline__ int pad16(int i) { return i + (i >> 4); }

struct WfFftParams {
    const float2* src;       // wideband IQ
    const float* window;     // M floats
    const float2* tw2;       // [16][16]   exp(-2 pi i r k / 256)
    const float2* tw3;       // [R3][256]  exp(-2 pi i r k / M)
    float* partial;          // [line][subset][M] partial power sums
    int every_n;             // hop E between frames
    int frames_per_line;     // avg (or 1)
    int subsets;             // S frame-subsets per line
    long long first_frame;   // global frame index of line 0 of this launch
    int units;               // wf_fft2_kernel: (line, subset) units of this launch, handed out through `counter`
    int* counter;            // wf_fft2_kernel: zeroed before the launch
};

// One CTA per (line, frame subset).  M = 2^LOG2M points, T = M/16 threads.
template <int LOG2M>
__global__ void __launch_bounds__((1 << LOG2M) / 16 < 32 ? 32 : (1 << LOG2M) / 16, LOG2M >= 11 ? 2 : 1)
wf_fft_kernel(WfFftParams p)
{
    constexpr int M = 1 << LOG2M;
    constexpr int T = M / 16;
    constexpr int R3 = M / 256;
    constexpr int BUF = M + M / 16;
    extern __shared__ float2 smem[];
    float2* bufA = smem;
    float2* bufB = smem + BUF;
    // |X|^2 accumulators live in shared memory (slot q of thread t at accS[q*T + t]: conflict-free), which keeps
    // the kernel under 128 registers so that two CTAs share an SM and cover each other's barriers and load latency
    float* accS = reinterpret_cast<float*>(smem + 2 * BUF);

    const int tid = threadIdx.x;
    const bool active = tid < T;
    const int subset = blockIdx.x % p.subsets;
    const int line = blockIdx.x / p.subsets;

    const int per = (p.frames_per_line + p.subsets - 1) / p.subsets;
    const int a0 = subset * per;
    const int a1 = min(p.frames_per_line, a0 + per);

    if (active) {
#pragma unroll
        for (int q = 0; q < 16; q++) accS[q * T + tid] = 0.0f;
    }

    // the Hamming window values of this thread's 16 points are the same for every frame of the line: keep them in registers
    float wreg[16];
    if (active) {
#pragma unroll
        for (int r = 0; r < 16; r++) wreg[r] = __ldg(p.window + tid + r * T);
    }

    for (int a = a0; a < a1; a++) {
        float2 v[16];
        const long long frame = (long long)line * p.frames_per_line + a;
        if (active) {
            const float2* x = p.src + (p.first_frame + frame) * (long long)p.every_n;
            if (a + 1 < a1) {
                // pull the next frame (M * 8 bytes = M/16 lines of 128 B: one per thread) towards the SM while this one is
                // transformed: its loads then find L2 instead of HBM
                const char* nx = reinterpret_cast<const char*>(x + p.every_n) + (size_t)tid * 128;
                asm volatile("prefetch.global.L2 [%0];" ::"l"(nx));
            }
#pragma unroll
            for (int r = 0; r < 16; r++) {
                float2 s = __ldg(x + tid + r * T);
                v[r] = make_float2(s.x * wreg[r], s.y * wreg[r]);
            }
            // pass 1: radix 16, Ns = 1
            dft<16>(v);
#pragma unroll
            for (int q = 0; q < 16; q++) bufA[pad16(tid * 16 + slot<16>(q))] = v[q];
        }
        __syncthreads();
        if (active) {
            // pass 2: radix 16, Ns = 16
            const int k = tid & 15;
#pragma unroll
            for (int r = 0; r < 16; r++) v[r] = bufA[pad16(tid + r * T)];
#pragma unroll
            for (int r = 1; r < 16; r++) v[r] = cmul(v[r], __ldg(p.tw2 + r * 16 + k));
            dft<16>(v);
            if (R3 > 1) {
                const int base = (tid >> 4) * 256 + k;
#pragma unroll
                for (int q = 0; q < 16; q++) bufB[pad16(base + slot<16>(q) * 16)] = v[q];
            }
        }
        if (R3 > 1) {
            __syncthreads();
            if (active) {
                // pass 3: radix R3, Ns = 256; 16/R3 butterflies per thread
#pragma unroll
                for (int b = 0; b < 16 / R3; b++) {
                    const int jb = tid + b * T;
#pragma unroll
                    for (int r = 0; r < R3; r++) v[b * R3 + r] = bufB[pad16(jb + r * 256)];
#pragma unroll
                    for (int r = 1; r < R3; r++) v[b * R3 + r] = cmul(v[b * R3 + r], __ldg(p.tw3 + r * 256 + jb));
                    dft<R3>(v + b * R3);
                }
            }
        }
        if (active) {
#pragma unroll
            for (int q = 0; q < 16; q++) accS[q * T + tid] += v[q].x * v[q].x + v[q].y * v[q].y;
        }
    }

    if (active) {
        float* out = p.partial + ((size_t)line * p.subsets + subset) * (size_t)M;
#pragma unroll
        for (int q = 0; q < 16; q++) {
            int bin;
            if (R3 > 1) {
                const int b = q / R3, r = q % R3;
                const int jb = tid + b * T;            // k = jb (< 256), jb >> 8 == 0
                bin = jb + slot<R3>(r) * 256;
            } else {
                bin = tid + slot<16>(q) * 16;          // M == 256
            }
            out[bin] = accS[q * T + tid];
        }
    }
}

// ------------------------------------------------------------------------------------------------
// wf_fft2_kernel — the same Stockham FFT on PACKED FP32 (Blackwell FADD2 / FMUL2 / FFMA2), two frames of a line per pass.
// A thread's 16 points carry BOTH frames: re = (re of frame a, re of frame a + 1), im likewise, so every butterfly add,
// twiddle multiply, window multiply and |X|^2 is one packed instruction for two frames, the twiddles and window values
// are fetched once per pair, and one CTA barrier serves two frames.  Shared memory holds one float4 (re0, re1, im0, im1)
// per point: 128-bit LDS / STS, a quarter-warp per wavefront, conflict-free with the pad-every-16 layout.
// Against wf_fft_kernel (one frame per pass, scalar FP32) the issued instructions per frame roughly halve; what remains is
// the L1 / shared-memory datapath: 2 exchanges x (write + read) x 8 bytes per point per frame, plus the frame itself.
// ------------------------------------------------------------------------------------------------
struct C2 {
    float2 re, im;
};
#define OWRX_P2(x) make_float2((x), (x))
__device__ __forceinline__ float2 neg2(float2 a) { return make_float2(-a.x, -a.y); }          // folds into operand modifiers
__device__ __forceinline__ C2 c2add(C2 a, C2 b) { return C2{__fadd2_rn(a.re, b.re), __fadd2_rn(a.im, b.im)}; }
__device__ __forceinline__ C2 c2sub(C2 a, C2 b) { return C2{__fadd2_rn(a.re, neg2(b.re)), __fadd2_rn(a.im, neg2(b.im))}; }
__device__ __forceinline__ C2 c2mul(C2 a, float c, float s)                                   // a * (c + i s), both frames
{
    C2 r;
    r.re = __ffma2_rn(a.re, OWRX_P2(c), __fmul2_rn(a.im, OWRX_P2(-s)));
    r.im = __ffma2_rn(a.re, OWRX_P2(s), __fmul2_rn(a.im, OWRX_P2(c)));
    return r;
}
__device__ __forceinline__ void c2dft2(C2& a, C2& b)
{
    const C2 t = a;
    a = c2add(t, b);
    b = c2sub(t, b);
}
__device__ __forceinline__ void c2dft4(C2& a, C2& b, C2& c, C2& d)
{
    const C2 t0 = c2add(a, c), t1 = c2sub(a, c), t2 = c2add(b, d), bd = c2sub(b, d);
    // t3 = -i (b - d) = (bd.im, -bd.re)
    a = c2add(t0, t2);
    c = c2sub(t0, t2);
    b = C2{__fadd2_rn(t1.re, bd.im), __fadd2_rn(t1.im, neg2(bd.re))};
    d = C2{__fadd2_rn(t1.re, neg2(bd.im)), __fadd2_rn(t1.im, bd.re)};
}
// v * W8^1 = ((re + im), (im - re)) / sqrt 2;   v * W8^3 = ((im - re), -(re + im)) / sqrt 2;   v * W4^1 = (im, -re)
__device__ __forceinline__ C2 c2w8_1(C2 v) { return C2{__fmul2_rn(__fadd2_rn(v.re, v.im), OWRX_P2(OWRX_SQRT1_2)), __fmul2_rn(__fadd2_rn(v.im, neg2(v.re)), OWRX_P2(OWRX_SQRT1_2))}; }
__device__ __forceinline__ C2 c2w8_3(C2 v) { return C2{__fmul2_rn(__fadd2_rn(v.im, neg2(v.re)), OWRX_P2(OWRX_SQRT1_2)), __fmul2_rn(__fadd2_rn(v.re, v.im), OWRX_P2(-OWRX_SQRT1_2))}; }
__device__ __forceinline__ C2 c2mi(C2 v) { return C2{v.im, neg2(v.re)}; }
__device__ __forceinline__ void c2dft16(C2* v)
{
    // same index algebra as dft<16> (fft_small.cuh): n = 4 n1 + n2, m = m1 + 4 m2
#pragma unroll
    for (int n2 = 0; n2 < 4; n2++) c2dft4(v[n2], v[4 + n2], v[8 + n2], v[12 + n2]);
    v[5] = c2mul(v[5], OWRX_COS_PI_8, -OWRX_SIN_PI_8);
    v[6] = c2w8_1(v[6]);
    v[7] = c2mul(v[7], OWRX_SIN_PI_8, -OWRX_COS_PI_8);
    v[9] = c2w8_1(v[9]);
    v[10] = c2mi(v[10]);
    v[11] = c2w8_3(v[11]);
    v[13] = c2mul(v[13], OWRX_SIN_PI_8, -OWRX_COS_PI_8);
    v[14] = c2w8_3(v[14]);
    v[15] = c2mul(v[15], -OWRX_COS_PI_8, OWRX_SIN_PI_8);
#pragma unroll
    for (int m1 = 0; m1 < 4; m1++) c2dft4(v[4 * m1], v[4 * m1 + 1], v[4 * m1 + 2], v[4 * m1 + 3]);
}

// M = 4096 points: 256 threads x 16 points, radix 16 x 16 x 16; one CTA per (line, frame subset).
__global__ void __launch_bounds__(256, 2)
wf_fft2_kernel(WfFftParams p)
{
    constexpr int M = 4096, T = 256;
    extern __shared__ float4 smem4[];                       // [M + M / 16]
    __shared__ int s_next;
    const int tid = threadIdx.x;
    const int k = tid & 15;
    const int base2 = (tid >> 4) * 256 + k;
    const int per = (p.frames_per_line + p.subsets - 1) / p.subsets;
    // Persistent CTAs take (line, subset) units from a global counter: the grid is one resident wave, and an SM that is late
    // (or held by the side-stream ADPCM encoder) simply takes fewer units — no wave quantisation.
    for (int cur = blockIdx.x; cur < p.units;) {
    const int subset = cur % p.subsets;
    const int line = cur / p.subsets;
    const int a0 = subset * per;
    const int a1 = min(p.frames_per_line, a0 + per);
    if (tid == 0) s_next = atomicAdd(p.counter, 1) + (int)gridDim.x;

    float acc[16];
#pragma unroll
    for (int q = 0; q < 16; q++) acc[q] = 0.0f;

    for (int a = a0; a < a1; a += 2) {
        const bool two = a + 1 < a1;
        C2 v[16];
        const long long frame = (long long)line * p.frames_per_line + a;
        const float2* x0 = p.src + (p.first_frame + frame) * (long long)p.every_n;
        const float2* x1 = x0 + p.every_n;
        if (a + 2 < a1) {
            // pull the next pair of frames towards L2 while this one is transformed (one 128-byte line per thread and frame)
            const char* nx = reinterpret_cast<const char*>(x1 + p.every_n) + (size_t)tid * 128;
            asm volatile("prefetch.global.L2 [%0];" ::"l"(nx));
            if (a + 3 < a1) asm volatile("prefetch.global.L2 [%0];" ::"l"(nx + (size_t)p.every_n * 8));
        }
#pragma unroll
        for (int r = 0; r < 16; r++) {
            const float2 s0 = __ldg(x0 + tid + r * T);
            const float2 s1 = two ? __ldg(x1 + tid + r * T) : make_float2(0.f, 0.f);
            const float w = __ldg(p.window + tid + r * T);
            v[r].re = __fmul2_rn(make_float2(s0.x, s1.x), OWRX_P2(w));
            v[r].im = __fmul2_rn(make_float2(s0.y, s1.y), OWRX_P2(w));
        }
        // pass 1: radix 16, Ns = 1
        c2dft16(v);
        __syncthreads();                                    // the previous pair's pass-3 reads are done
#pragma unroll
        for (int q = 0; q < 16; q++) smem4[pad16(tid * 16 + slot<16>(q))] = make_float4(v[q].re.x, v[q].re.y, v[q].im.x, v[q].im.y);
        __syncthreads();
        // pass 2: radix 16, Ns = 16
#pragma unroll
        for (int r = 0; r < 16; r++) {
            const float4 t = smem4[pad16(tid + r * T)];
            v[r].re = make_float2(t.x, t.y);
            v[r].im = make_float2(t.z, t.w);
        }
#pragma unroll
        for (int r = 1; r < 16; r++) {
            const float2 w = __ldg(p.tw2 + r * 16 + k);
            v[r] = c2mul(v[r], w.x, w.y);
        }
        c2dft16(v);
        __syncthreads();                                    // every pass-2 read is done: the buffer is reused in place
#pragma unroll
        for (int q = 0; q < 16; q++) smem4[pad16(base2 + slot<16>(q) * 16)] = make_float4(v[q].re.x, v[q].re.y, v[q].im.x, v[q].im.y);
        __syncthreads();
        // pass 3: radix 16, Ns = 256
#pragma unroll
        for (int r = 0; r < 16; r++) {
            const float4 t = smem4[pad16(tid + r * 256)];
            v[r].re = make_float2(t.x, t.y);
            v[r].im = make_float2(t.z, t.w);
        }
#pragma unroll
        for (int r = 1; r < 16; r++) {
            const float2 w = __ldg(p.tw3 + r * 256 + tid);
            v[r] = c2mul(v[r], w.x, w.y);
        }
        c2dft16(v);
#pragma unroll
        for (int q = 0; q < 16; q++) {
            const float2 pw = __ffma2_rn(v[q].im, v[q].im, __fmul2_rn(v[q].re, v[q].re));
            acc[q] += pw.x + pw.y;
        }
    }
    float* out = p.partial + ((size_t)line * p.subsets + subset) * (size_t)M;
#pragma unroll
    for (int q = 0; q < 16; q++) out[tid + slot<16>(q) * 256] = acc[q];
    __syncthreads();                                        // s_next is visible; every read of the shared buffer is done
    cur = s_next;
    }
}

// ------------------------------------------------------------------------------------------------
// wf_big_kernel<R0> — the whole four-step FFT of N = R0 x 4096 points (8192 ... 65536) in ONE persistent kernel.
// A thread-block CLUSTER of R0 CTAs (16 for 65536 points: the non-portable size, two CTAs per SM) owns a frame pair at a time:
//   stage A  every CTA takes 4096 / R0 columns (one per thread for R0 = 16): windowed loads of both frames, packed radix-R0
//            column DFT, W_N twiddle, and writes its columns of all R0 rows into the cluster's PRIVATE scratch
//            Y[row][4096] (float4 = both frames);
//   cluster barrier (release / acquire);
//   stage B  every CTA transforms ONE row: the packed radix 16 x 16 x 16 passes of wf_fft2_kernel, |X|^2 in registers.
// The scratch is double-buffered, so one cluster barrier per frame pair orders everything, and it is only 2 x R0 x 64 KB
// per cluster (~40 MB for all resident clusters of a 65536-point run): it is rewritten every frame pair and stays in L2.
// The separate column-pass kernel it replaces wrote every transformed frame to HBM and read it back: 3 x the input bytes.
// Two CTAs of DIFFERENT clusters share an SM, so one cluster's barrier wait is the other's compute time.
// ------------------------------------------------------------------------------------------------
template <int R> __device__ __forceinline__ void c2dft(C2* v);
template <> __device__ __forceinline__ void c2dft<2>(C2* v) { c2dft2(v[0], v[1]); }
template <> __device__ __forceinline__ void c2dft<4>(C2* v) { c2dft4(v[0], v[1], v[2], v[3]); }
template <> __device__ __forceinline__ void c2dft<8>(C2* v)
{
    c2dft4(v[0], v[2], v[4], v[6]);
    c2dft4(v[1], v[3], v[5], v[7]);
    v[3] = c2w8_1(v[3]);
    v[5] = c2mi(v[5]);
    v[7] = c2w8_3(v[7]);
    c2dft2(v[0], v[1]);
    c2dft2(v[2], v[3]);
    c2dft2(v[4], v[5]);
    c2dft2(v[6], v[7]);
}
template <> __device__ __forceinline__ void c2dft<16>(C2* v) { c2dft16(v); }

struct WfBigParams {
    const float2* iq;        // wideband IQ
    const float* window;     // N floats
    const float2* twn;       // [R0][4096] exp(-2 pi i k1 n2 / N)
    const float2* tw2;       // [16][16]
    const float2* tw3;       // [16][256]
    float4* y;               // [cluster][2][R0][4096] scratch
    float* partial;          // [line][subset][N]
    int every_n, frames_per_line, subsets, n, units;
    long long first_frame;
};

__device__ __forceinline__ void team_sync(int team) { asm volatile("bar.sync %0, 256;" ::"r"(team + 1) : "memory"); }
__device__ __forceinline__ void cluster_sync_all()
{
    asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
__device__ __forceinline__ float4 ldcg4(const float4* p)
{
    float4 v;
    asm volatile("ld.global.cg.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}

template <int R0>
__global__ void __launch_bounds__(256, 2)
wf_big_kernel(WfBigParams p)
{
    constexpr int M = 4096;
    constexpr int CS = R0;                                  // CTAs per cluster: one row each
    extern __shared__ float4 smem4[];                       // [M + M / 16]
    const int tid = threadIdx.x;
    unsigned crank;
    asm("mov.u32 %0, %%cluster_ctarank;" : "=r"(crank));
    const int cid = blockIdx.x / CS, n_clusters = gridDim.x / CS;
    float4* const ybase = p.y + (size_t)cid * 2 * R0 * M;
    const int k = tid & 15;
    const int base2 = (tid >> 4) * 256 + k;
    const int k1 = (int)crank;                              // the row this CTA transforms
    constexpr int COLS = M / CS / 256;                      // columns a thread transforms in stage A (1 for R0 = 16)
    const int per = (p.frames_per_line + p.subsets - 1) / p.subsets;
    unsigned pc = 0;                                        // frame pairs done by this cluster: scratch parity

    for (int unit = cid; unit < p.units; unit += n_clusters) {
        const int subset = unit % p.subsets, line = unit / p.subsets;
        const int a0 = subset * per, a1 = min(p.frames_per_line, a0 + per);
        float acc[16];
#pragma unroll
        for (int q = 0; q < 16; q++) acc[q] = 0.0f;
        for (int a = a0; a < a1; a += 2, pc++) {
            const bool two = a + 1 < a1;
            float4* const y = ybase + (size_t)(pc & 1) * R0 * M;
            const long long frame = (long long)line * p.frames_per_line + a;
            const float2* x0 = p.iq + (p.first_frame + frame) * (long long)p.every_n;
            const float2* x1 = x0 + p.every_n;
            // ---- stage A: column pass over this CTA's M / CS columns
#pragma unroll 1
            for (int c = 0; c < COLS; c++) {
                const int n2 = (int)crank * (M / CS) + c * 256 + tid;
                C2 u[R0];
#pragma unroll
                for (int n1 = 0; n1 < R0; n1++) {
                    const float2 s0 = __ldg(x0 + n2 + M * n1);
                    const float2 s1 = two ? __ldg(x1 + n2 + M * n1) : make_float2(0.f, 0.f);
                    const float w = __ldg(p.window + n2 + M * n1);
                    u[n1].re = __fmul2_rn(make_float2(s0.x, s1.x), OWRX_P2(w));
                    u[n1].im = __fmul2_rn(make_float2(s0.y, s1.y), OWRX_P2(w));
                }
                if (a + 2 < a1) {
                    // the next frame pair's samples of this column go to L2 while this pair is transformed (8 threads share a
                    // 128-byte line: one request per line)
                    if ((tid & 15) == 0) {
#pragma unroll
                        for (int n1 = 0; n1 < R0; n1++) {
                            asm volatile("prefetch.global.L2 [%0];" ::"l"(x1 + p.every_n + n2 + M * n1));
                            if (a + 3 < a1) asm volatile("prefetch.global.L2 [%0];" ::"l"(x1 + 2 * (size_t)p.every_n + n2 + M * n1));
                        }
                    }
                }
                c2dft<R0>(u);
#pragma unroll
                for (int q = 0; q < R0; q++) {
                    const int row = slot<R0>(q);
                    C2 o = u[q];
                    if (row > 0) {
                        const float2 w = __ldg(p.twn + row * M + n2);
                        o = c2mul(o, w.x, w.y);
                    }
                    y[(size_t)row * M + n2] = make_float4(o.re.x, o.re.y, o.im.x, o.im.y);
                }
            }
            cluster_sync_all();                             // every row of this frame pair is in the scratch
            // ---- stage B: this CTA's row, packed radix 16 x 16 x 16
            C2 v[16];
            const float4* yr = y + (size_t)k1 * M;
#pragma unroll
            for (int r = 0; r < 16; r++) {
                const float4 t = ldcg4(yr + tid + r * 256);
                v[r].re = make_float2(t.x, t.y);
                v[r].im = make_float2(t.z, t.w);
            }
            c2dft16(v);
            __syncthreads();                                // the previous pair's pass-3 reads are done
#pragma unroll
            for (int q = 0; q < 16; q++) smem4[pad16(tid * 16 + slot<16>(q))] = make_float4(v[q].re.x, v[q].re.y, v[q].im.x, v[q].im.y);
            __syncthreads();
#pragma unroll
            for (int r = 0; r < 16; r++) {
                const float4 t = smem4[pad16(tid + r * 256)];
                v[r].re = make_float2(t.x, t.y);
                v[r].im = make_float2(t.z, t.w);
            }
#pragma unroll
            for (int r = 1; r < 16; r++) {
                const float2 w = __ldg(p.tw2 + r * 16 + k);
                v[r] = c2mul(v[r], w.x, w.y);
            }
            c2dft16(v);
            __syncthreads();
#pragma unroll
            for (int q = 0; q < 16; q++) smem4[pad16(base2 + slot<16>(q) * 16)] = make_float4(v[q].re.x, v[q].re.y, v[q].im.x, v[q].im.y);
            __syncthreads();
#pragma unroll
            for (int r = 0; r < 16; r++) {
                const float4 t = smem4[pad16(tid + r * 256)];
                v[r].re = make_float2(t.x, t.y);
                v[r].im = make_float2(t.z, t.w);
            }
#pragma unroll
            for (int r = 1; r < 16; r++) {
                const float2 w = __ldg(p.tw3 + r * 256 + tid);
                v[r] = c2mul(v[r], w.x, w.y);
            }
            c2dft16(v);
#pragma unroll
            for (int q = 0; q < 16; q++) {
                const float2 pw = __ffma2_rn(v[q].im, v[q].im, __fmul2_rn(v[q].re, v[q].re));
                acc[q] += pw.x + pw.y;
            }
        }
        float* out = p.partial + ((size_t)line * p.subsets + subset) * (size_t)p.n;
#pragma unroll
        for (int q = 0; q < 16; q++) out[(size_t)k1 + (size_t)R0 * (tid + slot<16>(q) * 256)] = acc[q];
    }
    cluster_sync_all();                                     // no CTA of the cluster exits while another may still arrive
}

// Spectral-subtraction noise filter (BASELINE config 4: "65536-pt high-zoom waterfall ... with spectral-subtraction noise
// filter").  SPEC-DEFINED — the reference has no waterfall noise filter (SURVEY 8d C4); same arithmetic as the oracle's
// oc_wf_noise_filter.  One thread per bin walks the lines of the batch in order (the floor estimate is a recurrence across
// lines): sums the frame-subset partials, updates N = first ? P : min(P, N (1 + growth)), and leaves
// P' = max(P - alpha N, beta P) in subset 0 (the other subsets are zeroed) for wf_finalize_kernel.
__global__ void __launch_bounds__(256)
wf_noise_kernel(float* __restrict__ partial, int subsets, int n, size_t n_lines, float* __restrict__ noise, int first, float alpha,
                float beta, float growth)
{
    const int bin = blockIdx.x * blockDim.x + threadIdx.x;
    if (bin >= n) return;
    float nf = first ? 0.0f : noise[bin];
    for (size_t line = 0; line < n_lines; line++) {
        float* ps = partial + line * (size_t)subsets * (size_t)n + bin;
        float s = 0.0f;
        for (int k = 0; k < subsets; k++) { s += ps[(size_t)k * n]; if (k) ps[(size_t)k * n] = 0.0f; }
        nf = (first && line == 0) ? s : fminf(s, nf * (1.0f + growth));
        ps[0] = fmaxf(s - alpha * nf, beta * s);
    }
    noise[bin] = nf;
}

// sums partials, log, swap, optional quantise.  One thread per output position.
__global__ void __launch_bounds__(256)
wf_finalize_kernel(const float* __restrict__ partial, int subsets, int n, float corr, size_t n_lines,
                   float* __restrict__ db_out, int16_t* __restrict__ s16_out)
{
    const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= n_lines * (size_t)n) return;
    const size_t line = gid / (size_t)n;
    const int i = (int)(gid % (size_t)n);
    const int bin = (i + n / 2) & (n - 1);                     // FftSwap: out[i] = in[(i + N/2) mod N]
    const float* ps = partial + line * (size_t)subsets * (size_t)n + bin;
    float s = 0.0f;
    for (int k = 0; k < subsets; k++) s += ps[(size_t)k * n];
    const float db = 10.0f * log10f(s) + corr;
    if (db_out) db_out[gid] = db;
    if (s16_out) {
        // FftAdpcm quantiser (SURVEY A.5): (int16)(dB * 100), C truncation, clamped
        float v = db * 100.0f;
        int q;
        if (!(v > -32768.0f)) q = -32768;
        else if (v > 32767.0f) q = 32767;
        else q = __float2int_rz(v);
        int16_t* row = s16_out + line * (size_t)(n + 10);
        row[10 + i] = (int16_t)q;
        if (i == 0) {
#pragma unroll
            for (int k = 0; k < 10; k++) row[k] = (int16_t)q;  // COMPRESS_FFT_PAD_N copies of s[0]
        }
    }
}

// FftAdpcm encoder, warp-cooperative: a warp owns 32 lines (one per lane: the codec state is strictly
// sequential within a line, lines are independent and reset per line).  Each iteration the warp stages a
// 64-sample chunk of all 32 lines through shared memory with coalesced 128-byte row loads (cp.async, one chunk
// ahead of the encoder), every lane encodes its own line's chunk from padded (conflict-free) shared memory, and
// the 32 output bytes per line leave through shared memory as one 32-byte sector per line.
// Four such warps per CTA, one per scheduler of the SM (a lone warp issues at ~0.35 IPC, so they do not slow each other down):
// the encoder then holds a quarter of the SMs it would with one warp per CTA — every SM it holds is one the FFT pass of the
// next batch does not get (C1: 5 SMs instead of 19 for 592 lines).
constexpr int ADPCM_CH = 64;
constexpr int ADPCM_WARPS = 4;
__global__ void __launch_bounds__(32 * ADPCM_WARPS)
wf_adpcm_kernel(const int16_t* __restrict__ s16, uint8_t* __restrict__ out, int n_samples, size_t n_lines)
{
    __shared__ uint4 cand[IMA_TABLE_ENTRIES];
    __shared__ unsigned tile_all[ADPCM_WARPS][2][32][ADPCM_CH / 2 + 1];
    __shared__ unsigned otile_all[ADPCM_WARPS][32][ADPCM_CH / 8 + 1];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    ima_build_table(cand, threadIdx.x, 32 * ADPCM_WARPS);
    __syncthreads();
    unsigned (*tile)[32][ADPCM_CH / 2 + 1] = tile_all[wid];
    unsigned (*otile)[ADPCM_CH / 8 + 1] = otile_all[wid];
    const size_t line0 = ((size_t)blockIdx.x * ADPCM_WARPS + wid) * 32;
    if (line0 >= n_lines) return;
    const int nl = (int)min((size_t)32, n_lines - line0);
    const int n_chunks = (n_samples + ADPCM_CH - 1) / ADPCM_CH;
    auto stage = [&](int chunk, int buf) {
        const int c0 = chunk * ADPCM_CH;
        if (chunk < n_chunks && c0 + 2 * lane < n_samples) {
            for (int l = 0; l < nl; l++) {
                const unsigned dst = (unsigned)__cvta_generic_to_shared(&tile[buf][l][lane]);
                const int16_t* src = s16 + (line0 + l) * (size_t)n_samples + c0 + 2 * lane;
                asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(dst), "l"(src));
            }
        }
        asm volatile("cp.async.commit_group;\n" ::);
    };
    stage(0, 0);
    __syncwarp();
    ImaState cs = ima_state(0, 0);
    for (int chunk = 0; chunk < n_chunks; chunk++) {
        const int buf = chunk & 1;
        const int c0 = chunk * ADPCM_CH;
        const int valid = min(ADPCM_CH, n_samples - c0);          // even
        stage(chunk + 1, buf ^ 1);
        asm volatile("cp.async.wait_group 1;\n" ::);
        __syncwarp();
        if (lane < nl) {
            for (int w4 = 0; w4 < valid / 8; w4++) {
                unsigned packed = 0;
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const unsigned v = tile[buf][lane][4 * w4 + k];
                    const unsigned lo = ima_encode((int)(short)(v & 0xffffu), cs, cand);
                    const unsigned hi = ima_encode((int)(short)(v >> 16), cs, cand);
                    packed |= (lo | (hi << 4)) << (8 * k);
                }
                otile[lane][w4] = packed;
            }
            // trailing samples of the last chunk (valid is even, not necessarily a multiple of 8)
            const int done = (valid / 8) * 8;
            if (done < valid) {
                unsigned packed = 0;
                for (int k = 0; k < (valid - done) / 2; k++) {
                    const unsigned v = tile[buf][lane][done / 2 + k];
                    const unsigned lo = ima_encode((int)(short)(v & 0xffffu), cs, cand);
                    const unsigned hi = ima_encode((int)(short)(v >> 16), cs, cand);
                    packed |= (lo | (hi << 4)) << (8 * k);
                }
                otile[lane][valid / 8] = packed;
            }
        }
        __syncwarp();
        const unsigned char* ob = reinterpret_cast<const unsigned char*>(&otile[0][0]);
        for (int l = 0; l < nl; l++)
            if (lane < valid / 2) out[(line0 + l) * (size_t)(n_samples / 2) + c0 / 2 + lane] = ob[l * (ADPCM_CH / 8 + 1) * 4 + lane];
        __syncwarp();
    }
}

}  // namespace owrx

// ================================================================================================
// host side
// ================================================================================================
using namespace owrx;

struct owrx_wf {
    int device = 0, sm_count = 0;
    uint64_t h2d_pinned = 0, h2d_pageable = 0;                 // host-path ingress bytes by source memory kind
    int n = 0, every_n = 0, avg = 0, compression = 0;
    float add_db = 0.0f;
    int m = 0, log2m = 0, r0 = 1;
    cudaStream_t stream = nullptr;
    float* d_window = nullptr;
    float2 *d_tw2 = nullptr, *d_tw3 = nullptr, *d_twn = nullptr;
    // scratch
    float* d_partial = nullptr; size_t partial_cap = 0;
    int* d_counter = nullptr;                                  // work counter of the persistent FFT kernel
    float4* d_ybig = nullptr; size_t ybig_cap = 0;            // wf_big_kernel: per-cluster row scratch (L2-resident)
    int big_clusters = 0;                                      // clusters of the fused kernel the device keeps resident
    int16_t* d_s16 = nullptr;   size_t s16_cap = 0;
    // pipelined mode: the (latency-bound, one warp per 32 lines) ADPCM pass of batch i runs on a high-priority side
    // stream beside the FFT pass of batch i+1; the int16 scratch is double-buffered
    bool pipelined = false;
    cudaStream_t side = nullptr;
    int16_t* d_s16_alt = nullptr; size_t s16_alt_cap = 0;
    cudaEvent_t fin_done = nullptr, adpcm_done[2] = {nullptr, nullptr};
    int s16_cur = 0;
    // streaming
    float2* d_in = nullptr;     size_t in_cap = 0, in_fill = 0, skip = 0;
    float2* d_in_alt = nullptr;
    uint8_t* d_out = nullptr;   size_t out_cap = 0;
    uint8_t* h_out = nullptr;   size_t h_out_cap = 0;
    std::deque<std::vector<uint8_t>> queue;
    std::mutex mu;
    // spec-defined noise filter (owrx_wf_set_noise_filter): per-bin floor estimate carried across lines
    bool nf_on = false, nf_primed = false;
    float nf_alpha = 0.f, nf_beta = 0.f, nf_growth = 0.f;
    float* d_noise = nullptr;
    unsigned char* d_raw = nullptr; size_t raw_cap = 0;      // staging for raw (non-float) ingress (owrx_wf_feed_fmt)
};

static size_t wf_line_bytes(const owrx_wf* wf)
{
    return wf->compression == OWRX_COMPRESSION_ADPCM ? (size_t)(wf->n + 10) / 2 : (size_t)wf->n * 4;
}

static size_t wf_lines_for(const owrx_wf* wf, size_t n_samples)
{
    if (wf->every_n <= 0 || n_samples < (size_t)wf->n) return 0;
    const size_t frames = (n_samples - (size_t)wf->n) / (size_t)wf->every_n + 1;
    return frames / (size_t)(wf->avg > 0 ? wf->avg : 1);
}

template <typename T> static int grow(T** ptr, size_t* cap, size_t need)
{
    if (need <= *cap) return OWRX_OK;
    if (*ptr) cudaFree(*ptr);
    *ptr = nullptr;
    *cap = 0;
    OWRX_CUDA(cudaMalloc((void**)ptr, need * sizeof(T)));
    *cap = need;
    return OWRX_OK;
}

template <int LOG2M> static int launch_fft(const WfFftParams& p, size_t units, cudaStream_t st)
{
    constexpr int M = 1 << LOG2M;
    constexpr int threads = M / 16 < 32 ? 32 : M / 16;
    const size_t smem = 2 * (size_t)(M + M / 16) * sizeof(float2) + (size_t)M * sizeof(float);
    OWRX_CUDA(cudaFuncSetAttribute(wf_fft_kernel<LOG2M>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    wf_fft_kernel<LOG2M><<<(unsigned)units, threads, smem, st>>>(p);
    OWRX_LAUNCH_CHECK();
    return OWRX_OK;
}

static int launch_fft2(const WfFftParams& p, size_t units, int sm_count, cudaStream_t st)
{
    const size_t smem = (size_t)(4096 + 4096 / 16) * sizeof(float4);
    OWRX_CUDA(cudaFuncSetAttribute(wf_fft2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    OWRX_CUDA(cudaMemsetAsync(p.counter, 0, sizeof(int), st));
    const unsigned grid = (unsigned)std::min<size_t>(units, (size_t)2 * sm_count);       // 2 CTAs per SM (128 registers, 70 KB)
    wf_fft2_kernel<<<grid, 256, smem, st>>>(p);
    OWRX_LAUNCH_CHECK();
    return OWRX_OK;
}

// the fused four-step kernel: clusters of R0 / 2 CTAs, as many clusters as the device keeps resident at once
template <int R0> static int launch_big(owrx_wf* wf, WfBigParams& p, cudaStream_t st)
{
    constexpr int CS = R0;
    const size_t smem = (size_t)(4096 + 4096 / 16) * sizeof(float4);
    OWRX_CUDA(cudaFuncSetAttribute(wf_big_kernel<R0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (CS > 8) OWRX_CUDA(cudaFuncSetAttribute(wf_big_kernel<R0>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg{};
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CS; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.blockDim = dim3(256); cfg.dynamicSmemBytes = smem; cfg.stream = st; cfg.attrs = attr; cfg.numAttrs = 1;
    if (wf->big_clusters <= 0) {
        cfg.gridDim = dim3((unsigned)(2 * wf->sm_count / CS * CS));
        int nc = 0;
        OWRX_CUDA(cudaOccupancyMaxActiveClusters(&nc, wf_big_kernel<R0>, &cfg));
        if (nc <= 0) return fail(OWRX_E_CUDA, "no resident cluster of %d CTAs for the fused four-step FFT", CS);
        static const int cap = getenv("OWRX_WF_CLUSTERS") ? atoi(getenv("OWRX_WF_CLUSTERS")) : 0;
        wf->big_clusters = cap > 0 ? std::min(cap, nc) : nc;
        if (getenv("OWRX_TRACE")) fprintf(stderr, "[owrx wf] fused four-step kernel: clusters of %d CTAs, %d resident at once (%d SMs)\n", CS, nc, wf->sm_count);
    }
    const int n_clusters = (int)std::min<long long>(wf->big_clusters, p.units);
    const size_t y_need = (size_t)wf->big_clusters * 2 * R0 * 4096;
    if (y_need > wf->ybig_cap) {
        OWRX_CUDA(cudaStreamSynchronize(st));
        cudaFree(wf->d_ybig); wf->d_ybig = nullptr; wf->ybig_cap = 0;
        OWRX_CUDA(cudaMalloc((void**)&wf->d_ybig, y_need * sizeof(float4)));
        wf->ybig_cap = y_need;
    }
    p.y = wf->d_ybig;
    cfg.gridDim = dim3((unsigned)(n_clusters * CS));
    OWRX_CUDA(cudaLaunchKernelEx(&cfg, wf_big_kernel<R0>, p));
    OWRX_LAUNCH_CHECK();
    return OWRX_OK;
}

static int wf_run_lines(owrx_wf* wf, const float2* iq_dev, size_t lines, uint8_t* out_dev, float* db_dev, int16_t* s16_dev,
                        cudaStream_t st)
{
    const int fpl = wf->avg > 0 ? wf->avg : 1;
    const int n = wf->n;
    int subsets = 1;
    if (wf->r0 > 1) {
        // fused four-step kernel: units are (line, subset), dealt round-robin to ~2 sm_count / r0 clusters
        const size_t clusters = std::max<size_t>(1, (size_t)2 * wf->sm_count / (size_t)wf->r0);
        subsets = (int)std::min<size_t>((size_t)std::max(1, std::min(fpl / 12, 8)), std::max<size_t>(1, (8 * clusters + lines - 1) / lines));
    } else {
        // frame subsets: enough CTAs to cover the SMs twice when few lines are in flight
        if (lines < (size_t)2 * wf->sm_count)
            subsets = (int)std::min<size_t>((size_t)std::min(fpl, 8), ((size_t)2 * wf->sm_count + lines - 1) / lines);
        // the persistent packed kernel balances through its work counter: aim at ~8 units per resident CTA, each of at least
        // 8 frame pairs (a subset costs one more partial-sum row for wf_finalize_kernel to add)
        if (wf->m == 4096 && lines < (size_t)16 * wf->sm_count)
            subsets = (int)std::max<size_t>(subsets, std::min<size_t>((size_t)std::max(1, std::min(fpl / 16, 8)),
                                                                      ((size_t)16 * wf->sm_count + lines - 1) / lines));
    }
    int rc;
    if ((rc = grow(&wf->d_partial, &wf->partial_cap, lines * (size_t)subsets * (size_t)n)) != OWRX_OK) return rc;
    const size_t units = lines * (size_t)subsets;
    if (units > (size_t)0x7fffffff) return fail(OWRX_E_INVALID, "batch too large");

    if (wf->r0 == 1) {
        WfFftParams p;
        p.src = iq_dev; p.window = wf->d_window; p.tw2 = wf->d_tw2; p.tw3 = wf->d_tw3; p.partial = wf->d_partial;
        p.every_n = wf->every_n; p.frames_per_line = fpl; p.subsets = subsets; p.first_frame = 0;
        p.units = (int)units; p.counter = wf->d_counter;
        switch (wf->log2m) {
        case 8:  rc = launch_fft<8>(p, units, st); break;
        case 9:  rc = launch_fft<9>(p, units, st); break;
        case 10: rc = launch_fft<10>(p, units, st); break;
        case 11: rc = launch_fft<11>(p, units, st); break;
        case 12: rc = launch_fft2(p, units, wf->sm_count, st); break;
        default: return fail(OWRX_E_INVALID, "unsupported fft size");
        }
        if (rc != OWRX_OK) return rc;
    } else {
        WfBigParams b;
        b.iq = iq_dev; b.window = wf->d_window; b.twn = wf->d_twn; b.tw2 = wf->d_tw2; b.tw3 = wf->d_tw3; b.y = nullptr;
        b.partial = wf->d_partial; b.every_n = wf->every_n; b.frames_per_line = fpl; b.subsets = subsets; b.n = n;
        b.units = (int)units; b.first_frame = 0;
        switch (wf->r0) {
        case 2:  rc = launch_big<2>(wf, b, st); break;
        case 4:  rc = launch_big<4>(wf, b, st); break;
        case 8:  rc = launch_big<8>(wf, b, st); break;
        case 16: rc = launch_big<16>(wf, b, st); break;
        default: return fail(OWRX_E_INVALID, "unsupported fft size");
        }
        if (rc != OWRX_OK) return rc;
    }

    // finalize: log / swap / quantise.  The ADPCM encoder runs once per batch (wf_process), not here: its run time is the
    // serial latency of ONE line however many lines are in flight.
    const bool adpcm = wf->compression == OWRX_COMPRESSION_ADPCM;
    float* db = db_dev;
    if (!adpcm && out_dev) db = (float*)out_dev;   // compression "none": the line IS the float32 dB row
    const float corr = wf->avg > 0 ? wf->add_db - 10.0f * log10f((float)wf->avg) : wf->add_db;
    const size_t total = lines * (size_t)n;
    if (wf->nf_on && lines) {
        if (!wf->d_noise) OWRX_CUDA(cudaMalloc((void**)&wf->d_noise, (size_t)n * sizeof(float)));
        wf_noise_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(wf->d_partial, subsets, n, lines, wf->d_noise, wf->nf_primed ? 0 : 1,
                                                                    wf->nf_alpha, wf->nf_beta, wf->nf_growth);
        OWRX_LAUNCH_CHECK();
        wf->nf_primed = true;
    }
    wf_finalize_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(wf->d_partial, subsets, n, corr, lines, db,
                                                                       adpcm ? s16_dev : nullptr);
    OWRX_LAUNCH_CHECK();
    if (!adpcm && db_dev && out_dev && db_dev != (float*)out_dev)
        OWRX_CUDA(cudaMemcpyAsync(db_dev, out_dev, total * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return OWRX_OK;
}

static int wf_process(owrx_wf* wf, const float2* iq_dev, size_t n_samples, uint8_t* out_dev, size_t out_cap,
                      float* db_dev, int16_t* s16_dev, size_t* n_lines, cudaStream_t st)
{
    const size_t lines = wf_lines_for(wf, n_samples);
    const size_t lb = wf_line_bytes(wf);
    if (out_dev && lines * lb > out_cap) return fail(OWRX_E_OVERFLOW, "output buffer too small: need %zu bytes", lines * lb);
    const bool adpcm = wf->compression == OWRX_COMPRESSION_ADPCM;
    const int n = wf->n;
    int16_t* s16 = s16_dev;
    int rc;
    const bool side_adpcm = adpcm && out_dev && wf->pipelined && !s16_dev;
    if (adpcm && !s16 && lines) {
        const bool alt = wf->pipelined && wf->s16_cur;
        if (wf->pipelined) {
            // the encoder of two batches ago was reading this buffer (growing it would also free it under the encoder)
            OWRX_CUDA(cudaStreamWaitEvent(st, wf->adpcm_done[wf->s16_cur], 0));
            if (lines * (size_t)(n + 10) > (alt ? wf->s16_alt_cap : wf->s16_cap)) OWRX_CUDA(cudaStreamSynchronize(wf->side));
        }
        if ((rc = alt ? grow(&wf->d_s16_alt, &wf->s16_alt_cap, lines * (size_t)(n + 10))
                      : grow(&wf->d_s16, &wf->s16_cap, lines * (size_t)(n + 10))) != OWRX_OK)
            return rc;
        s16 = alt ? wf->d_s16_alt : wf->d_s16;
    }
    if (lines && (rc = wf_run_lines(wf, iq_dev, lines, out_dev, db_dev, s16, st)) != OWRX_OK) return rc;
    if (adpcm && out_dev && lines) {
        cudaStream_t sa = st;
        if (side_adpcm) {
            OWRX_CUDA(cudaEventRecord(wf->fin_done, st));
            OWRX_CUDA(cudaStreamWaitEvent(wf->side, wf->fin_done, 0));
            sa = wf->side;
        }
        // the encoder is a latency-bound serial chain per line (one warp per 32 lines): beside the FFT pass of the next batch
        // its warps lose issue slots to 16 FFT warps per SM.  Claiming shared memory it does not use keeps a second FFT CTA
        // (86 KB) off its SM: 150 KB leaves its 19 CTAs alone on their SMs (C1, 592 lines per batch: 0.87 -> 0.78 ms per batch;
        // OWRX_WF_ADPCM_PAD_KB overrides)
        static const int adpcm_pad = (getenv("OWRX_WF_ADPCM_PAD_KB") ? atoi(getenv("OWRX_WF_ADPCM_PAD_KB")) : 150) << 10;
        if (adpcm_pad) OWRX_CUDA(cudaFuncSetAttribute(wf_adpcm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, adpcm_pad));
        wf_adpcm_kernel<<<(unsigned)((lines + 32 * ADPCM_WARPS - 1) / (32 * ADPCM_WARPS)), 32 * ADPCM_WARPS, side_adpcm ? adpcm_pad : 0, sa>>>(
            s16, out_dev, n + 10, lines);
        OWRX_LAUNCH_CHECK();
        if (side_adpcm) {
            OWRX_CUDA(cudaEventRecord(wf->adpcm_done[wf->s16_cur], sa));
            wf->s16_cur ^= 1;
        }
    }
    if (n_lines) *n_lines = lines;
    return OWRX_OK;
}

static int wf_build_tables(owrx_wf* wf)
{
    const int n = wf->n, m = wf->m, r3 = m / 256;
    std::vector<float> win((size_t)n);
    for (int i = 0; i < n; i++) win[i] = (float)(0.54 - 0.46 * cos(2.0 * M_PI * i / (double)(n - 1)));  // SURVEY A.2
    std::vector<float2> tw2(256), tw3((size_t)std::max(r3, 1) * 256), twn;
    for (int r = 0; r < 16; r++)
        for (int k = 0; k < 16; k++) {
            double a = -2.0 * M_PI * r * k / 256.0;
            tw2[r * 16 + k] = make_float2((float)cos(a), (float)sin(a));
        }
    for (int r = 0; r < r3; r++)
        for (int k = 0; k < 256; k++) {
            double a = -2.0 * M_PI * (double)r * k / (double)m;
            tw3[(size_t)r * 256 + k] = make_float2((float)cos(a), (float)sin(a));
        }
    OWRX_CUDA(cudaMalloc((void**)&wf->d_counter, sizeof(int)));
    OWRX_CUDA(cudaMalloc((void**)&wf->d_window, win.size() * sizeof(float)));
    OWRX_CUDA(cudaMalloc((void**)&wf->d_tw2, tw2.size() * sizeof(float2)));
    OWRX_CUDA(cudaMalloc((void**)&wf->d_tw3, tw3.size() * sizeof(float2)));
    OWRX_CUDA(cudaMemcpy(wf->d_window, win.data(), win.size() * sizeof(float), cudaMemcpyHostToDevice));
    OWRX_CUDA(cudaMemcpy(wf->d_tw2, tw2.data(), tw2.size() * sizeof(float2), cudaMemcpyHostToDevice));
    OWRX_CUDA(cudaMemcpy(wf->d_tw3, tw3.data(), tw3.size() * sizeof(float2), cudaMemcpyHostToDevice));
    if (wf->r0 > 1) {
        twn.resize((size_t)n);
        for (int k1 = 0; k1 < wf->r0; k1++)
            for (int n2 = 0; n2 < m; n2++) {
                double a = -2.0 * M_PI * (double)k1 * n2 / (double)n;
                twn[(size_t)k1 * m + n2] = make_float2((float)cos(a), (float)sin(a));
            }
        OWRX_CUDA(cudaMalloc((void**)&wf->d_twn, twn.size() * sizeof(float2)));
        OWRX_CUDA(cudaMemcpy(wf->d_twn, twn.data(), twn.size() * sizeof(float2), cudaMemcpyHostToDevice));
    }
    return OWRX_OK;
}

extern "C" {

int owrx_wf_create(int device, int fft_size, int every_n_samples, int avg_number, float add_db, int compression,
                   owrx_wf_t** out)
{
    if (!out) return fail(OWRX_E_INVALID, "out is NULL");
    *out = nullptr;
    if (fft_size < 256 || fft_size > 65536 || (fft_size & (fft_size - 1)))
        return fail(OWRX_E_INVALID, "fft_size must be a power of two in [256, 65536], got %d", fft_size);
    if (every_n_samples < 0 || avg_number < 0) return fail(OWRX_E_INVALID, "negative every_n_samples / avg_number");
    if (compression != OWRX_COMPRESSION_NONE && compression != OWRX_COMPRESSION_ADPCM)
        return fail(OWRX_E_INVALID, "unknown compression %d", compression);
    int sm = 0, rc = select_device(device, &sm);
    if (rc != OWRX_OK) return rc;
    owrx_wf* wf = new (std::nothrow) owrx_wf();
    if (!wf) return fail(OWRX_E_NOMEM, "out of host memory");
    wf->device = device; wf->sm_count = sm;
    wf->n = fft_size; wf->every_n = every_n_samples; wf->avg = avg_number; wf->add_db = add_db;
    wf->compression = compression;
    if (fft_size <= 4096) { wf->m = fft_size; wf->r0 = 1; } else { wf->m = 4096; wf->r0 = fft_size / 4096; }
    wf->log2m = 0;
    while ((1 << wf->log2m) < wf->m) wf->log2m++;
    cudaError_t e = cudaStreamCreateWithFlags(&wf->stream, cudaStreamNonBlocking);
    int prio_lo = 0, prio_hi = 0;
    if (e == cudaSuccess) e = cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&wf->side, cudaStreamNonBlocking, prio_hi);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&wf->fin_done, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&wf->adpcm_done[0], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&wf->adpcm_done[1], cudaEventDisableTiming);
    if (e != cudaSuccess) { delete wf; return fail(OWRX_E_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e)); }
    rc = wf_build_tables(wf);
    if (rc != OWRX_OK) { owrx_wf_destroy(wf); return rc; }
    *out = wf;
    return OWRX_OK;
}

void owrx_wf_destroy(owrx_wf_t* wf)
{
    if (!wf) return;
    cudaSetDevice(wf->device);
    if (wf->stream) cudaStreamSynchronize(wf->stream);
    cudaFree(wf->d_window); cudaFree(wf->d_tw2); cudaFree(wf->d_tw3); cudaFree(wf->d_twn); cudaFree(wf->d_counter); cudaFree(wf->d_ybig);
    cudaDeviceSynchronize();
    cudaFree(wf->d_partial); cudaFree(wf->d_s16); cudaFree(wf->d_s16_alt);
    if (wf->fin_done) cudaEventDestroy(wf->fin_done);
    if (wf->adpcm_done[0]) cudaEventDestroy(wf->adpcm_done[0]);
    if (wf->adpcm_done[1]) cudaEventDestroy(wf->adpcm_done[1]);
    if (wf->side) cudaStreamDestroy(wf->side);
    cudaFree(wf->d_in); cudaFree(wf->d_in_alt); cudaFree(wf->d_out); cudaFree(wf->d_noise); cudaFree(wf->d_raw);
    if (wf->h_out) cudaFreeHost(wf->h_out);
    if (wf->stream) cudaStreamDestroy(wf->stream);
    delete wf;
}

int owrx_wf_set_every_n_samples(owrx_wf_t* wf, int every_n_samples)
{
    if (!wf || every_n_samples < 0) return fail(OWRX_E_INVALID, "bad every_n_samples");
    std::lock_guard<std::mutex> g(wf->mu);
    wf->every_n = every_n_samples;
    return OWRX_OK;
}

int owrx_wf_set_avg_number(owrx_wf_t* wf, int avg_number)
{
    if (!wf || avg_number < 0) return fail(OWRX_E_INVALID, "bad avg_number");
    std::lock_guard<std::mutex> g(wf->mu);
    if (wf->avg != avg_number) wf->nf_primed = false;           // the power scale (sum over avg frames) changes: re-seed the floor
    wf->avg = avg_number;
    return OWRX_OK;
}

int owrx_wf_set_noise_filter(owrx_wf_t* wf, int enable, float alpha, float beta, float growth)
{
    if (!wf) return fail(OWRX_E_INVALID, "NULL waterfall");
    if (enable && !(alpha >= 0.f && alpha <= 4.f && beta >= 0.f && beta <= 1.f && growth >= 0.f && growth <= 1.f))
        return fail(OWRX_E_INVALID, "noise filter parameters out of range (alpha 0..4, beta 0..1, growth 0..1)");
    std::lock_guard<std::mutex> g(wf->mu);
    wf->nf_on = enable != 0;
    wf->nf_alpha = alpha; wf->nf_beta = beta; wf->nf_growth = growth;
    wf->nf_primed = false;
    return OWRX_OK;
}

int owrx_wf_set_compression(owrx_wf_t* wf, int compression)
{
    if (!wf || (compression != OWRX_COMPRESSION_NONE && compression != OWRX_COMPRESSION_ADPCM))
        return fail(OWRX_E_INVALID, "bad compression");
    std::lock_guard<std::mutex> g(wf->mu);
    if (compression != wf->compression) wf->queue.clear();   // queued lines have the old format
    wf->compression = compression;
    return OWRX_OK;
}

size_t owrx_wf_line_bytes(const owrx_wf_t* wf) { return wf ? wf_line_bytes(wf) : 0; }

size_t owrx_wf_lines_for(const owrx_wf_t* wf, size_t n_samples) { return wf ? wf_lines_for(wf, n_samples) : 0; }

int owrx_wf_process_device(owrx_wf_t* wf, const void* iq_dev, size_t n_samples, void* out_dev, size_t out_cap_bytes,
                           void* db_dev, void* s16_dev, size_t* n_lines, void* stream)
{
    if (!wf || !iq_dev) return fail(OWRX_E_INVALID, "NULL argument");
    std::lock_guard<std::mutex> g(wf->mu);
    OWRX_CUDA(cudaSetDevice(wf->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : wf->stream;
    return wf_process(wf, (const float2*)iq_dev, n_samples, (uint8_t*)out_dev, out_cap_bytes, (float*)db_dev,
                      (int16_t*)s16_dev, n_lines, st);
}

int owrx_wf_feed(owrx_wf_t* wf, const float* iq, size_t n_samples)
{
    return owrx_wf_feed_fmt(wf, iq, n_samples, OWRX_IQ_CF32, 1.0f);
}

int owrx_wf_feed_fmt(owrx_wf_t* wf, const void* iq_raw, size_t n_samples, int format, float gain)
{
    if (!wf || (!iq_raw && n_samples)) return fail(OWRX_E_INVALID, "NULL argument");
    const size_t in_bytes = iq_format_bytes(format);
    if (!in_bytes) return fail(OWRX_E_INVALID, "unknown IQ format %d", format);
    std::lock_guard<std::mutex> g(wf->mu);
    OWRX_CUDA(cudaSetDevice(wf->device));
    // honour a pending skip (every_n > fft_size leaves a gap after the last consumed frame)
    if (wf->skip) {
        const size_t d = std::min(wf->skip, n_samples);
        iq_raw = static_cast<const unsigned char*>(iq_raw) + d * in_bytes; n_samples -= d; wf->skip -= d;
    }
    if (!n_samples) return OWRX_OK;
    (host_is_pinned(iq_raw) ? wf->h2d_pinned : wf->h2d_pageable) += n_samples * in_bytes;
    const size_t need = wf->in_fill + n_samples;
    if (need > wf->in_cap) {
        const size_t cap = std::max(need, wf->in_cap * 2);
        float2* nb = nullptr;
        OWRX_CUDA(cudaMalloc((void**)&nb, cap * sizeof(float2)));
        if (wf->in_fill) OWRX_CUDA(cudaMemcpyAsync(nb, wf->d_in, wf->in_fill * sizeof(float2), cudaMemcpyDeviceToDevice, wf->stream));
        OWRX_CUDA(cudaStreamSynchronize(wf->stream));
        cudaFree(wf->d_in); cudaFree(wf->d_in_alt);
        wf->d_in = nb; wf->d_in_alt = nullptr; wf->in_cap = cap;
        OWRX_CUDA(cudaMalloc((void**)&wf->d_in_alt, cap * sizeof(float2)));
    }
    if (format == OWRX_IQ_CF32) {
        OWRX_CUDA(cudaMemcpyAsync(wf->d_in + wf->in_fill, iq_raw, n_samples * sizeof(float2), cudaMemcpyHostToDevice, wf->stream));
    } else {
        // raw samples cross PCIe as they are; Convert (+ Gain) on the GPU (owrx/source/fifi_sdr.py:27-28)
        if (n_samples * in_bytes > wf->raw_cap) {
            OWRX_CUDA(cudaStreamSynchronize(wf->stream));
            cudaFree(wf->d_raw); wf->d_raw = nullptr; wf->raw_cap = 0;
            OWRX_CUDA(cudaMalloc((void**)&wf->d_raw, n_samples * in_bytes));
            wf->raw_cap = n_samples * in_bytes;
        }
        OWRX_CUDA(cudaMemcpyAsync(wf->d_raw, iq_raw, n_samples * in_bytes, cudaMemcpyHostToDevice, wf->stream));
        int rcc = iq_convert_launch(format, wf->d_raw, wf->d_in + wf->in_fill, n_samples, gain, wf->stream);
        if (rcc != OWRX_OK) return rcc;
    }
    wf->in_fill += n_samples;
    const size_t lines = wf_lines_for(wf, wf->in_fill);
    if (!lines) { OWRX_CUDA(cudaStreamSynchronize(wf->stream)); return OWRX_OK; }
    const size_t lb = wf_line_bytes(wf);
    if (lines * lb > wf->out_cap) {
        cudaFree(wf->d_out); wf->d_out = nullptr; wf->out_cap = 0;
        OWRX_CUDA(cudaMalloc((void**)&wf->d_out, lines * lb));
        wf->out_cap = lines * lb;
    }
    if (lines * lb > wf->h_out_cap) {
        if (wf->h_out) cudaFreeHost(wf->h_out);
        wf->h_out = nullptr; wf->h_out_cap = 0;
        OWRX_CUDA(cudaMallocHost((void**)&wf->h_out, lines * lb));
        wf->h_out_cap = lines * lb;
    }
    size_t got = 0;
    int rc = wf_process(wf, wf->d_in, wf->in_fill, wf->d_out, wf->out_cap, nullptr, nullptr, &got, wf->stream);
    if (rc != OWRX_OK) return rc;
    OWRX_CUDA(cudaMemcpyAsync(wf->h_out, wf->d_out, got * lb, cudaMemcpyDeviceToHost, wf->stream));
    // carry the unconsumed tail to the front of the alternate buffer
    const size_t fpl = (size_t)(wf->avg > 0 ? wf->avg : 1);
    const size_t consumed = got * fpl * (size_t)wf->every_n;
    if (consumed >= wf->in_fill) {
        wf->skip = consumed - wf->in_fill;
        wf->in_fill = 0;
    } else {
        const size_t tail = wf->in_fill - consumed;
        OWRX_CUDA(cudaMemcpyAsync(wf->d_in_alt, wf->d_in + consumed, tail * sizeof(float2), cudaMemcpyDeviceToDevice, wf->stream));
        std::swap(wf->d_in, wf->d_in_alt);
        wf->in_fill = tail;
    }
    OWRX_CUDA(cudaStreamSynchronize(wf->stream));
    for (size_t l = 0; l < got; l++) wf->queue.emplace_back(wf->h_out + l * lb, wf->h_out + (l + 1) * lb);
    return OWRX_OK;
}

int owrx_wf_get_h2d_bytes(const owrx_wf_t* wf, uint64_t* pinned_bytes, uint64_t* pageable_bytes)
{
    if (!wf || !pinned_bytes || !pageable_bytes) return fail(OWRX_E_INVALID, "NULL argument");
    *pinned_bytes = wf->h2d_pinned; *pageable_bytes = wf->h2d_pageable;
    return OWRX_OK;
}

int owrx_wf_read(owrx_wf_t* wf, void* out, size_t cap_bytes, size_t* n_bytes)
{
    if (!wf || !out || !n_bytes) return fail(OWRX_E_INVALID, "NULL argument");
    std::lock_guard<std::mutex> g(wf->mu);
    size_t o = 0;
    while (!wf->queue.empty() && o + wf->queue.front().size() <= cap_bytes) {
        memcpy((uint8_t*)out + o, wf->queue.front().data(), wf->queue.front().size());
        o += wf->queue.front().size();
        wf->queue.pop_front();
    }
    *n_bytes = o;
    if (o == 0 && !wf->queue.empty()) return fail(OWRX_E_OVERFLOW, "buffer smaller than one line");
    return OWRX_OK;
}

int owrx_wf_read_message(owrx_wf_t* wf, void* out, size_t cap_bytes, size_t* n_bytes)
{
    if (!wf || !out || !n_bytes) return fail(OWRX_E_INVALID, "NULL argument");
    std::lock_guard<std::mutex> g(wf->mu);
    *n_bytes = 0;
    if (wf->queue.empty()) return OWRX_OK;
    const size_t len = wf->queue.front().size();
    if (len + 1 > cap_bytes) return fail(OWRX_E_OVERFLOW, "buffer smaller than one framed line (%zu bytes)", len + 1);
    uint8_t* o = (uint8_t*)out;
    o[0] = 0x01;                                               // write_spectrum_data: bytes([0x01]) + data (owrx/connection.py:473-475)
    memcpy(o + 1, wf->queue.front().data(), len);
    wf->queue.pop_front();
    *n_bytes = len + 1;
    return OWRX_OK;
}

int owrx_wf_set_pipelined(owrx_wf_t* wf, int enable)
{
    if (!wf) return fail(OWRX_E_INVALID, "NULL waterfall");
    std::lock_guard<std::mutex> g(wf->mu);
    OWRX_CUDA(cudaSetDevice(wf->device));
    OWRX_CUDA(cudaDeviceSynchronize());
    wf->pipelined = enable != 0;
    return OWRX_OK;
}

int owrx_wf_join(owrx_wf_t* wf, void* stream)
{
    if (!wf) return fail(OWRX_E_INVALID, "NULL waterfall");
    std::lock_guard<std::mutex> g(wf->mu);
    OWRX_CUDA(cudaSetDevice(wf->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : wf->stream;
    OWRX_CUDA(cudaStreamWaitEvent(st, wf->adpcm_done[0], 0));
    OWRX_CUDA(cudaStreamWaitEvent(st, wf->adpcm_done[1], 0));
    return OWRX_OK;
}

int owrx_fft_adpcm_encode_device(int device, const void* s16_dev, int fft_size, size_t n_lines, void* out_dev, void* stream)
{
    if (!s16_dev || !out_dev || fft_size <= 0 || (fft_size & 1)) return fail(OWRX_E_INVALID, "bad argument");
    int rc = select_device(device, nullptr);
    if (rc != OWRX_OK) return rc;
    if (!n_lines) return OWRX_OK;
    wf_adpcm_kernel<<<(unsigned)((n_lines + 32 * ADPCM_WARPS - 1) / (32 * ADPCM_WARPS)), 32 * ADPCM_WARPS, 0, (cudaStream_t)stream>>>(
        (const int16_t*)s16_dev, (uint8_t*)out_dev, fft_size + 10, n_lines);
    OWRX_LAUNCH_CHECK();
    return OWRX_OK;
}

}  // extern "C"
