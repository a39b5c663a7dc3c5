// fastconv.cu — K3F kernels: polyphase fast-convolution channeliser (see fastconv.cuh for the algebra).
// Replaces pycsdr Shift + FirDecimate (reference call sites csdr/chain/selector.py:29,57,95,140) for all client
// channels of a decimator group at once.  Hand-written for sm_100a; no cuFFT / cuBLAS.
#include "fastconv.cuh"
#include "fft_small.cuh"

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>

namespace owrx {

namespace {

// ------------------------------------------------------------------------------------------------
// Tab[q][r][slot] = sum_{s<P} h[D s + r] e^{j 2 pi rate (D s + r)} e^{+j 2 pi q s / M}
// Phases in double (two sincospi per entry, then a 27-step double recurrence), rounded once to float.
// ------------------------------------------------------------------------------------------------
// x = h + m + l with three bf16 terms (the operand planes of the tensor-core contraction, fastconv_tc.cu)
__device__ __forceinline__ void split_bf16x3(float x, __nv_bfloat16& h, __nv_bfloat16& m, __nv_bfloat16& l)
{
    h = __float2bfloat16_rn(x);
    const float r1 = x - __bfloat162float(h);
    m = __float2bfloat16_rn(r1);
    l = __float2bfloat16_rn(r1 - __bfloat162float(m));
}

// x 2^k = h + m with two fp16 terms (the block-scaled operand planes of the tensor-core contraction's default form)
__device__ __forceinline__ void split_f16x2(float x, __half& h, __half& m)
{
    h = __float2half_rn(x);
    m = __float2half_rn(x - __half2float(h));
}

// TC = 0: tab[q][r][slot] complex float32.  TC = 3: bf16 planes Tp[2 level + part][q * slots + slot][r].  TC = 2: fp16 planes of
// the entries times tab_scale (a power of two).
template <int TC>
__global__ void __launch_bounds__(256)
fc_table_kernel(const float* __restrict__ h, int T, int D, int Dp, int P, int slots, int M, const int* __restrict__ slot_list,
                const double* __restrict__ rate_list, void* __restrict__ tab_out, float tab_scale)
{
    const long long idx = (long long)blockIdx.x * 256 + threadIdx.x;
    if (idx >= (long long)M * D) return;
    const int q = (int)(idx / D), r = (int)(idx % D);
    const double rate = rate_list[blockIdx.y];
    const int slot = slot_list[blockIdx.y];
    double a0 = rate * (double)r;
    a0 -= floor(a0);
    double aw = rate * (double)D;
    aw -= floor(aw);
    aw += (double)q / M;
    double c0, s0, cw, sw;
    sincospi(2.0 * a0, &s0, &c0);
    sincospi(2.0 * aw, &sw, &cw);
    double ar = 0.0, ai = 0.0;
    for (int s = 0; s < P; s++) {
        const int t = D * s + r;
        if (t < T) {
            const double hv = (double)__ldg(h + t);
            ar += hv * c0;
            ai += hv * s0;
        }
        const double nc = c0 * cw - s0 * sw, ns = c0 * sw + s0 * cw;
        c0 = nc; s0 = ns;
    }
    if (TC == 0) {
        reinterpret_cast<float2*>(tab_out)[((size_t)q * Dp + r) * slots + slot] = make_float2((float)ar, (float)ai);
    } else if (TC == 2) {
        __half* tp = reinterpret_cast<__half*>(tab_out);
        const size_t plane = (size_t)M * slots * Dp, at = ((size_t)q * slots + slot) * Dp + r;
        __half a[2], b[2];
        split_f16x2((float)ar * tab_scale, a[0], a[1]);
        split_f16x2((float)ai * tab_scale, b[0], b[1]);
#pragma unroll
        for (int l = 0; l < 2; l++) {
            tp[(size_t)(2 * l) * plane + at] = a[l];
            tp[(size_t)(2 * l + 1) * plane + at] = b[l];
        }
    } else {
        __nv_bfloat16* tp = reinterpret_cast<__nv_bfloat16*>(tab_out);
        const size_t plane = (size_t)M * slots * Dp, at = ((size_t)q * slots + slot) * Dp + r;
        __nv_bfloat16 a[3], b[3];
        split_bf16x3((float)ar, a[0], a[1], a[2]);
        split_bf16x3((float)ai, b[0], b[1], b[2]);
#pragma unroll
        for (int l = 0; l < 3; l++) {
            tp[(size_t)(2 * l) * plane + at] = a[l];
            tp[(size_t)(2 * l + 1) * plane + at] = b[l];
        }
    }
}

// ------------------------------------------------------------------------------------------------
// 256-point FFT of 32 interleaved sequences per CTA (16 threads x 16 points each per sequence, radix 16 x 16).
// Thread (g = tid >> 5, j = tid & 31): sequence j, pass-1 residue n2 = g, pass-2 output residue k1 = g.
// A warp = one g, 32 adjacent sequences -> every global access of a warp is one 256-byte row.
// ------------------------------------------------------------------------------------------------
constexpr int FC_SEQ = 32;
constexpr int FC_STR = FC_M + 1;            // odd sequence stride (in float2): conflict-free across the 32 lanes

__device__ __forceinline__ void fc_fill_twiddles(float2* tw)
{
    // tw[r * 16 + k] = e^{-2 pi i r k / 256}
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        const int e = ((i >> 4) * (i & 15)) & 255;
        float s, c;
        sincospif(-(float)e / 128.0f, &s, &c);
        tw[i] = make_float2(c, s);
    }
}

// V x V-point FFT (V = 16: 256 points, V = 8: 64 points), V threads per sequence, V points per thread.
// tw[r * V + k] = e^{-2 pi i r k / V^2};  in: v[n1] = x[V n1 + g];  out: v[q] = X[g + V slot<V>(q)]
template <int V>
__device__ __forceinline__ void fc_fill_twiddles_v(float2* tw)
{
    for (int i = threadIdx.x; i < V * V; i += blockDim.x) {
        const int e = ((i / V) * (i % V)) & (V * V - 1);
        float s, c;
        sincospif(-(float)e / (float)(V * V / 2), &s, &c);
        tw[i] = make_float2(c, s);
    }
}
template <int V>
__device__ __forceinline__ void fc_fft_vv(float2* v, float2* seq, const float2* tw, int g)
{
    dft<V>(v);
#pragma unroll
    for (int q = 0; q < V; q++) seq[g * V + slot<V>(q)] = v[q];
    __syncthreads();
#pragma unroll
    for (int r = 0; r < V; r++) v[r] = seq[r * V + g];
#pragma unroll
    for (int r = 1; r < V; r++) v[r] = cmul(v[r], tw[r * V + g]);
    dft<V>(v);
}
__device__ __forceinline__ void fc_fft256(float2* v, float2* seq, const float2* tw, int g) { fc_fft_vv<16>(v, seq, tw, g); }

// TC = 0: F[q][b][r] as (re, re, -im, im).  TC = 3: bf16 planes Fp[2 level + part][q * B + b][r].  TC = 2: fp16 planes of the
// spectra times *scale (the pass's power of two, fc_scale_kernel).
// V = 16: 256-point FFTs (16 threads x 16 points per sequence), V = 8: 64-point FFTs (8 x 8).
template <int TC, int V>
__global__ void __launch_bounds__(V * FC_SEQ)
fc_forward_kernel(const float2* __restrict__ iq, long long n_lim, int D, int Dp, int Kb, int B, void* __restrict__ F_out,
                  const float* __restrict__ scale)
{
    constexpr int M = V * V;
    extern __shared__ float2 fc_smem[];
    float2* tw = fc_smem;                       // [M]
    float2* seqs = fc_smem + M;                 // [32][M + 1]
    const int tid = threadIdx.x, j = tid & 31, g = tid >> 5;
    const int b = blockIdx.y;
    const int r = blockIdx.x * FC_SEQ + j;
    fc_fill_twiddles_v<V>(tw);
    float2 v[V];
    const long long s0 = (long long)b * Kb * D + r;
#pragma unroll
    for (int n1 = 0; n1 < V; n1++) {
        const long long s = s0 + (long long)(V * n1 + g) * D;
        v[n1] = (r < D && s < n_lim) ? __ldg(iq + s) : make_float2(0.f, 0.f);
    }
    __syncthreads();                            // twiddles visible
    fc_fft_vv<V>(v, seqs + j * (M + 1), tw, g);
#pragma unroll
    for (int q = 0; q < V; q++) {
        const int bin = g + V * slot<V>(q);
        if (TC == 0) {
            // operand layout of the contraction's packed FMAs: (re, re) and (-im, im)
            reinterpret_cast<float4*>(F_out)[((size_t)bin * B + b) * Dp + r] = make_float4(v[q].x, v[q].x, -v[q].y, v[q].y);
        } else if (TC == 2) {
            __half* fp = reinterpret_cast<__half*>(F_out);
            const size_t plane = (size_t)M * B * Dp, at = ((size_t)bin * B + b) * Dp + r;
            const float sc = __ldg(scale);
            __half a[2], c[2];
            split_f16x2(v[q].x * sc, a[0], a[1]);
            split_f16x2(v[q].y * sc, c[0], c[1]);
#pragma unroll
            for (int l = 0; l < 2; l++) {
                fp[(size_t)(2 * l) * plane + at] = a[l];
                fp[(size_t)(2 * l + 1) * plane + at] = c[l];
            }
        } else {
            __nv_bfloat16* fp = reinterpret_cast<__nv_bfloat16*>(F_out);
            const size_t plane = (size_t)M * B * Dp, at = ((size_t)bin * B + b) * Dp + r;
            __nv_bfloat16 a[3], c[3];
            split_bf16x3(v[q].x, a[0], a[1], a[2]);
            split_bf16x3(v[q].y, c[0], c[1], c[2]);
#pragma unroll
            for (int l = 0; l < 3; l++) {
                fp[(size_t)(2 * l) * plane + at] = a[l];
                fp[(size_t)(2 * l + 1) * plane + at] = c[l];
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Z[q][b][c] = sum_{r<Dp} F[q][b][r] * Tab[q][r][c]     (complex x complex, FP32 FMA pipe)
// CTA = (bin q, tile of BT = 16 NW blocks, 64 channel slots).  A warp owns 16 rows x 64 columns; its lanes form a
// 2 x 16 grid: lane (lr, lc) holds rows 16w + 2i + lr (i < 8) and columns {2lc, 2lc+1, 32+2lc, 33+2lc} — an 8 x 4
// register tile of complex accumulators, so one staged operand feeds 4 (F) or 8 (table) complex MACs and the
// shared-memory wavefronts per MAC stay well under the FMA pipe's demand.
// Blackwell packed FP32 (fma.rn.f32x2 -> FFMA2): an accumulator is the (re, im) pair of one output,
//   acc += (f.re, f.re) * (t.re, t.im);   acc += (-f.im, f.im) * (t.im, t.re)
// The forward pass stores F already as (re, re, -im, im): one LDS.128 per (row, branch) yields both packed
// multiplicands; the table pairs (t.re, t.im) of two columns come from one LDS.128 and the swapped pair costs two
// register moves per column.  Per branch and thread: 10 LDS.128 + 8 MOV + 64 FFMA2.  Operand chunks of 32 branches
// stream through a 3-stage TMA (cp.async.bulk) ring guarded by mbarriers; two warp groups split the branches of a chunk
// (even / odd) and meet in shared memory at the end, so a 96-row CTA runs 12 consumer warps + 1 producer warp.
// ------------------------------------------------------------------------------------------------
constexpr int FC_ST = 3;
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float lo, float hi)
{
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void upk2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ void ffma2(f32x2& c, f32x2 a, f32x2 b) { asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(c) : "l"(a), "l"(b)); }
__device__ __forceinline__ void lds2x64(f32x2& a, f32x2& b, unsigned addr)
{
    asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "r"(addr));
}
__device__ __forceinline__ f32x2 swap2(f32x2 v)
{
    float a, b;
    upk2(v, a, b);
    return pk2(b, a);
}

// ---- TMA (bulk async copy) + mbarrier plumbing for the operand pipeline
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "FC_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra FC_DONE;\n"
        "bra FC_WAIT;\n"
        "FC_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity)
        : "memory");
}
// one TMA tile: box (128 floats x rows) of a 2D row-major float tensor -> dense [rows][128] floats in shared memory
__device__ __forceinline__ void tma_load_2d(unsigned dst, const CUtensorMap* map, int c0, int c1, unsigned bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n" ::"r"(dst),
                 "l"(reinterpret_cast<unsigned long long>(map)), "r"(c0), "r"(c1), "r"(bar)
                 : "memory");
}

// Warp roles: 2 NW consumer warps (two groups: even / odd branches of a chunk) + 1 producer warp whose elected lane streams
// the operand chunks with two TMA tile loads each (F: BT blocks x 32 branches; table: 32 branches x 64 slots) into a 3-stage
// ring guarded by full/empty mbarriers; no CTA-wide barrier inside the branch loop.
template <int NW>
__global__ void __launch_bounds__(NW * 64 + 32, 1)
fc_contract_kernel(const __grid_constant__ CUtensorMap mapF, const __grid_constant__ CUtensorMap mapT, float2* __restrict__ Z, int B, int Dp,
                   int slots, int nbt, int nsplit, int M)
{
    constexpr int BT = 16 * NW;
    constexpr unsigned F_STAGE = BT * FC_KC * sizeof(float4), T_STAGE = FC_KC * FC_CG * sizeof(float2);
    extern __shared__ __align__(128) float4 fc_smem4[];
    __shared__ unsigned long long bars[2 * FC_ST];                   // full[ST], empty[ST]
    float4* Fs = fc_smem4;                                            // [ST][BT][KC]   (re, re, -im, im)
    float2* Ts = reinterpret_cast<float2*>(Fs + FC_ST * BT * FC_KC);  // [ST][KC][64]
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const bool producer = wid == 2 * NW;
    const int grp = wid / NW, warp = wid % NW;
    const int lr = lane >> 4, lc = lane & 15;
    const int q = blockIdx.x / nbt, bt = blockIdx.x % nbt;
    const int cg = blockIdx.y;
    const int b0 = bt * BT;
    const int rows = min(BT, B - b0);
    // split-K: this CTA contracts branch chunks [ch0, ch0 + nchunks) and writes partial-sum plane blockIdx.z of Z (the
    // planes are added by fc_inverse_kernel): used when the bin tiles alone leave a poorly filled last wave and a tile is long
    // enough (many chunks: large D) to amortise the ring fill
    const int all_chunks = Dp / FC_KC;
    const int ch0 = (int)(((long long)all_chunks * blockIdx.z) / nsplit);
    const int nchunks = (int)(((long long)all_chunks * (blockIdx.z + 1)) / nsplit) - ch0;
    Z += (size_t)blockIdx.z * M * B * slots;
    // rows 16w + 2i + lr of this warp that exist: i < ni (the lr = 1 half of a last odd row reads a stale row; not stored)
    const int ni = min(8, max(0, (rows - warp * 16 + 1) / 2));

    const unsigned bar0 = (unsigned)__cvta_generic_to_shared(bars);
    const unsigned fs0 = (unsigned)__cvta_generic_to_shared(Fs), ts0 = (unsigned)__cvta_generic_to_shared(Ts);
    if (tid == 0) {
        for (int s = 0; s < FC_ST; s++) {
            mbar_init(bar0 + 8 * s, 1);                               // full: the producer's expect_tx arrival
            mbar_init(bar0 + 8 * (FC_ST + s), 2 * NW);                // empty: one arrival per consumer warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncthreads();

    f32x2 acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
        for (int c = 0; c < 4; c++) acc[i][c] = 0ull;

    if (producer) {
        if (lane == 0) {
            for (int ch = 0; ch < nchunks; ch++) {
                const int stage = ch % FC_ST, use = ch / FC_ST;
                const unsigned full = bar0 + 8 * stage, empty = bar0 + 8 * (FC_ST + stage);
                mbar_wait(empty, (use & 1) ^ 1);                      // every consumer warp has released this slot
                mbar_expect_tx(full, F_STAGE + T_STAGE);
                // rows past the last block of a short tile come from the next bin (or are zero-filled past the tensor):
                // they only feed accumulators that are never stored
                tma_load_2d(fs0 + stage * F_STAGE, &mapF, (ch0 + ch) * FC_KC * 4, q * B + b0, full);
                tma_load_2d(ts0 + stage * T_STAGE, &mapT, cg * FC_CG * 2, q * Dp + (ch0 + ch) * FC_KC, full);
            }
        }
    } else {
        const unsigned fs_base = fs0 + (unsigned)(((warp * 16 + lr) * FC_KC + grp) * sizeof(float4));
        const unsigned ts_base = ts0 + (unsigned)((grp * FC_CG + lc * 2) * sizeof(float2));
        for (int ch = 0; ch < nchunks; ch++) {
            const int stage = ch % FC_ST, use = ch / FC_ST;
            mbar_wait(bar0 + 8 * stage, use & 1);                     // the chunk's bytes have landed
            const unsigned fsa = fs_base + stage * F_STAGE;
            const unsigned tsa = ts_base + stage * T_STAGE;
            // this group's branches of the chunk: k = 2 kk + grp
#define FC_BRANCH_STEP(ROW_GUARD)                                                                       \
            for (int kk = 0; kk < FC_KC / 2; kk++) {                                                    \
                f32x2 t[4], s[4];                                                                       \
                lds2x64(t[0], t[1], tsa + (unsigned)(2 * kk * FC_CG * sizeof(float2)));                 \
                lds2x64(t[2], t[3], tsa + (unsigned)((2 * kk * FC_CG + 32) * sizeof(float2)));          \
                _Pragma("unroll") for (int c = 0; c < 4; c++) s[c] = swap2(t[c]);                       \
                _Pragma("unroll") for (int i = 0; i < 8; i++) {                                         \
                    if (ROW_GUARD) {                                                                    \
                        f32x2 fa, fb;                                                                   \
                        lds2x64(fa, fb, fsa + (unsigned)((2 * i * FC_KC + 2 * kk) * sizeof(float4)));   \
                        _Pragma("unroll") for (int c = 0; c < 4; c++) ffma2(acc[i][c], fa, t[c]);       \
                        _Pragma("unroll") for (int c = 0; c < 4; c++) ffma2(acc[i][c], fb, s[c]);       \
                    }                                                                                   \
                }                                                                                       \
            }
            if (ni == 8) {
#pragma unroll 2
                FC_BRANCH_STEP(true)
            } else {
#pragma unroll 1
                FC_BRANCH_STEP(i < ni)
            }
#undef FC_BRANCH_STEP
            __syncwarp();
            if (lane == 0) mbar_arrive(bar0 + 8 * (FC_ST + stage));   // this warp is done reading the slot
        }
    }
    // the odd-branch group hands its partial sums over through shared memory (every chunk has been consumed)
    __syncthreads();
    f32x2* red = reinterpret_cast<f32x2*>(fc_smem4);                  // [NW][32 accumulators][32 lanes]
    if (!producer && grp == 1) {
#pragma unroll
        for (int i = 0; i < 8; i++)
#pragma unroll
            for (int c = 0; c < 4; c++) red[(warp * 32 + i * 4 + c) * 32 + lane] = acc[i][c];
    }
    __syncthreads();
    if (!producer && grp == 0) {
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int row = warp * 16 + 2 * i + lr;
            float o[8];
#pragma unroll
            for (int c = 0; c < 4; c++) {
                float x0, y0, x1, y1;
                upk2(acc[i][c], x0, y0);
                upk2(red[(warp * 32 + i * 4 + c) * 32 + lane], x1, y1);
                o[2 * c] = x0 + x1; o[2 * c + 1] = y0 + y1;
            }
            if (row < rows) {
                float4* zr = reinterpret_cast<float4*>(Z + ((size_t)q * B + b0 + row) * slots + (size_t)cg * FC_CG) + lc;
                zr[0] = make_float4(o[0], o[1], o[2], o[3]);
                zr[16] = make_float4(o[4], o[5], o[6], o[7]);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// z[m] = (1/M) IFFT_M over q of Z[q][b][c]; valid m < Kb; post-rotation e^{j 2 pi (ph + rate (kD + 1))}; store s1.
// IFFT(x) = conj(FFT(conj(x))).
// ------------------------------------------------------------------------------------------------
template <int V>
__global__ void __launch_bounds__(V * FC_SEQ)
fc_inverse_kernel(const float2* __restrict__ Z, int nsplit, int B, int slots, int D, int Kb, const double* __restrict__ ch_rate,
                  const double* __restrict__ ch_phase, long long k0, long long n_k, float2* __restrict__ out,
                  const float* __restrict__ out_scale)
{
    constexpr int M = V * V;
    const float osc = out_scale ? __ldg(out_scale) : 1.0f / M;       // a power of two either way
    extern __shared__ float2 fc_smem[];
    float2* tw = fc_smem;
    float2* seqs = fc_smem + M;
    const int tid = threadIdx.x, j = tid & 31, g = tid >> 5;
    const int b = blockIdx.y;
    const int c = blockIdx.x * FC_SEQ + j;
    fc_fill_twiddles_v<V>(tw);
    float2 v[V];
#pragma unroll
    for (int n1 = 0; n1 < V; n1++) {
        const size_t at = ((size_t)(V * n1 + g) * B + b) * slots + c;
        float2 z = __ldg(Z + at);
        for (int sp = 1; sp < nsplit; sp++) {                      // split-K partial sums of the contraction
            const float2 zz = __ldg(Z + (size_t)sp * M * B * slots + at);
            z.x += zz.x; z.y += zz.y;
        }
        v[n1] = make_float2(z.x, -z.y);
    }
    __syncthreads();
    fc_fft_vv<V>(v, seqs + j * (M + 1), tw, g);
    const double rate = ch_rate[c], ph = ch_phase[c];
#pragma unroll
    for (int q = 0; q < V; q++) {
        const int m = g + V * slot<V>(q);
        const long long k = k0 + (long long)b * Kb + m;
        if (m < Kb && k < n_k) {
            double t = ph + rate * (double)(k * D + 1);
            t -= floor(t);
            float sn, cs;
            sincospif(2.0f * (float)t, &sn, &cs);
            const float2 z = make_float2(v[q].x * osc, -v[q].y * osc);
            out[(size_t)k * slots + c] = cmul(z, make_float2(cs, sn));
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Block scaling of the fp16 x 2 operand form: the largest |re|, |im| of the pass's input, then the two powers of two.
// Non-negative floats order like their bit patterns, so the running maximum is an atomicMax on unsigned.
// ------------------------------------------------------------------------------------------------
// CTA = 8192 consecutive samples (64 KB), CTAs in REVERSE order of the block: the forward FFTs that follow read the block
// from its start, so what this pass read last is what they need first and the 126 MB L2 still holds it.  Small fixed-size CTAs
// rather than a grid-stride loop: beside the other streams' kernels not every CTA of a persistent grid finds a slot at once,
// and a late one would run the whole duration again.
constexpr int FC_AMAX_CHUNK = 8192;
__global__ void __launch_bounds__(256)
fc_absmax_kernel(const float2* __restrict__ iq, long long n, unsigned* __restrict__ out)
{
    __shared__ float wmax[8];
    float m = 0.0f;
    const long long c0 = (long long)(gridDim.x - 1 - blockIdx.x) * FC_AMAX_CHUNK;
    const float2* p = iq + c0 + threadIdx.x;
    const int left = (int)min((long long)FC_AMAX_CHUNK, n - c0);
    if (left == FC_AMAX_CHUNK) {
#pragma unroll
        for (int k = 0; k < FC_AMAX_CHUNK / 256; k += 8) {          // eight independent loads in flight per thread
            float2 v[8];
#pragma unroll
            for (int u = 0; u < 8; u++) v[u] = __ldg(p + (k + u) * 256);
#pragma unroll
            for (int u = 0; u < 8; u++) m = fmaxf(m, fmaxf(fabsf(v[u].x), fabsf(v[u].y)));
        }
    } else {
        for (int i = threadIdx.x; i < left; i += 256) {
            const float2 v = __ldg(iq + c0 + i);
            m = fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y)));
        }
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {                                 // one atomic per CTA: same-address atomics serialise in L2
#pragma unroll
        for (int w = 1; w < 8; w++) m = fmaxf(m, wmax[w]);
        if (m > 0.0f) atomicMax(out, __float_as_uint(m));
    }
}

__global__ void fc_scale_kernel(const unsigned* __restrict__ absmax_bits, int M, float tab_scale, float* __restrict__ scale)
{
    const float a = __uint_as_float(*absmax_bits);
    int kf = 0;
    if (a > 0.0f && a < 3.0e38f) {
        // |F| <= M sqrt(2) max|x|;  2^kf = the largest power of two with M sqrt(2) max|x| 2^kf <= 2^15
        int e;
        frexpf(a * (float)M * 1.41421356f, &e);                       // a M sqrt2 = f 2^e, 0.5 <= f < 1  =>  < 2^e
        kf = max(-100, min(100, 15 - e));
    }
    scale[0] = ldexpf(1.0f, kf);
    scale[1] = ldexpf(1.0f / ((float)M * tab_scale), -kf);            // M and tab_scale are powers of two
}

constexpr size_t kFftSmem = (256 + FC_SEQ * FC_STR) * sizeof(float2);
constexpr size_t kFftSmemSmall = (FC_M_SMALL + FC_SEQ * (FC_M_SMALL + 1)) * sizeof(float2);

// ------------------------------------------------------------------------------------------------
// K4F band-pass kernels (see fastconv.cuh).  Streams are channel-minor ([row][slot]), so a warp's 32 lanes are 32
// adjacent channels and every access is a 256-byte row.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(16 * FC_SEQ)
bpf_forward_kernel(const float2* __restrict__ in, int slots, int last_row, int P, float2* __restrict__ X)
{
    extern __shared__ float2 fc_smem[];
    float2* tw = fc_smem;
    float2* seqs = fc_smem + 256;
    const int tid = threadIdx.x, lane = tid & 31, g = tid >> 5;
    const int ch = blockIdx.x * FC_SEQ + lane;
    const int jj = (int)blockIdx.y - P;                       // block index relative to output 0
    fc_fill_twiddles(tw);
    float2 v[16];
#pragma unroll
    for (int n1 = 0; n1 < 16; n1++) {
        const int row = min(BPF_H * (jj - 1) + 16 * n1 + g, last_row);
        v[n1] = __ldg(in + (ptrdiff_t)row * slots + ch);
    }
    __syncthreads();
    fc_fft256(v, seqs + lane * FC_STR, tw, g);
#pragma unroll
    for (int q = 0; q < 16; q++) {
        const int bin = g + 16 * slot<16>(q);
        X[((size_t)blockIdx.y * FC_M + bin) * slots + ch] = v[q];
    }
}

// Y[j][q][c] = sum_{p<P} X[j-p][q][c] * H[p][q][c]: a P-tap complex FIR along the block index for every (bin, channel).
// A thread owns one (bin, channel) and a segment of blocks; it slides the X window through registers.
template <int PP>
__global__ void __launch_bounds__(128)
bpf_mac_kernel(const float2* __restrict__ X, const float2* __restrict__ H, int slots, int nblk, int seg, float2* __restrict__ Y)
{
    constexpr int U = 5;                                              // outputs per window shift
    const size_t idx = (size_t)blockIdx.x * 128 + threadIdx.x;        // bin * slots + slot
    const size_t plane = (size_t)FC_M * slots;
    const int j0 = blockIdx.y * seg, j1 = min(nblk, j0 + seg);
    if (j0 >= j1) return;
    const float2* Xp = X + idx + (size_t)PP * plane;                  // Xp[j * plane] = X[j], j >= -PP
    float2 h[PP], w[PP + U - 1];                                      // w[k] = X[j + U - 1 - k] for the group starting at j
#pragma unroll
    for (int p = 0; p < PP; p++) h[p] = __ldg(H + (size_t)p * plane + idx);
#pragma unroll
    for (int k = U; k < PP + U - 1; k++) w[k] = __ldg(Xp + (ptrdiff_t)(j0 + U - 1 - k) * (ptrdiff_t)plane);
    float2 nx[U];
#pragma unroll
    for (int u = 0; u < U; u++) nx[u] = __ldg(Xp + (size_t)min(j0 + u, nblk - 1) * plane);
    for (int j = j0; j < j1; j += U) {
#pragma unroll
        for (int u = 0; u < U; u++) w[U - 1 - u] = nx[u];
        if (j + U < j1) {                                             // next group's spectra, in flight during the MACs
#pragma unroll
            for (int u = 0; u < U; u++) nx[u] = __ldg(Xp + (size_t)min(j + U + u, nblk - 1) * plane);
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
            float2 acc = make_float2(0.f, 0.f);
#pragma unroll
            for (int p = 0; p < PP; p++) {
                const float2 x = w[U - 1 - u + p];
                acc.x = fmaf(x.x, h[p].x, acc.x); acc.x = fmaf(-x.y, h[p].y, acc.x);
                acc.y = fmaf(x.x, h[p].y, acc.y); acc.y = fmaf(x.y, h[p].x, acc.y);
            }
            if (j + u < j1) Y[(size_t)(j + u) * plane + idx] = acc;
        }
#pragma unroll
        for (int k = PP + U - 2; k >= U; k--) w[k] = w[k - U];
    }
}

// generic partition count (window re-read from L2)
__global__ void __launch_bounds__(128)
bpf_mac_generic_kernel(const float2* __restrict__ X, const float2* __restrict__ H, int slots, int P, int nblk, float2* __restrict__ Y)
{
    const size_t idx = (size_t)blockIdx.x * 128 + threadIdx.x;
    const size_t plane = (size_t)FC_M * slots;
    const int j = blockIdx.y;
    if (j >= nblk) return;
    float2 acc = make_float2(0.f, 0.f);
    for (int p = 0; p < P; p++) {
        const float2 w = __ldg(X + (size_t)(j - p + P) * plane + idx), h = __ldg(H + (size_t)p * plane + idx);
        acc.x = fmaf(w.x, h.x, acc.x); acc.x = fmaf(-w.y, h.y, acc.x);
        acc.y = fmaf(w.x, h.y, acc.y); acc.y = fmaf(w.y, h.x, acc.y);
    }
    Y[(size_t)j * plane + idx] = acc;
}

__global__ void __launch_bounds__(16 * FC_SEQ)
bpf_inverse_kernel(const float2* __restrict__ Y, const float2* __restrict__ in, const int* __restrict__ enabled, int slots, int n_out,
                   float2* __restrict__ out)
{
    extern __shared__ float2 fc_smem[];
    float2* tw = fc_smem;
    float2* seqs = fc_smem + 256;
    const int tid = threadIdx.x, lane = tid & 31, g = tid >> 5;
    const int ch = blockIdx.x * FC_SEQ + lane;
    const int j = blockIdx.y;
    fc_fill_twiddles(tw);
    float2 v[16];
#pragma unroll
    for (int n1 = 0; n1 < 16; n1++) {
        const float2 y = __ldg(Y + ((size_t)j * FC_M + 16 * n1 + g) * slots + ch);
        v[n1] = make_float2(y.x, -y.y);
    }
    __syncthreads();
    fc_fft256(v, seqs + lane * FC_STR, tw, g);
    const bool en = enabled[ch] != 0;
#pragma unroll
    for (int q = 0; q < 16; q++) {
        const int n = g + 16 * slot<16>(q);
        const int row = BPF_H * j + n - BPF_H;
        if (n >= BPF_H && row < n_out) {
            const size_t o = (size_t)row * slots + ch;
            out[o] = en ? make_float2(v[q].x * (1.0f / FC_M), -v[q].y * (1.0f / FC_M)) : __ldg(in + o);   // disabled: pass through
        }
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// 2D row-major float32 tensor [rows][cols] with a (box_cols x box_rows) tile
int make_map(CUtensorMap* map, const void* base, size_t cols, size_t rows, unsigned box_cols, unsigned box_rows)
{
    static EncodeTiledFn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qr;
        OWRX_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr));
        if (!fn || qr != cudaDriverEntryPointSuccess) return fail(OWRX_E_CUDA, "cuTensorMapEncodeTiled is not available");
        encode = reinterpret_cast<EncodeTiledFn>(fn);
    }
    const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)cols * sizeof(float)};
    const cuuint32_t box[2] = {box_cols, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(OWRX_E_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    return OWRX_OK;
}

template <int NW>
int launch_contract_nw(const FcShape& sh, const float4* F, const float2* tab, int B, float2* Z, int nsplit, cudaStream_t st)
{
    constexpr int BT = 16 * NW;
    const size_t smem = (size_t)FC_ST * (BT * FC_KC * sizeof(float4) + FC_KC * FC_CG * sizeof(float2));
    OWRX_CUDA(cudaFuncSetAttribute(fc_contract_kernel<NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int nbt = (B + BT - 1) / BT;
    CUtensorMap mapF, mapT;
    int rc;
    if ((rc = make_map(&mapF, F, (size_t)sh.Dp * 4, (size_t)sh.M * B, FC_KC * 4, BT)) != OWRX_OK) return rc;
    if ((rc = make_map(&mapT, tab, (size_t)sh.slots * 2, (size_t)sh.M * sh.Dp, FC_CG * 2, FC_KC)) != OWRX_OK) return rc;
    fc_contract_kernel<NW><<<dim3((unsigned)(sh.M * nbt), (unsigned)(sh.slots / FC_CG), (unsigned)nsplit), NW * 64 + 32, smem, st>>>(mapF, mapT, Z, B, sh.Dp,
                                                                                                                                     sh.slots, nbt, nsplit, sh.M);
    OWRX_LAUNCH_CHECK();
    return OWRX_OK;
}

}  // namespace

int fc_pick_fft_size(int D, int P, int force_m)
{
    if ((force_m == FC_M || force_m == FC_M_SMALL) && P <= force_m / 2) return force_m;
    return (D >= 2048 && P <= FC_M_SMALL / 2) ? FC_M_SMALL : FC_M;
}

int fc_launch_table(const FcShape& sh, const float* d_h, const int* d_slot_list, const double* d_rate_list, int n, float2* d_tab,
                    cudaStream_t st)
{
    if (n <= 0) return OWRX_OK;
    const long long total = (long long)sh.M * sh.D;
    fc_table_kernel<0><<<dim3((unsigned)((total + 255) / 256), (unsigned)n), 256, 0, st>>>(d_h, sh.T, sh.D, sh.Dp, sh.P, sh.slots, sh.M, d_slot_list,
                                                                                          d_rate_list, d_tab, 1.0f);
    OWRX_LAUNCH_CHECK();
    return OWRX_OK;
}

int fc_launch_table_tc(const FcShape& sh, const float* d_h, const int* d_slot_list, const double* d_rate_list, int n, void* d_tabp,
                       float tab_scale, cudaStream_t st)
{
    if (n <= 0) return OWRX_OK;
    const long long total = (long long)sh.M * sh.D;
    const dim3 grid((unsigned)((total + 255) / 256), (unsigned)n);
    if (sh.tc_levels == 2)
        fc_table_kernel<2><<<grid, 256, 0, st>>>(d_h, sh.T, sh.D, sh.Dp, sh.P, sh.slots, sh.M, d_slot_list, d_rate_list, d_tabp, tab_scale);
    else
        fc_table_kernel<3><<<grid, 256, 0, st>>>(d_h, sh.T, sh.D, sh.Dp, sh.P, sh.slots, sh.M, d_slot_list, d_rate_list, d_tabp, 1.0f);
    OWRX_LAUNCH_CHECK();
    return OWRX_OK;
}

int fc_pick_tc_levels(int D, int force_levels)
{
    if (force_levels == 2 || force_levels == 3) return force_levels;
    // fp16 x 2 pays where the contraction is what a pass costs — large decimations: few outputs per table entry (C3: 2.83 ->
    // 2.05 ms per step).  With a short decimation (C2, C5) the contraction is a third of the FIR chain, the chain is not what
    // bounds the step, and the extra read of the input for max|x| costs the other streams what the smaller operands save.
    return D >= 2048 ? 2 : 3;
}

float fc_tab_scale(const FcShape& sh, const float* h_taps)
{
    if (sh.tc_levels != 2) return 1.0f;
    // |Tab[q][r]| <= sum_s |h[D s + r]|
    double bound = 0.0;
    for (int r = 0; r < sh.D; r++) {
        double a = 0.0;
        for (int t = r; t < sh.T; t += sh.D) a += fabs((double)h_taps[t]);
        bound = std::max(bound, a);
    }
    if (!(bound > 0.0) || !std::isfinite(bound)) return 1.0f;
    int e;
    frexp(bound, &e);                                                 // bound < 2^e
    return ldexpf(1.0f, std::max(-100, std::min(100, 14 - e)));
}

int fc_launch_scale(const FcShape& sh, const float2* iq, long long n, float tab_scale, unsigned* d_work, float* d_scale, cudaStream_t st)
{
    OWRX_CUDA(cudaMemsetAsync(d_work, 0, sizeof(unsigned), st));
    if (sh.tc_levels == 2 && n > 0) {
        const unsigned blocks = (unsigned)((n + FC_AMAX_CHUNK - 1) / FC_AMAX_CHUNK);
        fc_absmax_kernel<<<blocks, 256, 0, st>>>(iq, n, d_work);
        OWRX_LAUNCH_CHECK();
    }
    // levels = 3: the maximum stays 0 => scale (1, 1 / M)
    fc_scale_kernel<<<1, 1, 0, st>>>(d_work, sh.M, sh.tc_levels == 2 ? tab_scale : 1.0f, d_scale);
    OWRX_LAUNCH_CHECK();
    return OWRX_OK;
}

int fc_launch_forward(const FcShape& sh, const float2* iq, long long n_lim, int B, float4* d_F, cudaStream_t st)
{
    if (sh.M == FC_M_SMALL) {
        fc_forward_kernel<0, 8><<<dim3((unsigned)(sh.Dp / FC_SEQ), (unsigned)B), 8 * FC_SEQ, kFftSmemSmall, st>>>(iq, n_lim, sh.D, sh.Dp, sh.Kb, B, d_F,
                                                                                                             nullptr);
    } else {
        OWRX_CUDA(cudaFuncSetAttribute(fc_forward_kernel<0, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFftSmem));
        fc_forward_kernel<0, 16><<<dim3((unsigned)(sh.Dp / FC_SEQ), (unsigned)B), 16 * FC_SEQ, kFftSmem, st>>>(iq, n_lim, sh.D, sh.Dp, sh.Kb, B, d_F,
                                                                                                            nullptr);
    }
    OWRX_LAUNCH_CHECK();
    return OWRX_OK;
}

template <int TC>
static int launch_forward_tc(const FcShape& sh, const float2* iq, long long n_lim, int B, void* d_Fp, const float* d_scale, cudaStream_t st)
{
    const dim3 grid((unsigned)(sh.Dp / FC_SEQ), (unsigned)B);
    if (sh.M == FC_M_SMALL) {
        fc_forward_kernel<TC, 8><<<grid, 8 * FC_SEQ, kFftSmemSmall, st>>>(iq, n_lim, sh.D, sh.Dp, sh.Kb, B, d_Fp, d_scale);
    } else {
        OWRX_CUDA(cudaFuncSetAttribute(fc_forward_kernel<TC, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFftSmem));
        fc_forward_kernel<TC, 16><<<grid, 16 * FC_SEQ, kFftSmem, st>>>(iq, n_lim, sh.D, sh.Dp, sh.Kb, B, d_Fp, d_scale);
    }
    OWRX_LAUNCH_CHECK();
    return OWRX_OK;
}

int fc_launch_forward_tc(const FcShape& sh, const float2* iq, long long n_lim, int B, void* d_Fp, const float* d_scale, cudaStream_t st)
{
    return sh.tc_levels == 2 ? launch_forward_tc<2>(sh, iq, n_lim, B, d_Fp, d_scale, st) : launch_forward_tc<3>(sh, iq, n_lim, B, d_Fp, d_scale, st);
}

// CTA shape and split-K factor for B blocks: as few row tiles as 96-row CTAs allow, the smallest CTA that covers them, and
// the split (<= FC_MAXSPLIT) that wastes the least of the last wave
void fc_contract_plan(const FcShape& sh, int B, int sm_count, int* nw_out, int* nsplit_out)
{
    const int nbt0 = (B + 95) / 96;
    const int nw = std::max(1, std::min(6, ((B + nbt0 - 1) / nbt0 + 15) / 16));
    const int nbt = (B + 16 * nw - 1) / (16 * nw);
    const size_t smem = (size_t)FC_ST * (16 * nw * FC_KC * sizeof(float4) + FC_KC * FC_CG * sizeof(float2));
    const int per_sm = std::max(1, std::min((int)((size_t)(220 << 10) / smem), 2048 / (nw * 64 + 32)));
    const long long tiles = (long long)sh.M * nbt * (sh.slots / FC_CG), slots = (long long)sm_count * per_sm;
    const int chunks = sh.Dp / FC_KC;
    int best = 1;
    double best_cost = 1e30;
    for (int sp = 1; sp <= std::min(FC_MAXSPLIT, chunks); sp++) {
        // waves of CTAs, each 1/sp of a tile plus a fixed prologue/epilogue worth about three chunks (measured: with 27
        // chunks per tile, C2, splitting only moves the cost into the ring fill and the extra Z planes)
        const double cost = (double)((tiles * sp + slots - 1) / slots) * (1.0 / sp + 3.0 / chunks);
        if (cost < best_cost * 0.97) { best_cost = cost; best = sp; }
    }
    *nw_out = nw;
    *nsplit_out = best;
}

int fc_launch_contract(const FcShape& sh, const float4* d_F, const float2* d_tab, int B, float2* d_Z, int sm_count, int* nsplit_out, cudaStream_t st)
{
    int nw, nsplit;
    fc_contract_plan(sh, B, sm_count, &nw, &nsplit);
    *nsplit_out = nsplit;
    switch (nw) {
    case 1: return launch_contract_nw<1>(sh, d_F, d_tab, B, d_Z, nsplit, st);
    case 2: return launch_contract_nw<2>(sh, d_F, d_tab, B, d_Z, nsplit, st);
    case 3: return launch_contract_nw<3>(sh, d_F, d_tab, B, d_Z, nsplit, st);
    case 4: return launch_contract_nw<4>(sh, d_F, d_tab, B, d_Z, nsplit, st);
    case 5: return launch_contract_nw<5>(sh, d_F, d_tab, B, d_Z, nsplit, st);
    default: return launch_contract_nw<6>(sh, d_F, d_tab, B, d_Z, nsplit, st);
    }
}

int bpf_launch_forward(const float2* in, int slots, int last_row, int P, int nblk, float2* X, cudaStream_t st)
{
    OWRX_CUDA(cudaFuncSetAttribute(bpf_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFftSmem));
    bpf_forward_kernel<<<dim3((unsigned)(slots / FC_SEQ), (unsigned)(nblk + P)), 16 * FC_SEQ, kFftSmem, st>>>(in, slots, last_row, P, X);
    OWRX_LAUNCH_CHECK();
    return OWRX_OK;
}

int bpf_launch_mac(const float2* X, const float2* H, int slots, int P, int nblk, float2* Y, cudaStream_t st)
{
    const unsigned gx = (unsigned)((size_t)FC_M * slots / 128);
    // enough block segments to fill the machine; each segment re-reads P-1 warm-up spectra
    const int nseg = std::max(1, std::min((nblk + 4 * P - 1) / (4 * P), (int)(4 * 148 / std::max(1u, gx)) + 1));
    const int seg = (nblk + nseg - 1) / nseg;
    const dim3 grid(gx, (unsigned)((nblk + seg - 1) / seg));
    switch (P) {
    case 1: bpf_mac_kernel<1><<<grid, 128, 0, st>>>(X, H, slots, nblk, seg, Y); break;
    case 2: bpf_mac_kernel<2><<<grid, 128, 0, st>>>(X, H, slots, nblk, seg, Y); break;
    case 5: bpf_mac_kernel<5><<<grid, 128, 0, st>>>(X, H, slots, nblk, seg, Y); break;
    case 25: bpf_mac_kernel<25><<<grid, 128, 0, st>>>(X, H, slots, nblk, seg, Y); break;
    default: bpf_mac_generic_kernel<<<dim3(gx, (unsigned)nblk), 128, 0, st>>>(X, H, slots, P, nblk, Y); break;
    }
    OWRX_LAUNCH_CHECK();
    return OWRX_OK;
}

int bpf_launch_inverse(const float2* Y, const float2* in, const int* enabled, int slots, int nblk, int n_out, float2* out, cudaStream_t st)
{
    OWRX_CUDA(cudaFuncSetAttribute(bpf_inverse_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFftSmem));
    bpf_inverse_kernel<<<dim3((unsigned)(slots / FC_SEQ), (unsigned)nblk), 16 * FC_SEQ, kFftSmem, st>>>(Y, in, enabled, slots, n_out, out);
    OWRX_LAUNCH_CHECK();
    return OWRX_OK;
}

int fc_launch_inverse(const FcShape& sh, const float2* d_Z, int nsplit, int B, const double* d_rate, const double* d_phase, long long k0, long long n_k,
                      float2* out, const float* d_out_scale, cudaStream_t st)
{
    const dim3 grid((unsigned)(sh.slots / FC_SEQ), (unsigned)B);
    if (sh.M == FC_M_SMALL) {
        fc_inverse_kernel<8><<<grid, 8 * FC_SEQ, kFftSmemSmall, st>>>(d_Z, nsplit, B, sh.slots, sh.D, sh.Kb, d_rate, d_phase, k0, n_k, out, d_out_scale);
    } else {
        OWRX_CUDA(cudaFuncSetAttribute(fc_inverse_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFftSmem));
        fc_inverse_kernel<16><<<grid, 16 * FC_SEQ, kFftSmem, st>>>(d_Z, nsplit, B, sh.slots, sh.D, sh.Kb, d_rate, d_phase, k0, n_k, out, d_out_scale);
    }
    OWRX_LAUNCH_CHECK();
    return OWRX_OK;
}

}  // namespace owrx
