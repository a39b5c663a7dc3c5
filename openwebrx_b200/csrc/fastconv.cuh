// fastconv.cuh — K3F: Shift + FirDecimate of every client channel as a polyphase fast convolution.
//
// Same arithmetic contract as K3 (selector_kernels.cuh / SURVEY Appendix A.6-A.7):
//   y_c[k] = sum_{t<T} x[kD+t] * e^{j 2 pi (ph_c + rate_c (kD+t+1))} * h[t]
//          = e^{j 2 pi (ph_c + rate_c (kD+1))} * z_c[k],   z_c[k] = sum_t g_c[t] x[kD+t],  g_c[t] = h[t] e^{j 2 pi rate_c t}
// With t = D s + r (polyphase branch r, s < P = ceil(T/D)) and x_r[a] = x[D a + r]:
//   z_c[k] = sum_{r<D} sum_{s<P} g_c[D s + r] x_r[k + s]
// i.e. D short correlations at the OUTPUT rate.  Each is evaluated with M-point FFTs (overlap-save, block of
// M branch samples -> Kb = M-P+1 outputs):
//   F_b[q][r]   = FFT_M over a of x[(b Kb + a) D + r]                    (shared by ALL channels)        fc_forward_kernel
//   Z_b[q][c]   = sum_r F_b[q][r] * Tab[q][r][c]                         (dense contraction, K = D)      fc_contract_kernel
//   z_c[bKb+m]  = (1/M) IFFT_M over q of Z_b[q][c],  m < Kb, then the post-rotation                    fc_inverse_kernel
//   Tab[q][r][c] = sum_s g_c[D s + r] e^{+j 2 pi q s / M}                (rebuilt when a channel retunes) fc_table_kernel
// Exact (no bin slicing: every alias of the decimation is carried by the per-branch FFTs), works for any D, and
// costs 4 M/Kb ~ 4.5 FMA per input sample per channel instead of the direct form's 2 T/D ~ 53.
#pragma once
#include "common.cuh"

namespace owrx {

constexpr int FC_M = 256;        // branch FFT size (default; also the block size of the K4F band-pass)
constexpr int FC_M_SMALL = 64;   // branch FFT size of groups with a large decimation (fc_pick_fft_size)
constexpr int FC_KC = 32;        // contraction chunk (branches per pipeline stage)
constexpr int FC_DPAD = 32;      // D is padded to a multiple of this (forward pass: 32 branches per CTA)
constexpr int FC_CG = 64;        // channel slots per contraction CTA
constexpr int FC_MAXSPLIT = 4;   // split-K planes of Z (scratch is sized for this many)

struct FcShape {
    int D, T, P, Kb, Dp, slots;
    int M;                       // branch FFT size: FC_M or FC_M_SMALL; Kb = M - P + 1
    int tc_levels;               // operand split of the tensor-core form: 2 = fp16 x 2 (block-scaled), 3 = bf16 x 3
};

// Branch FFT size of a group.  Bytes a pass moves ~ 12 M Dp (S + 2 n_k / (M - P + 1)): the per-channel table (M Dp S entries,
// read once per pass) against the branch spectra (written and read once, M / Kb times the input).  With D in the thousands
// a pass holds few outputs n_k per channel slot S and the table dominates: 64-point FFTs (Kb = 38 at P = 27) cut the table
// to a quarter for 1.5 times the spectra (C3, D = 5120, 2^25 samples: 16.4 -> 5.3 GB at 1024 slots, 2.9 -> 1.9 GB at 128).
// Short decimations keep 256 points (C2, D = 833, 64 slots: 61 vs 90 k per unit).  force_m = 64 | 256 overrides (when P fits).
int fc_pick_fft_size(int D, int P, int force_m);

// rebuild the table columns of `n` slots: slot_list[i], rate_list[i] (device arrays)
int fc_launch_table(const FcShape& sh, const float* d_h, const int* d_slot_list, const double* d_rate_list, int n, float2* d_tab,
                    cudaStream_t st);
// F[q][b][r] (stored as the packed-FMA operand (re, re, -im, im)) for blocks b < B of the stream starting at iq (sample 0 = first tap of output 0)
int fc_launch_forward(const FcShape& sh, const float2* iq, long long n_lim, int B, float4* d_F, cudaStream_t st);
// d_Z holds FC_MAXSPLIT planes of [M][B][slots]; *nsplit = how many partial-sum planes this launch wrote
int fc_launch_contract(const FcShape& sh, const float4* d_F, const float2* d_tab, int B, float2* d_Z, int sm_count, int* nsplit, cudaStream_t st);
// out[(k0 + b Kb + m) * slots + c] for k0 + b Kb + m < n_k; phases are relative to iq[-1] of the whole call
// d_out_scale: device float the result is multiplied by instead of 1 / M (fc_launch_scale's d_scale + 1), or nullptr
int fc_launch_inverse(const FcShape& sh, const float2* d_Z, int nsplit, int B, const double* d_rate, const double* d_phase, long long k0,
                      long long n_k, float2* out, const float* d_out_scale, cudaStream_t st);

// ---- tensor-core form of the contraction (fastconv_tc.cu): every float operand as `levels` 16-bit terms, real and imaginary
// parts in separate K-major planes, plane p = 2 * level + part:
//   Fp[p][q * B + b][r]  (fc_tc_plane_elems_F 16-bit words per plane)      Tp[p][q * slots + c][r]  (fc_tc_plane_elems_tab per plane)
//   levels = 3: x = h + m + l in bf16 (float's exponent range, no scaling), six partial products;
//   levels = 2 (default of groups with a large decimation): x = h + m in fp16 (11 + 11 significand bits), three partial products hh + hm + mh — half the tensor-pipe
//     work and two thirds of the operand bytes.  fp16 has 5 exponent bits, so both operands are scaled by exact powers of two:
//     the table by 2^kt with max_r sum_s |h[D s + r]| * 2^kt <= 2^14 (fc_tab_scale, host, from the taps), the spectra of a pass by
//     2^kf with M * sqrt(2) * max|x| * 2^kf <= 2^15, max|x| measured over the pass's input by fc_launch_scale (one extra read
//     of the block); the inverse FFT multiplies by 2^-(kf + kt) / M.  Powers of two commute with every rounding in between,
//     so the result does not depend on the scale and IF(x / 2) == IF(x) / 2 stays exact.
constexpr int FC_TC_MAXPLANES = 6;
inline int fc_tc_planes(const FcShape& sh) { return 2 * sh.tc_levels; }
// operand split of a new group: fp16 x 2 for D >= 2048, else bf16 x 3; force_levels = 2 | 3 overrides
int fc_pick_tc_levels(int D, int force_levels);
// exact power of two 2^kt for the table of a group with these taps (1 for levels = 3)
float fc_tab_scale(const FcShape& sh, const float* h_taps);
size_t fc_tc_plane_elems_F(const FcShape& sh, int B);
size_t fc_tc_plane_elems_tab(const FcShape& sh);
int fc_launch_table_tc(const FcShape& sh, const float* d_h, const int* d_slot_list, const double* d_rate_list, int n, void* d_tabp,
                       float tab_scale, cudaStream_t st);
// levels = 2 only: d_scale[0] = 2^kf (what the forward pass multiplies by), d_scale[1] = 2^-(kf + kt) / M (the inverse pass).
// d_work: 4 bytes of device scratch (the running maximum)
int fc_launch_scale(const FcShape& sh, const float2* iq, long long n, float tab_scale, unsigned* d_work, float* d_scale, cudaStream_t st);
int fc_launch_forward_tc(const FcShape& sh, const float2* iq, long long n_lim, int B, void* d_Fp, const float* d_scale, cudaStream_t st);
// force_form: 0 = blocks in the MMA's M, 1 = slots in M, < 0 = whichever the cycle model picks
int fc_launch_contract_tc(const FcShape& sh, const void* d_Fp, const void* d_tabp, int B, float2* d_Z, int sm_count, int force_form,
                          int* nsplit, cudaStream_t st);

// ------------------------------------------------------------------------------------------------
// K4F: Bandpass (csdr/chain/selector.py:115-117,159-166; per-channel complex taps at the selector output rate) as a
// uniformly partitioned overlap-save convolution on 256-point FFTs: the T taps are cut into P = ceil(T/128) partitions
// of 128, H[p] = FFT_256([h_p | 0]);  X[j] = FFT_256 of input rows [128(j-1), 128(j+1));  Y[j] = sum_p X[j-p] H[p];
// output rows [128 j, 128(j+1)) = last half of IFFT_256(Y[j]).  4 P complex MACs per output instead of T
// (T = 3125 at the 250 kHz WFM IF: 100 instead of 3125).  The reference computes the same linear convolution by FFT
// overlap-add (Bandpass(use_fft=True)).
// ------------------------------------------------------------------------------------------------
constexpr int BPF_H = 128;       // hop / partition length
// X[(j + P) * 256 + q][slot] for j in [-P, nblk): rows are relative to `in` (row 0 = output 0; >= 128 (P+1) history rows before it);
// rows past last_row are clamped (they only reach outputs that are not stored)
int bpf_launch_forward(const float2* in, int slots, int last_row, int P, int nblk, float2* X, cudaStream_t st);
int bpf_launch_mac(const float2* X, const float2* H, int slots, int P, int nblk, float2* Y, cudaStream_t st);
int bpf_launch_inverse(const float2* Y, const float2* in, const int* enabled, int slots, int nblk, int n_out, float2* out, cudaStream_t st);

}  // namespace owrx
