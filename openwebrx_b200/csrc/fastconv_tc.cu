// fastconv_tc.cu — K3F-b on the 5th-generation tensor cores (tcgen05 + TMEM + TMA), sm_100a only.
//
// Same contraction as fc_contract_kernel (fastconv.cu): Z[q][b][c] = sum_{r<Dp} F[q][b][r] * Tab[q][r][c], complex, the
// per-channel half of pycsdr Shift + FirDecimate (reference call sites csdr/chain/selector.py:29,57,95,140).  Per bin q it
// is a dense GEMM [B blocks x Dp branches] . [Dp x slots] — the "true dense contraction" north_star asks for before
// tensor cores may be used.  FP32 results are required (1e-4 relative RMS on channels up to 50 dB below the wideband
// power), so every FP32 operand is carried as several 16-bit terms and the product is assembled from the partial products
// that matter, accumulated in FP32 in TMEM (fastconv.cuh, FcShape::tc_levels):
//   2 levels (default): block-scaled fp16, x 2^k = h + m (11 + 11 significand bits), products hh + hm + mh;
//   3 levels: bf16, x = h + m + l (8 + 8 + 8 bits, float's exponent range, no scaling), products hh, hm, mh, hl, lh, mm
//             (the "bf16x9" scheme minus its three smallest terms) — twice the tensor-pipe work, 1.5 x the bytes.
//
// Complex arithmetic without duplicating an operand in HBM: real and imaginary parts are separate planes,
//   D1 = F_re . [T_re | T_im]   (TMEM columns   0..127)         D2 = F_im . [T_re | T_im]   (TMEM columns 128..255)
//   Z_re = D1[:, c] - D2[:, 64 + c]        Z_im = D1[:, 64 + c] + D2[:, c]        (combined by the epilogue warps)
// so both MMAs of a product share one B descriptor and every instruction is M128 x N128 x K16 (fc_contract_tc_kernel:
// overlap-save blocks in the MMA's M, 64 slots per CTA); fc_contract_tct_kernel exchanges the roles (128 channel slots in M,
// the blocks in N) for passes with few blocks — see there.
//
// Operand planes (K-major, written by fc_forward_kernel<TC> / fc_table_kernel<TC>), plane p = 2 * level + part:
//   Fp[p][q * B + b][r]        Tp[p][q * slots + c][r]            r < Dp contiguous
// CTA = (bin q, row tile of <= 128 blocks, 64 or 128 channel slots, split-K plane).  Warp 0: TMA producer (one 3D box per
// operand and stage: 16 branches x rows x planes, SWIZZLE_32B).  Warp 1: TMEM allocation + MMA issue (one thread;
// tcgen05.commit releases the stage).  Warps 2-5: epilogue (tcgen05.ld -> combine -> Z).
#include "fastconv.cuh"

#include <cuda.h>
#include <cuda_bf16.h>

#include <algorithm>

namespace owrx {

namespace {

constexpr unsigned TC_COLS = 256;                           // TMEM columns: D1 | D2
constexpr int TC_KC = 16;                                   // branches per ring stage: one K = 16 MMA step
constexpr unsigned TC_ROWB = 2 * TC_KC;                     // bytes per operand row of a stage: one SWIZZLE_32B atom

__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "TC_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra TC_DONE;\n"
        "bra TC_WAIT;\n"
        "TC_DONE:\n"
        "}\n" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_3d(unsigned dst, const CUtensorMap* map, int c0, int c1, int c2, unsigned bar)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];\n" ::"r"(dst),
                 "l"(reinterpret_cast<unsigned long long>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void umma_commit(unsigned bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(unsigned taddr, float* v)
{
    unsigned r[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
                   "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 16; i++) v[i] = __uint_as_float(r[i]);
}

constexpr int TT_MAXST = 8;                                 // most ring stages (mbarrier slots)

__device__ __forceinline__ void umma_desc(unsigned tmem_d, unsigned long long da, unsigned long long db, unsigned idesc, unsigned accumulate)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate)
        : "memory");
}
// K-major shared-memory matrix descriptor (cute::UMMA::SmemDescriptor) for operand rows of TC_ROWB = 32 bytes — one SWIZZLE_32B
// atom along K: start >> 4 in [0,14), LBO unused, SBO = 8 rows >> 4 in [32,46), version 1 in [46,48), layout type 6 in [61,64)
__device__ __forceinline__ unsigned long long smem_desc_rows(unsigned addr)
{
    return (unsigned long long)((addr & 0x3FFFFu) >> 4) | ((unsigned long long)((8u * TC_ROWB) >> 4) << 32) | (1ull << 46) | (6ull << 61);
}

// the partial products (A level, B level), smallest first: three levels (bf16) keep the six of weight > 2^-24, two levels (fp16)
// the three of weight > 2^-22
__constant__ int kTcProd3[6][2] = {{1, 1}, {2, 0}, {0, 2}, {1, 0}, {0, 1}, {0, 0}};
__constant__ int kTcProd2[3][2] = {{1, 0}, {0, 1}, {0, 0}};
// instruction descriptor (cute::UMMA::InstrDescriptor): D = F32 (1 << 4), A and B formats at bits 7 and 10 (0 = F16, 1 = BF16),
// both K-major, N >> 3 at bit 17, M >> 4 at bit 24
__device__ __forceinline__ unsigned tc_idesc(int levels, unsigned n)
{
    const unsigned fmt = levels == 3 ? 1u : 0u;
    return (1u << 4) | (fmt << 7) | (fmt << 10) | ((n >> 3) << 17) | ((128u >> 4) << 24);
}

// With 16-branch stages (TC_KC) three stages of a 64-slot x 88-block tile are 88 KB, so TWO CTAs share an SM (256 TMEM columns
// each): C2's 256 tiles are all resident at once — no second, 73 %-full wave — and an SM keeps two operand streams in flight.
__global__ void __launch_bounds__(192, 2)
fc_contract_tc_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, float2* __restrict__ Z, int B, int Dp,
                      int slots, int nbt, int mrows, int nsplit, int M, int nst, int levels)
{
    extern __shared__ unsigned char tc_smem_raw[];
    __shared__ unsigned long long bars[2 * TT_MAXST + 1];            // full[nst], empty[nst], accumulators ready
    __shared__ unsigned tmem_slot;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    // channel groups fastest: the CTAs that share a spectra tile (same bin and row tile, different 64-slot groups) are launched
    // side by side, so the tile is read from DRAM once and from L2 by the others
    const int ngroups = slots / FC_CG;
    const int cg = blockIdx.x % ngroups;
    const int q = (blockIdx.x / ngroups) / nbt, bt = (blockIdx.x / ngroups) % nbt;
    const int b0 = bt * mrows;
    const int rows = min(mrows, B - b0);
    const int all_chunks = Dp / TC_KC;
    const int ch0 = (int)(((long long)all_chunks * blockIdx.z) / nsplit);
    const int nchunks = (int)(((long long)all_chunks * (blockIdx.z + 1)) / nsplit) - ch0;
    Z += (size_t)blockIdx.z * M * B * slots;

    const unsigned npl = 2u * (unsigned)levels;                      // operand planes: levels x (re, im)
    const unsigned a_plane = (unsigned)mrows * TC_ROWB;              // mrows is a multiple of 8: every plane starts on a swizzle atom
    const unsigned a_stage = npl * a_plane;
    const unsigned b_plane = FC_CG * TC_ROWB;
    const unsigned stage_bytes = a_stage + npl * b_plane;
    const unsigned smem0 = ((unsigned)__cvta_generic_to_shared(tc_smem_raw) + 1023u) & ~1023u;
    const unsigned bar0 = (unsigned)__cvta_generic_to_shared(bars);
    const unsigned bar_acc = bar0 + 8 * (2 * TT_MAXST);

    if (tid == 0) {
        for (int s = 0; s < nst; s++) {
            mbar_init(bar0 + 8 * s, 1);                               // full: the producer's expect_tx arrival
            mbar_init(bar0 + 8 * (TT_MAXST + s), 1);                  // empty: one tcgen05.commit arrival
        }
        mbar_init(bar_acc, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (wid == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(&tmem_slot)),
                     "r"(TC_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const unsigned tmem = tmem_slot;

    if (wid == 0) {
        if (lane == 0) {
            int stage = 0;
            unsigned phase = 0;
            for (int ch = 0; ch < nchunks; ch++) {
                const unsigned full = bar0 + 8 * stage, empty = bar0 + 8 * (TT_MAXST + stage);
                mbar_wait(empty, phase ^ 1);                          // the MMAs that read this slot have completed
                mbar_expect_tx(full, stage_bytes);
                const unsigned sa = smem0 + stage * stage_bytes;
                // rows past the tile's last block come from the next bin (or are zero-filled past the tensor): they only
                // feed accumulator rows that are never stored
                tma_load_3d(sa, &mapA, (ch0 + ch) * TC_KC, q * B + b0, 0, full);
                tma_load_3d(sa + a_stage, &mapB, (ch0 + ch) * TC_KC, q * slots + cg * FC_CG, 0, full);
                if (++stage == nst) { stage = 0; phase ^= 1; }
            }
        }
        __syncwarp();
    } else if (wid == 1) {
        if (lane == 0) {
            const unsigned idesc = tc_idesc(levels, 128u);
            const int nprod = levels == 3 ? 6 : 3;
            int stage = 0;
            unsigned phase = 0;
            for (int ch = 0; ch < nchunks; ch++) {
                mbar_wait(bar0 + 8 * stage, phase);                   // the stage's bytes have landed
                asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                const unsigned sa = smem0 + stage * stage_bytes, sb = sa + a_stage;
                for (int p = 0; p < nprod; p++) {
                    const int la = levels == 3 ? kTcProd3[p][0] : kTcProd2[p][0], lb = levels == 3 ? kTcProd3[p][1] : kTcProd2[p][1];
                    const unsigned long long d_re = smem_desc_rows(sa + (unsigned)(2 * la) * a_plane);
                    const unsigned long long d_im = smem_desc_rows(sa + (unsigned)(2 * la + 1) * a_plane);
                    const unsigned long long d_b = smem_desc_rows(sb + (unsigned)(2 * lb) * b_plane);
                    const unsigned acc = (ch | p) != 0;
                    umma_desc(tmem, d_re, d_b, idesc, acc);           // D1 += F_re . [T_re | T_im]
                    umma_desc(tmem + 128, d_im, d_b, idesc, acc);     // D2 += F_im . [T_re | T_im]
                }
                umma_commit(bar0 + 8 * (TT_MAXST + stage));           // slot free once these MMAs have read it
                if (++stage == nst) { stage = 0; phase ^= 1; }
            }
            umma_commit(bar_acc);                                     // accumulators complete
        }
        __syncwarp();
    } else {
        // epilogue: warp w may touch TMEM lanes 32 (w % 4) .. +31; thread <-> row (block) of the tile
        const int quarter = wid & 3;
        const int row = quarter * 32 + lane;
        mbar_wait(bar_acc, 0);
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
        const unsigned trow = tmem + ((unsigned)(quarter * 32) << 16);
        float4* zr = reinterpret_cast<float4*>(Z + ((size_t)q * B + b0 + row) * slots + (size_t)cg * FC_CG);
#pragma unroll 1
        for (int c0 = 0; c0 < FC_CG; c0 += 16) {
            float d1r[16], d1i[16], d2r[16], d2i[16];
            tmem_ld16(trow + c0, d1r);                                // F_re . T_re
            tmem_ld16(trow + 64 + c0, d1i);                           // F_re . T_im
            tmem_ld16(trow + 128 + c0, d2r);                          // F_im . T_re
            tmem_ld16(trow + 192 + c0, d2i);                          // F_im . T_im
            asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
            if (row < rows) {
#pragma unroll
                for (int i = 0; i < 16; i += 2)
                    zr[(c0 + i) >> 1] = make_float4(d1r[i] - d2i[i], d1i[i] + d2r[i], d1r[i + 1] - d2i[i + 1], d1i[i + 1] + d2r[i + 1]);
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (wid == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem), "r"(TC_COLS) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------
// The same contraction with the operand roles exchanged ("slots in M"): A = table tile of 128 channel slots, B = the
// spectra rows of a tile of <= 128 overlap-save blocks, re and im planes stacked along N (they are adjacent in the stage):
//   D1 = T_re . [F_re | F_im]^T  (TMEM columns 0 .. 2 mrows)        D2 = T_im . [F_re | F_im]^T  (columns 2 mrows .. 4 mrows)
//   Z_re[c][b] = D1[c][b] - D2[c][mrows + b]                         Z_im[c][b] = D1[c][mrows + b] + D2[c][b]
// A tcgen05.mma of M = 128 costs max(M, 128) N / 256 cycles whatever its rows hold, so the block rows belong on the N side
// when a pass has few of them: C3 (D = 5120: 29 blocks per 2^25-sample step) issues M128 x N64 instead of M128 x N128 with
// 29 of 128 rows used, for twice the slots — a quarter of the tensor-pipe time per slot — and reads every spectra tile once per
// 128 slots instead of once per 64.  TMEM lane = channel slot: an epilogue warp stores 32 adjacent slots of one block per
// instruction (256-byte rows of Z[q][b][slots]).  Row tiles hold up to 128 blocks (N up to 256, all 512 TMEM columns), so the
// table — what such a pass is bound by — is streamed once per 128 blocks (row tiles of one table tile start whenever an SM
// frees up: measured at C3, three 64-block tiles re-read most of the table from DRAM, not from L2).
// ------------------------------------------------------------------------------------------------
constexpr int TT_SLOTS = 128;                               // channel slots per CTA (the MMA's M)
// Ring stages of 16 branches (TC_KC): what a table-bound pass needs is bytes in flight, and an SM streams (stages x stage bytes)
// per (load latency + MMA time of a stage).  With 128-slot table tiles a 32-branch stage would be 48 KB + 6 x 64 B per block row —
// only two fit beside 96 block rows, and the ring then delivers 2 stages per (2.0 + 1.2) us: 52 GB/s per SM, below the SM's share
// of DRAM.  16-branch stages halve the granule: five of 42 KB fit, 5 per (2.0 + 0.6) us.
__global__ void __launch_bounds__(192, 1)
fc_contract_tct_kernel(const __grid_constant__ CUtensorMap mapF, const __grid_constant__ CUtensorMap mapT, float2* __restrict__ Z, int B, int Dp,
                       int slots, int nbt, int mrows, int nsplit, int M, int nst, unsigned tmem_cols, int levels)
{
    extern __shared__ unsigned char tc_smem_raw[];
    __shared__ unsigned long long bars[2 * TT_MAXST + 1];            // full[nst], empty[nst], accumulators ready
    __shared__ unsigned tmem_slot;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    // slot groups fastest: the CTAs that share a spectra tile run side by side (one DRAM read, L2 hits for the others); row
    // tiles next, so that a table tile needed by several row tiles is still in L2
    const int ngroups = (slots + TT_SLOTS - 1) / TT_SLOTS;
    const int cg = blockIdx.x % ngroups;
    const int q = (blockIdx.x / ngroups) / nbt, bt = (blockIdx.x / ngroups) % nbt;
    const int b0 = bt * mrows;
    const int rows = min(mrows, B - b0);
    const int all_chunks = Dp / TC_KC;
    const int ch0 = (int)(((long long)all_chunks * blockIdx.z) / nsplit);
    const int nchunks = (int)(((long long)all_chunks * (blockIdx.z + 1)) / nsplit) - ch0;
    Z += (size_t)blockIdx.z * M * B * slots;

    const unsigned npl = 2u * (unsigned)levels;                      // operand planes: levels x (re, im)
    const unsigned t_plane = TT_SLOTS * TC_ROWB, t_stage = npl * t_plane;
    const unsigned f_plane = (unsigned)mrows * TC_ROWB;              // mrows is a multiple of 8: every plane starts on a swizzle atom
    const unsigned stage_bytes = t_stage + npl * f_plane;
    const unsigned smem0 = ((unsigned)__cvta_generic_to_shared(tc_smem_raw) + 1023u) & ~1023u;
    const unsigned bar0 = (unsigned)__cvta_generic_to_shared(bars);
    const unsigned bar_acc = bar0 + 8 * (2 * TT_MAXST);
    const unsigned ncols = 2u * (unsigned)mrows;                     // N of one MMA = width of D1 (and of D2)

    if (tid == 0) {
        for (int s = 0; s < nst; s++) {
            mbar_init(bar0 + 8 * s, 1);
            mbar_init(bar0 + 8 * (TT_MAXST + s), 1);
        }
        mbar_init(bar_acc, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (wid == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(&tmem_slot)),
                     "r"(tmem_cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const unsigned tmem = tmem_slot;

    if (wid == 0) {
        if (lane == 0) {
            int stage = 0;
            unsigned phase = 0;
            for (int ch = 0; ch < nchunks; ch++) {
                const unsigned full = bar0 + 8 * stage, empty = bar0 + 8 * (TT_MAXST + stage);
                mbar_wait(empty, phase ^ 1);
                mbar_expect_tx(full, stage_bytes);
                const unsigned sa = smem0 + stage * stage_bytes;
                // slot rows past the group's last slot / block rows past the tile's last block come from the next bin (or are
                // zero-filled past the tensor): they only feed accumulator lanes / columns that are never stored
                tma_load_3d(sa, &mapT, (ch0 + ch) * TC_KC, q * slots + cg * TT_SLOTS, 0, full);
                tma_load_3d(sa + t_stage, &mapF, (ch0 + ch) * TC_KC, q * B + b0, 0, full);
                if (++stage == nst) { stage = 0; phase ^= 1; }
            }
        }
        __syncwarp();
    } else if (wid == 1) {
        if (lane == 0) {
            const unsigned idesc = tc_idesc(levels, ncols);          // N = 2 mrows, M = 128
            const int nprod = levels == 3 ? 6 : 3;
            int stage = 0;
            unsigned phase = 0;
            for (int ch = 0; ch < nchunks; ch++) {
                mbar_wait(bar0 + 8 * stage, phase);
                asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                const unsigned sa = smem0 + stage * stage_bytes, sf = sa + t_stage;
                for (int p = 0; p < nprod; p++) {
                    const int lt = levels == 3 ? kTcProd3[p][0] : kTcProd2[p][0], lf = levels == 3 ? kTcProd3[p][1] : kTcProd2[p][1];
                    const unsigned long long d_re = smem_desc_rows(sa + (unsigned)(2 * lt) * t_plane);
                    const unsigned long long d_im = smem_desc_rows(sa + (unsigned)(2 * lt + 1) * t_plane);
                    const unsigned long long d_f = smem_desc_rows(sf + (unsigned)(2 * lf) * f_plane);   // [F_re ; F_im] of level lf
                    const unsigned acc = (ch | p) != 0;
                    umma_desc(tmem, d_re, d_f, idesc, acc);           // D1 += T_re . [F_re | F_im]^T
                    umma_desc(tmem + ncols, d_im, d_f, idesc, acc);   // D2 += T_im . [F_re | F_im]^T
                }
                umma_commit(bar0 + 8 * (TT_MAXST + stage));
                if (++stage == nst) { stage = 0; phase ^= 1; }
            }
            umma_commit(bar_acc);
        }
        __syncwarp();
    } else {
        // epilogue: warp w may touch TMEM lanes 32 (w % 4) .. +31; thread <-> channel slot, columns <-> blocks
        const int quarter = wid & 3;
        const int c = cg * TT_SLOTS + quarter * 32 + lane;
        mbar_wait(bar_acc, 0);
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
        const unsigned trow = tmem + ((unsigned)(quarter * 32) << 16);
        float2* zc = Z + ((size_t)q * B + b0) * slots + c;
#pragma unroll 1
        for (int bb = 0; bb < rows; bb += 16) {
            float d1r[16], d1i[16], d2r[16], d2i[16];
            tmem_ld16(trow + bb, d1r);                                 // T_re . F_re
            tmem_ld16(trow + mrows + bb, d1i);                         // T_re . F_im
            tmem_ld16(trow + ncols + bb, d2r);                         // T_im . F_re
            tmem_ld16(trow + ncols + mrows + bb, d2i);                 // T_im . F_im
            asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
            if (c < slots) {
#pragma unroll
                for (int i = 0; i < 16; i++)
                    if (bb + i < rows) zc[(size_t)(bb + i) * slots] = make_float2(d1r[i] - d2i[i], d1i[i] + d2r[i]);
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (wid == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem), "r"(tmem_cols) : "memory");
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// 16-bit tensor [2 levels planes][rows][cols] (cols contiguous) with a (TC_KC cols x box_rows x 2 levels planes) box, SWIZZLE_32B
int make_plane_map(CUtensorMap* map, const void* base, size_t cols, size_t rows, unsigned box_rows, int levels)
{
    static EncodeTiledFn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qr;
        OWRX_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qr));
        if (!fn || qr != cudaDriverEntryPointSuccess) return fail(OWRX_E_CUDA, "cuTensorMapEncodeTiled is not available");
        encode = reinterpret_cast<EncodeTiledFn>(fn);
    }
    const cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)(2 * levels)};
    const cuuint64_t strides[2] = {(cuuint64_t)cols * 2, (cuuint64_t)cols * rows * 2};
    const cuuint32_t box[3] = {(cuuint32_t)TC_KC, box_rows, (cuuint32_t)(2 * levels)};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = encode(map, levels == 3 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(OWRX_E_CUDA, "cuTensorMapEncodeTiled (operand planes) failed (%d)", (int)r);
    return OWRX_OK;
}

// split-K factor (one CTA per SM): waves of CTAs, each 1/sp of a tile plus a fixed prologue / epilogue worth about three chunks;
// the split that wastes the least of the last wave (192 tiles of 160 chunks on 148 SMs: 3 -> 4 waves of a third instead of 2 whole)
int tc_plan_split(long long tiles, int chunks, int sm_count)
{
    int best = 1;
    double best_cost = 1e30;
    for (int sp = 1; sp <= std::min(FC_MAXSPLIT, chunks); sp++) {
        const double cost = (double)((tiles * sp + sm_count - 1) / sm_count) * (1.0 / sp + 3.0 / chunks);
        if (cost < best_cost * 0.97) { best_cost = cost; best = sp; }
    }
    return best;
}

}  // namespace

size_t fc_tc_plane_elems_F(const FcShape& sh, int B) { return (size_t)sh.M * B * sh.Dp; }
size_t fc_tc_plane_elems_tab(const FcShape& sh) { return (size_t)sh.M * sh.slots * sh.Dp; }

int fc_launch_contract_tc(const FcShape& sh, const void* d_Fp, const void* d_tabp, int B, float2* d_Z, int sm_count, int force_form,
                          int* nsplit_out, cudaStream_t st)
{
    CUtensorMap mapA, mapB;
    int rc;
    // ---- blocks in M: row tiles of <= 128 blocks, balanced, a multiple of 8 rows (the swizzle atom); 64 slots per CTA
    const int nbt = (B + 127) / 128;
    const int mrows = std::min(128, (((B + nbt - 1) / nbt) + 7) / 8 * 8);
    // ---- slots in M: row tiles of <= 128 blocks, balanced, a multiple of 8 (the swizzle atom; N = 2 mrows is then a multiple
    // of 16) and at least 16 (the epilogue reads 16 TMEM columns at a time and must stay inside the allocation); 128 slots per CTA
    const int nbt_t = (B + 127) / 128;
    const int mrows_t = std::max(16, std::min(128, (((B + nbt_t - 1) / nbt_t) + 7) / 8 * 8));
    // tensor-pipe cycles per 32-branch chunk and 64 slots: 24 MMAs of max(M, 128) N / 256 cycles each
    const long long cyc_m = 24ll * 64 * nbt, cyc_t = 24ll * mrows_t * nbt_t / 2;   // (the same factor for either operand split)
    const int lv = sh.tc_levels;
    const unsigned npl = 2u * (unsigned)lv;
    const bool slots_in_m = force_form >= 0 ? (force_form == 1 && sh.slots >= FC_CG) : (sh.slots >= TT_SLOTS && cyc_t < cyc_m);

    if (slots_in_m) {
        const int chunks_t = sh.Dp / TC_KC;
        const int ngroups = (sh.slots + TT_SLOTS - 1) / TT_SLOTS;
        const unsigned stage_bytes = npl * (unsigned)(TT_SLOTS + mrows_t) * TC_ROWB;
        const int stages = std::max(2, std::min(TT_MAXST, (int)(((size_t)(220 << 10)) / stage_bytes)));
        const size_t smem = (size_t)stages * stage_bytes + 1024;
        const long long tiles = (long long)sh.M * nbt_t * ngroups;
        if ((rc = make_plane_map(&mapA, d_Fp, (size_t)sh.Dp, (size_t)sh.M * B, (unsigned)mrows_t, lv)) != OWRX_OK) return rc;
        if ((rc = make_plane_map(&mapB, d_tabp, (size_t)sh.Dp, (size_t)sh.M * sh.slots, (unsigned)TT_SLOTS, lv)) != OWRX_OK) return rc;
        const int nsplit = tc_plan_split(tiles, chunks_t, sm_count);
        *nsplit_out = nsplit;
        // TMEM columns: D1 | D2, each 2 mrows wide; the allocation is a power of two >= 32
        unsigned cols = 32;
        while (cols < 4u * (unsigned)mrows_t) cols *= 2;
        OWRX_CUDA(cudaFuncSetAttribute(fc_contract_tct_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        fc_contract_tct_kernel<<<dim3((unsigned)tiles, 1, (unsigned)nsplit), 192, smem, st>>>(mapA, mapB, d_Z, B, sh.Dp, sh.slots, nbt_t, mrows_t,
                                                                                               nsplit, sh.M, stages, cols, lv);
        OWRX_LAUNCH_CHECK();
        return OWRX_OK;
    }

    const int chunks_m = sh.Dp / TC_KC;
    const unsigned stage_bytes = npl * (unsigned)(mrows + FC_CG) * TC_ROWB;
    // as many stages as leave room for two CTAs per SM (<= 110 KB each), at least three
    const int stages = std::max(3, std::min(TT_MAXST, (int)(((size_t)(108 << 10)) / stage_bytes)));
    const size_t smem = (size_t)stages * stage_bytes + 1024;
    const long long tiles = (long long)sh.M * nbt * (sh.slots / FC_CG);
    if ((rc = make_plane_map(&mapA, d_Fp, (size_t)sh.Dp, (size_t)sh.M * B, (unsigned)mrows, lv)) != OWRX_OK) return rc;
    if ((rc = make_plane_map(&mapB, d_tabp, (size_t)sh.Dp, (size_t)sh.M * sh.slots, (unsigned)FC_CG, lv)) != OWRX_OK) return rc;
    const int per_sm = smem <= (size_t)(113 << 10) ? 2 : 1;
    const int nsplit = tc_plan_split(tiles, chunks_m, sm_count * per_sm);
    *nsplit_out = nsplit;
    OWRX_CUDA(cudaFuncSetAttribute(fc_contract_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    fc_contract_tc_kernel<<<dim3((unsigned)tiles, 1, (unsigned)nsplit), 192, smem, st>>>(mapA, mapB, d_Z, B, sh.Dp, sh.slots, nbt, mrows, nsplit, sh.M,
                                                                                          stages, lv);
    OWRX_LAUNCH_CHECK();
    return OWRX_OK;
}

}  // namespace owrx
