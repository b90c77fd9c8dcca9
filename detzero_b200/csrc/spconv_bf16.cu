// spconv_bf16.cu -- persistent, warp-specialised sparse convolution forward on tcgen05 with bf16 operand PLANES (sm_100a).
//
// Same contract as spconv.cu / spconv_tc.cu (SubMConv3d / SparseConv3d + folded BatchNorm1d + bias + residual + ReLU,
// detection/detzero_det/models/centerpoint_modules/backbone3d.py:64-83,105-121) for the modes DZ_BF16 and DZ_BF16X2.
//
// Feature storage ("planes"): a row holds PLANES x C bf16 values, [plane 0 | plane 1].
//   PLANES = 1 (DZ_BF16)   : x ~ p0                     = RN_bf16(x)                       2 bytes / value
//   PLANES = 2 (DZ_BF16X2) : x ~ p0 + p1, p1 = RN_bf16(x - p0)  (16 significand bits)      4 bytes / value (= fp32 storage)
// Weights are split the same way (w = w0 + w1).  The products are accumulated in fp32 TMEM as
//   PLANES = 1:  p0 * w0
//   PLANES = 2:  p0 * [w0 | w1]  (ONE MMA, N = 2*Cout: the two halves are summed in the epilogue)  +  p1 * w0
// i.e. x*w up to the dropped p1*w1 term and the 2^-18 representation error of each operand: per-layer error ~1e-6..1e-5
// relative to fp32 FMA (tests: <= 2e-5 per layer, <= 2e-4 through a whole backbone) at the MMA and gather cost of ONE
// TF32 pass (kind::f16 has K = 16 per instruction, a 128-byte smem row holds 64 channels).
//
// Kernel structure (one CTA per SM, persistent over the tile list; roles by warp):
//   warps 0-3      epilogue: tcgen05.ld of accumulator buffer t&1 -> scale/shift (+residual) -> ReLU -> plane split -> stores
//   warps 4-11     producers (all of them fill one pipeline stage at a time): cp.async zero-fill gather of the neighbour rows of a 64-element block of
//                  the (offset, channel) reduction dimension into K-major SW128 smem; one lane TMA-loads the weight tile
//   MMA warp       one thread issues tcgen05.mma kind::f16 (M128 x N x K16) into TMEM accumulator buffer t&1
//   fence warp     one thread turns "the cp.async data of stage s has landed" (async mbarrier arrival of the producers) into "stage s
//                  is visible to the tensor core": fence.proxy.async, then arrives on the barrier the MMA thread waits on.  The
//                  fence costs ~200 clk per step: in the MMA thread it was on the critical path, in the producers it would block
//                  them for the landing latency (both measured, profiles/r02_spconv_notes.md)
//   tile warp      walks the CTA's tiles (heaviest-first tile order of the rulebook schedule, serpentine over the CTAs), loads
//                  the 128 x 27 neighbour rows of tile t+1/t+2 into the double-buffered table while tile t is computed
// so a tile's prologue (table load) and epilogue hide under the neighbouring tiles' main loops, the smem ring never drains
// between tiles, and the TMEM accumulator is double-buffered.  No atomics: deterministic; a row's accumulation order over
// the reduction blocks never depends on the schedule, so results are bit-identical with or without it.
#include <stdlib.h>
#include <cuda_bf16.h>
#include "common.cuh"
#include "tc.cuh"

extern long long* g_dbgbuf;          // spconv_tc.cu: clock-trace buffer (dz_debug_trace), NULL in normal runs
extern bool g_trace_on;

namespace {

constexpr int SB_ROWS = 128;
constexpr int SB_A_BYTES = SB_ROWS * 128;          // one 64-element bf16 block for 128 rows
constexpr int SB_KMAX = 27;
constexpr int SB_NPLANES = SB_KMAX + 1;             // a tile block: plane k < K = neighbour rows, plane K = the tile's output rows

template <int COUT, int PLANES>
struct SbCfg {
    static constexpr int WROWS = PLANES * COUT;                     // rows of the weight tile: [w0 ; w1]
    static constexpr int W_BYTES = WROWS * 128;
    static constexpr int STAGE_BYTES = PLANES * SB_A_BYTES + W_BYTES;
    static constexpr int NBR_BYTES = 2 * SB_NPLANES * SB_ROWS * 4;   // double-buffered tile block: K neighbour planes + the row plane
    static constexpr int MISC_BYTES = 2 * 64 * 4 + 2 * COUT * 4 + 512;                     // block lists | scale,shift | barriers
    static constexpr int STAGES_FIT = (232448 - NBR_BYTES - MISC_BYTES - 1024) / STAGE_BYTES;
    static constexpr int STAGES = STAGES_FIT > 8 ? 8 : STAGES_FIT;   // as deep as shared memory allows: 3 .. 8
    // ALL producer warps fill ONE stage at a time (16 rows each): a stage is complete after 1/NPROD of the LSU time a
    // warp-per-stage split needs, so the oldest stage lands early and the ring covers the MMA -> commit -> refill latency
    static constexpr int NPROD = 8;
    static constexpr int WARP_MMA = 4 + NPROD;
    static constexpr int WARP_TILE = WARP_MMA + 1;
    static constexpr int WARP_FENCE = WARP_TILE + 1;
    static constexpr int THREADS = 32 * (WARP_FENCE + 1);
    static constexpr int ACC_COLS = WROWS < 32 ? 32 : WROWS;         // TMEM columns of one accumulator buffer
    static constexpr int TMEM_COLS = 2 * ACC_COLS;                   // 64 .. 512 (power of two)
    static constexpr int SMEM = STAGES * STAGE_BYTES + NBR_BYTES + MISC_BYTES + 1024;
};

__device__ __forceinline__ void cp_async16_zfill(uint32_t dst, const void* src, bool valid) {
    const int sz = valid ? 16 : 0;
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint64_t* bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(tc::smem_u32(bar)) : "memory");
}
// bounded wait: a protocol bug turns into a trap (CUDA error) instead of a hung GPU
__device__ __forceinline__ void mbar_wait_bounded(uint64_t* bar, uint32_t parity) {
    uint32_t spins = 0;
    while (!tc::mbar_try_wait(bar, parity)) {
        if (++spins > (1u << 24)) { printf("spconv_bf16: mbarrier timeout (block %d thread %d)\n", (int)blockIdx.x, (int)threadIdx.x); __trap(); }
    }
}
// 32 lanes x 32 columns, no wait (the caller waits once for several loads)
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}
// bulk copy global -> shared, completion counted in bytes on an mbarrier
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(tc::smem_u32(smem_dst)), "l"(src), "r"(bytes), "r"(tc::smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float bf16_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }

template <int CIN_PAD, int COUT, int PLANES>
__global__ void __launch_bounds__(SbCfg<COUT, PLANES>::THREADS, 1)
k_spconv_bf16(const __grid_constant__ CUtensorMap tmW, const uint16_t* __restrict__ in, const int32_t* __restrict__ tab, int K, int tab_rows,
              const int32_t* __restrict__ order, const int* __restrict__ d_n_out, int out_cap, const float* __restrict__ scale,
              const float* __restrict__ shift, const uint16_t* __restrict__ residual, int relu, uint16_t* __restrict__ out,
              const int32_t* __restrict__ tab_tiles, long long* __restrict__ dbg) {
    using Cfg = SbCfg<COUT, PLANES>;
    constexpr int S = Cfg::STAGES;
    const int n = min(*d_n_out, out_cap);
    const int tiles_cap = (tab_rows + SB_ROWS - 1) / SB_ROWS;            // tile_order has one entry per capacity tile
    const int tiles_n = (n + SB_ROWS - 1) / SB_ROWS;
    if ((int)blockIdx.x >= tiles_n) return;                              // more CTAs than tiles: nothing to do (uniform per CTA)

    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    int* s_nbr = reinterpret_cast<int*>(smem + S * Cfg::STAGE_BYTES);            // [2][28][128]: planes k < K neighbour rows, plane K = output rows (-1: none)
    int* s_blk = s_nbr + 2 * SB_NPLANES * SB_ROWS;                                // [2][64]  live reduction blocks; [63] = count, [62] = tile (-1: end)
    float* s_scale = reinterpret_cast<float*>(s_blk + 2 * 64);
    float* s_shift = s_scale + COUT;
    uint64_t* full = reinterpret_cast<uint64_t*>(s_shift + COUT);
    uint64_t* empty = full + S;
    uint64_t* landed = empty + S;                  // producers' cp.async data + weight TMA of a stage have landed (generic proxy)
    uint64_t* nbr_full = landed + S;
    uint64_t* nbr_empty = nbr_full + 2;
    uint64_t* acc_full = nbr_empty + 2;
    uint64_t* acc_empty = acc_full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool tr = dbg && blockIdx.x == 0;                            // clock trace of CTA 0 (tools/trace_spconv_bf16.py)
    long long tr_a = 0, tr_b = 0, tr_c = 0, tr_n = 0;                  // per-role wait / work accumulators
    const long long tr_t0 = tr ? clock64() : 0;
#define TR_WAIT(acc, stmt) do { if (tr) { const long long c0__ = clock64(); stmt; acc += clock64() - c0__; } else { stmt; } } while (0)
    const int ktot = K * CIN_PAD;
    const int nb_tot = (ktot + 63) / 64;

    if (threadIdx.x == 0) {
        tc::prefetch_tmap(&tmW);
        for (int s = 0; s < S; ++s) { tc::mbar_init(landed + s, 32 * Cfg::NPROD + 1); tc::mbar_init(full + s, 1); tc::mbar_init(empty + s, 1); }
        for (int b = 0; b < 2; ++b) {
            tc::mbar_init(nbr_full + b, 1);
            tc::mbar_init(nbr_empty + b, Cfg::NPROD + 2 + 4);
            tc::mbar_init(acc_full + b, 1);
            tc::mbar_init(acc_empty + b, 4);
        }
        tc::fence_barrier_init();
    }
    for (int c = threadIdx.x; c < COUT; c += blockDim.x) {
        s_scale[c] = scale ? __ldg(scale + c) : 1.f;
        s_shift[c] = shift ? __ldg(shift + c) : 0.f;
    }
    if (warp == Cfg::WARP_MMA) tc::tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
    tc::tcgen05_fence_before();
    __syncthreads();
    tc::tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == Cfg::WARP_TILE) {
        // ================= tile warp: neighbour rows + live block list of the CTA's next tile ===================================
        const int G = gridDim.x;
        int t = 0;
        for (int round = 0;; ++round) {
            const int q = round * G + ((round & 1) ? (G - 1 - (int)blockIdx.x) : (int)blockIdx.x);    // serpentine over the CTAs
            const bool end = round * G >= tiles_cap;
            int tile = -1;
            if (!end) {
                if (q >= tiles_cap) continue;
                tile = order ? __ldg(order + tab_rows + q) : q;
                if (tile * SB_ROWS >= n) continue;                       // capacity tile beyond the live rows
            }
            const int b = t & 1;
            if (t >= 2) TR_WAIT(tr_a, mbar_wait_bounded(nbr_empty + b, (((t >> 1) - 1) & 1)));
            int* nb_b = s_nbr + b * SB_NPLANES * SB_ROWS;
            if (end) {
                if (lane == 0) s_blk[b * 64 + 62] = -1;
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(nbr_full + b);
                if (tr && lane == 0) { dbg[2048 + 0] = tr_a; dbg[2048 + 1] = t; dbg[2048 + 2] = clock64() - tr_t0; }
                break;
            }
            unsigned mask = 0;
            if (tab_tiles) {
                mask = (unsigned)__ldg(order + tab_rows + tiles_cap + tile);       // precomputed OR of the tile's row masks
            } else {
#pragma unroll 1
            for (int i = 0; i < 4; ++i) {
                const int r = lane + 32 * i;
                const int pos = tile * SB_ROWS + r;
                const int src = pos < n ? (order ? __ldg(order + pos) : pos) : -1;
                int w[28];
                const int4* rowp = reinterpret_cast<const int4*>(tab) + (size_t)(src < 0 ? 0 : src) * 8;
#pragma unroll
                for (int qq = 0; qq < 7; ++qq) {
                    const int4 t4 = src >= 0 ? __ldg(rowp + qq) : make_int4(-1, -1, -1, 0);
                    w[4 * qq] = t4.x; w[4 * qq + 1] = t4.y; w[4 * qq + 2] = t4.z; w[4 * qq + 3] = t4.w;
                }
                if (src < 0) w[27] = 0;
#pragma unroll
                for (int k = 0; k < SB_KMAX; ++k)
                    if (k < K) nb_b[k * SB_ROWS + r] = w[k];
                mask |= (unsigned)w[27];
                nb_b[K * SB_ROWS + r] = src;
            }
            }
            mask = __reduce_or_sync(0xffffffffu, mask);
            // live blocks: block kb covers offsets [kb*64/CIN_PAD, (kb*64+63)/CIN_PAD]
            int cnt = 0;
            for (int kb0 = 0; kb0 < nb_tot; kb0 += 32) {
                const int kb = kb0 + lane;
                bool live = false;
                if (kb < nb_tot) {
                    const int k_lo = (kb * 64) / CIN_PAD, k_hi = min(K - 1, (kb * 64 + 63) / CIN_PAD);
                    for (int k = k_lo; k <= k_hi; ++k) live |= (mask >> k) & 1u;
                }
                const unsigned bal = __ballot_sync(0xffffffffu, live);
                if (live) s_blk[b * 64 + cnt + __popc(bal & ((1u << lane) - 1u))] = kb;
                cnt += __popc(bal);
            }
            if (lane == 0) { s_blk[b * 64 + 63] = cnt; s_blk[b * 64 + 62] = tile; }
            __syncwarp();
            if (lane == 0) {
                if (tab_tiles) {                                         // the tile's (K+1) x 128 block: ONE bulk copy, completes the phase
                    const uint32_t bytes = (uint32_t)(K + 1) * SB_ROWS * 4;
                    tc::mbar_arrive_expect_tx(nbr_full + b, bytes);
                    bulk_g2s(nb_b, tab_tiles + (size_t)tile * (K + 1) * SB_ROWS, bytes, nbr_full + b);
                } else {
                    tc::mbar_arrive(nbr_full + b);                       // release: smem writes of the warp are ordered before the arrive
                }
            }
            ++t;
        }
    } else if (warp >= 4 && warp < 4 + Cfg::NPROD) {
        // ================= producers ============================================================================================
        const int pw = warp - 4;
        constexpr int RPW = SB_ROWS / Cfg::NPROD;    // rows per producer warp (16)
        constexpr int RPL = RPW / 4;                 // rows per lane (8 lanes cover the 8 chunks of a row): 4 = one int4 of the table
        const int j = lane & 7, rg = lane >> 3;
        const int rbase = pw * RPW + rg * RPL;
        const uint32_t smem_u = tc::smem_u32(smem);
        int g = 0;                                   // CTA-wide step counter (same sequence in every role)
        for (int t = 0;; ++t) {
            const int b = t & 1;
            TR_WAIT(tr_a, mbar_wait_bounded(nbr_full + b, (t >> 1) & 1));
            if (s_blk[b * 64 + 62] < 0) {
                if (tr && pw == 0 && lane == 0) { dbg[2048 + 8] = tr_a; dbg[2048 + 9] = tr_b; dbg[2048 + 10] = tr_c; dbg[2048 + 11] = tr_n; }
                break;
            }
            const int nb = s_blk[b * 64 + 63];
            const int* nb_b = s_nbr + b * SB_NPLANES * SB_ROWS;
            for (int i = 0; i < nb; ++i) {
                const int gi = g + i;
                const int my_s = gi % S;
                const int kb = s_blk[b * 64 + i];
                TR_WAIT(tr_b, mbar_wait_bounded(empty + my_s, ((gi / S) & 1) ^ 1));
                const long long tr_i0 = tr ? clock64() : 0;
                const uint32_t sa_u = smem_u + (uint32_t)(my_s * Cfg::STAGE_BYTES);
                if (pw == 0 && lane == 0) {
                    tc::mbar_arrive_expect_tx(landed + my_s, Cfg::W_BYTES);
                    tc::tma_load_2d(smem + my_s * Cfg::STAGE_BYTES + PLANES * SB_A_BYTES, &tmW, landed + my_s, kb * 64, 0);
                }
                const int e = kb * 64 + j * 8;                       // position of this lane's chunk in the (offset, channel) dimension
                const int k = e / CIN_PAD, c = e % CIN_PAD;
                const bool k_ok = k < K;
                const int4* nb_k = reinterpret_cast<const int4*>(nb_b + (k_ok ? k : 0) * SB_ROWS + rbase);
                const uint16_t* in_c = in + c;
#pragma unroll
                for (int i0 = 0; i0 < RPL; i0 += 4) {
                    const int4 nq = nb_k[i0 / 4];
                    const int rows4[4] = {nq.x, nq.y, nq.z, nq.w};
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const int src_row = k_ok ? rows4[u] : -1;
                        const bool ok = src_row >= 0;
                        const int r = rbase + i0 + u;
                        const int rr = r & 7;
                        const uint32_t dst = sa_u + (uint32_t)((r >> 3) * 1024 + rr * 128 + ((j ^ rr) << 4));
                        const uint16_t* src = ok ? in_c + (size_t)src_row * (PLANES * CIN_PAD) : in;
#pragma unroll
                        for (int p = 0; p < PLANES; ++p)
                            cp_async16_zfill(dst + p * SB_A_BYTES, src + (ok ? p * CIN_PAD : 0), ok);
                    }
                }
                cp_async_mbar_arrive_noinc(landed + my_s);           // asynchronous: arrives when this thread's copies have landed
                if (tr) { tr_c += clock64() - tr_i0; ++tr_n; }
            }
            g += nb;
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(nbr_empty + b);
        }
    } else if (warp == Cfg::WARP_FENCE) {
        // ================= fence warp: landed[s] -> fence.proxy.async -> full[s] ===============================================
        if (lane == 0) {
            int g = 0;
            for (int t = 0;; ++t) {
                const int b = t & 1;
                mbar_wait_bounded(nbr_full + b, (t >> 1) & 1);
                if (s_blk[b * 64 + 62] < 0) break;
                const int nb = s_blk[b * 64 + 63];
                tc::mbar_arrive(nbr_empty + b);
                for (int i = 0; i < nb; ++i, ++g) {
                    const int s = g % S;
                    mbar_wait_bounded(landed + s, (g / S) & 1);
                    tc::fence_proxy_async();            // cp.async (generic proxy) writes -> tensor-core (async proxy) reads
                    tc::mbar_arrive(full + s);
                }
            }
        }
    } else if (warp == Cfg::WARP_MMA) {
        // ================= MMA issuer ==========================================================================================
        if (lane == 0) {
            constexpr uint32_t idesc0 = tc::instr_desc(1, 128, Cfg::WROWS);        // bf16 x bf16 -> fp32, N = PLANES * COUT
            constexpr uint32_t idesc1 = tc::instr_desc(1, 128, COUT);
            const uint32_t smem_u = tc::smem_u32(smem);
            int g = 0;
            for (int t = 0;; ++t) {
                const int b = t & 1;
                TR_WAIT(tr_a, mbar_wait_bounded(nbr_full + b, (t >> 1) & 1));
                if (s_blk[b * 64 + 62] < 0) {
                    if (tr) { dbg[2048 + 16] = tr_a; dbg[2048 + 17] = tr_b; dbg[2048 + 18] = tr_c; dbg[2048 + 19] = tr_n; dbg[2048 + 20] = clock64() - tr_t0; }
                    break;
                }
                const int nb = s_blk[b * 64 + 63];
                tc::mbar_arrive(nbr_empty + b);                         // only `nb` was needed
                TR_WAIT(tr_a, mbar_wait_bounded(acc_empty + b, ((t >> 1) & 1) ^ 1));   // epilogue of tile t-2 has drained this accumulator
                tc::tcgen05_fence_after();
                const uint32_t acc = tmem_base + (uint32_t)(b * Cfg::ACC_COLS);
                for (int i = 0; i < nb; ++i, ++g) {
                    const int s = g % S;
                    TR_WAIT(tr_b, mbar_wait_bounded(full + s, (g / S) & 1));
                    const long long tr_i0 = tr ? clock64() : 0;
                    tc::tcgen05_fence_after();          // (the generic->async proxy fence is executed by the producers before they arrive)
                    const uint32_t sa = smem_u + (uint32_t)(s * Cfg::STAGE_BYTES);
                    const uint64_t a0 = tc::smem_desc_sw128(sa), wd = tc::smem_desc_sw128(sa + PLANES * SB_A_BYTES);
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
                        tc::mma_f16(acc, a0 + (uint64_t)(kk * 2), wd + (uint64_t)(kk * 2), idesc0, (i | kk) ? 1u : 0u);
                    if (PLANES == 2) {
                        const uint64_t a1 = tc::smem_desc_sw128(sa + SB_A_BYTES);
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk)
                            tc::mma_f16(acc, a1 + (uint64_t)(kk * 2), wd + (uint64_t)(kk * 2), idesc1, 1u);
                    }
                    tc::mma_commit(empty + s);
                    if (tr) { tr_c += clock64() - tr_i0; ++tr_n; }
                }
                tc::mma_commit(acc_full + b);
            }
        }
    } else {
        // ================= epilogue (warps 0-3 <-> TMEM lane quarters) ========================================================
        const int q = warp;
        const int trow = q * 32 + lane;
        constexpr int CW = COUT < 32 ? COUT : 32;         // channels per pass
        for (int t = 0;; ++t) {
            const int b = t & 1;
            TR_WAIT(tr_a, mbar_wait_bounded(nbr_full + b, (t >> 1) & 1));
            if (s_blk[b * 64 + 62] < 0) {
                if (tr && threadIdx.x == 0) { dbg[2048 + 24] = tr_a; dbg[2048 + 25] = tr_b; dbg[2048 + 26] = tr_c; dbg[2048 + 27] = t; }
                break;
            }
            const int nb = s_blk[b * 64 + 63];
            const int r = s_nbr[b * SB_NPLANES * SB_ROWS + K * SB_ROWS + trow];
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(nbr_empty + b);
            TR_WAIT(tr_b, mbar_wait_bounded(acc_full + b, (t >> 1) & 1));
            const long long tr_e0 = tr ? clock64() : 0;
            tc::tcgen05_fence_after();
            const uint32_t acc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(b * Cfg::ACC_COLS);
#pragma unroll 1
            for (int c0 = 0; c0 < COUT; c0 += CW) {
                uint32_t v0[32], v1[32];
                tmem_ld32_nowait(acc + (uint32_t)c0, v0);
                if (PLANES == 2 && COUT >= 32) tmem_ld32_nowait(acc + (uint32_t)(COUT + c0), v1);
                tmem_ld_wait();
                if (c0 + CW >= COUT) {                    // last TMEM read of this tile: hand the accumulator back to the MMA warp
                    tc::tcgen05_fence_before();
                    __syncwarp();
                    if (lane == 0) tc::mbar_arrive(acc_empty + b);
                }
                if (r >= 0) {
                    float o[CW];
#pragma unroll
                    for (int jj = 0; jj < CW; ++jj) {
                        float a = __uint_as_float(v0[jj]);
                        if (PLANES == 2) a += (COUT >= 32) ? __uint_as_float(v1[jj]) : __uint_as_float(v0[COUT + jj]);
                        if (nb == 0) a = 0.f;
                        o[jj] = fmaf(a, s_scale[c0 + jj], s_shift[c0 + jj]);
                    }
                    if (residual) {
                        const uint4* rp = reinterpret_cast<const uint4*>(residual + (size_t)r * (PLANES * COUT) + c0);
#pragma unroll
                        for (int p = 0; p < PLANES; ++p)
#pragma unroll
                            for (int v = 0; v < CW / 8; ++v) {
                                const uint4 u = __ldg(rp + p * (COUT / 8) + v);
                                o[8 * v + 0] += bf16_lo(u.x); o[8 * v + 1] += bf16_hi(u.x); o[8 * v + 2] += bf16_lo(u.y); o[8 * v + 3] += bf16_hi(u.y);
                                o[8 * v + 4] += bf16_lo(u.z); o[8 * v + 5] += bf16_hi(u.z); o[8 * v + 6] += bf16_lo(u.w); o[8 * v + 7] += bf16_hi(u.w);
                            }
                    }
                    if (relu) {
#pragma unroll
                        for (int jj = 0; jj < CW; ++jj) o[jj] = fmaxf(o[jj], 0.f);
                    }
                    uint4* op = reinterpret_cast<uint4*>(out + (size_t)r * (PLANES * COUT) + c0);
#pragma unroll
                    for (int v = 0; v < CW / 8; ++v) {
                        uint4 h;
                        h.x = pack_bf16(o[8 * v + 0], o[8 * v + 1]); h.y = pack_bf16(o[8 * v + 2], o[8 * v + 3]);
                        h.z = pack_bf16(o[8 * v + 4], o[8 * v + 5]); h.w = pack_bf16(o[8 * v + 6], o[8 * v + 7]);
                        op[v] = h;
                        if (PLANES == 2) {
                            uint4 l;
                            l.x = pack_bf16(o[8 * v + 0] - bf16_lo(h.x), o[8 * v + 1] - bf16_hi(h.x));
                            l.y = pack_bf16(o[8 * v + 2] - bf16_lo(h.y), o[8 * v + 3] - bf16_hi(h.y));
                            l.z = pack_bf16(o[8 * v + 4] - bf16_lo(h.z), o[8 * v + 5] - bf16_hi(h.z));
                            l.w = pack_bf16(o[8 * v + 6] - bf16_lo(h.w), o[8 * v + 7] - bf16_hi(h.w));
                            op[COUT / 8 + v] = l;
                        }
                    }
                }
            }
            if (tr) tr_c += clock64() - tr_e0;
        }
    }
#undef TR_WAIT
    tc::tcgen05_fence_before();
    __syncthreads();
    if (warp == Cfg::WARP_MMA) tc::tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
}

// ---- tensor-map cache: the weight matrix of a layer never moves, encode its map once ---------------------------------------
struct TmKey { const void* p; int rows, ktot; };
struct TmEnt { TmKey k; CUtensorMap m; };
static TmEnt g_tm[128];
static int g_tm_n = 0;

static const CUtensorMap* weight_map(const void* w, int rows, int ktot) {
    for (int i = 0; i < g_tm_n; ++i)
        if (g_tm[i].k.p == w && g_tm[i].k.rows == rows && g_tm[i].k.ktot == ktot) return &g_tm[i].m;
    tc::EncodeTiledFn enc = tc::get_encode_tiled();
    if (!enc) { dz_set_error("cuTensorMapEncodeTiled unavailable"); return nullptr; }
    static CUtensorMap scratch;
    CUtensorMap* m = g_tm_n < 128 ? &g_tm[g_tm_n].m : &scratch;
    cuuint64_t dims[2] = {(cuuint64_t)ktot, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ktot * 2};
    cuuint32_t box[2] = {64, (cuuint32_t)rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(w), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { dz_set_error("cuTensorMapEncodeTiled(W bf16) failed: %d", (int)r); return nullptr; }
    if (g_tm_n < 128) { g_tm[g_tm_n].k = TmKey{w, rows, ktot}; ++g_tm_n; }
    return m;
}

static int g_ctas = -1;

template <int CIN_PAD, int COUT, int PLANES>
int launch(const void* in, const int32_t* tab, int K, int tab_rows, const int32_t* order, const int* d_n_out, int out_cap, const void* weight,
           const float* scale, const float* shift, const void* residual, int relu, void* out, const int32_t* tab_tiles, cudaStream_t st) {
    using Cfg = SbCfg<COUT, PLANES>;
    static_assert(Cfg::SMEM <= 232448, "shared memory budget");
    static bool configured = false;
    if (!configured) {
        DZ_CUDA(cudaFuncSetAttribute(k_spconv_bf16<CIN_PAD, COUT, PLANES>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM));
        configured = true;
    }
    if (g_ctas < 0) { const char* e = getenv("DZ_SPCONV_CTAS"); g_ctas = e ? atoi(e) : DZ_NUM_SMS; if (g_ctas < 1) g_ctas = DZ_NUM_SMS; }
    const CUtensorMap* tm = weight_map(weight, Cfg::WROWS, K * CIN_PAD);
    if (!tm) return DZ_ERR_CUDA;
    const int grid = min(g_ctas, dz_cdiv(out_cap, SB_ROWS));
    k_spconv_bf16<CIN_PAD, COUT, PLANES><<<grid, Cfg::THREADS, Cfg::SMEM, st>>>(
        *tm, (const uint16_t*)in, tab, K, tab_rows, order, d_n_out, out_cap, scale, shift, (const uint16_t*)residual, relu, (uint16_t*)out,
        order ? tab_tiles : nullptr, g_trace_on ? g_dbgbuf : nullptr);
    DZ_LAUNCH_CHECK();
    return DZ_OK;
}

// ---- fp32 (rows, c) <-> bf16 planes (rows, planes * c_pad) --------------------------------------------------------------
__global__ void __launch_bounds__(256) k_to_planes(const float* __restrict__ x, const int* __restrict__ d_n, int cap, int c, int c_pad, int planes,
                                                   uint16_t* __restrict__ out) {
    const int n = d_n ? min(*d_n, cap) : cap;
    const long long total = (long long)n * c_pad;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(i / c_pad), ch = (int)(i % c_pad);
        const float v = ch < c ? __ldg(x + (size_t)r * c + ch) : 0.f;
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        uint16_t* o = out + (size_t)r * planes * c_pad + ch;
        o[0] = *reinterpret_cast<const uint16_t*>(&h);
        if (planes == 2) {
            const __nv_bfloat16 l = __float2bfloat16_rn(v - __bfloat162float(h));
            o[c_pad] = *reinterpret_cast<const uint16_t*>(&l);
        }
    }
}
__global__ void __launch_bounds__(256) k_from_planes(const uint16_t* __restrict__ x, const int* __restrict__ d_n, int cap, int c, int planes,
                                                     float* __restrict__ out) {
    const int n = d_n ? min(*d_n, cap) : cap;
    const long long total = (long long)n * c;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(i / c), ch = (int)(i % c);
        const uint16_t* p = x + (size_t)r * planes * c + ch;
        float v = __uint_as_float((uint32_t)p[0] << 16);
        if (planes == 2) v += __uint_as_float((uint32_t)p[c] << 16);
        out[i] = v;
    }
}
// HeightCompression on a planes tensor: out[b,y,x,c*D+z] = feats[i,c] (fp32 NHWC, zero on entry)
__global__ void __launch_bounds__(256) k_sparse_to_bev_planes(const uint16_t* __restrict__ feats, const int32_t* __restrict__ coords,
                                                              const int* __restrict__ d_n, int cap, int c, int planes, int D, int H, int W,
                                                              float* __restrict__ out) {
    const int n = min(*d_n, cap);
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int i = warp; i < n; i += nwarps) {
        const int4 cd = __ldg(reinterpret_cast<const int4*>(coords) + i);            // b,z,y,x
        float* dst = out + (((size_t)cd.x * H + cd.z) * W + cd.w) * ((size_t)c * D) + cd.y;
        const uint16_t* src = feats + (size_t)i * planes * c;
        for (int ch = lane; ch < c; ch += 32) {
            float v = __uint_as_float((uint32_t)__ldg(src + ch) << 16);
            if (planes == 2) v += __uint_as_float((uint32_t)__ldg(src + c + ch) << 16);
            dst[(size_t)ch * D] = v;
        }
    }
}

}  // namespace

extern "C" int dz_to_planes(const float* x, const int* d_n, int cap, int c, int c_pad, int planes, void* out, dz_stream_t stream) {
    DZ_CHECK_ARG(x && out && cap >= 1 && c >= 1 && c_pad >= c && (planes == 1 || planes == 2));
    const int blocks = max(1, min(dz_cdiv((long long)cap * c_pad, 256), DZ_NUM_SMS * 8));
    k_to_planes<<<blocks, 256, 0, (cudaStream_t)stream>>>(x, d_n, cap, c, c_pad, planes, (uint16_t*)out);
    DZ_LAUNCH_CHECK();
    return DZ_OK;
}

extern "C" int dz_from_planes(const void* x, const int* d_n, int cap, int c, int planes, float* out, dz_stream_t stream) {
    DZ_CHECK_ARG(x && out && cap >= 1 && c >= 1 && (planes == 1 || planes == 2));
    const int blocks = max(1, min(dz_cdiv((long long)cap * c, 256), DZ_NUM_SMS * 8));
    k_from_planes<<<blocks, 256, 0, (cudaStream_t)stream>>>((const uint16_t*)x, d_n, cap, c, planes, out);
    DZ_LAUNCH_CHECK();
    return DZ_OK;
}

extern "C" int dz_sparse_to_bev_planes(const void* feats, const int32_t* coords, const int* d_n, int cap, int c, int planes, int B, int D,
                                       int H, int W, float* out, dz_stream_t stream) {
    DZ_CHECK_ARG(feats && coords && d_n && out && cap >= 1 && c >= 1 && (planes == 1 || planes == 2));
    (void)B;
    const int blocks = max(1, min(dz_cdiv((long long)cap * 32, 256), DZ_NUM_SMS * 8));
    k_sparse_to_bev_planes<<<blocks, 256, 0, (cudaStream_t)stream>>>((const uint16_t*)feats, coords, d_n, cap, c, planes, D, H, W, out);
    DZ_LAUNCH_CHECK();
    return DZ_OK;
}

extern "C" int dz_spconv_fwd_planes(const void* in, int cin, int in_rows, const int32_t* tab, int K, int tab_rows, const int32_t* row_order,
                                    const int* d_n_out, int out_cap, const void* weight, const float* scale, const float* shift,
                                    const void* residual, int relu, void* out, int cout, int planes, const int32_t* tab_tiles,
                                    dz_stream_t stream) {
    // tab may be NULL when the tile-major table and its schedule are given (the direct rulebook path builds no row-major table);
    // tab_rows is then the rulebook's capacity, which sizes `row_order`
    DZ_CHECK_ARG(in && (tab || (tab_tiles && row_order)) && d_n_out && weight && out && cin >= 1 && K >= 1 && K <= SB_KMAX && out_cap >= 1 &&
                 tab_rows >= out_cap);
    DZ_CHECK_ARG(planes == 1 || planes == 2);
    (void)in_rows;
    cudaStream_t st = (cudaStream_t)stream;
    const int cin_pad = cin <= 8 ? 8 : cin;
#define DZ_SB(CP, CO)                                                                                                                           \
    if (cin_pad == CP && cout == CO) {                                                                                                          \
        if (planes == 1) return launch<CP, CO, 1>(in, tab, K, tab_rows, row_order, d_n_out, out_cap, weight, scale, shift, residual, relu, out, tab_tiles, st); \
        return launch<CP, CO, 2>(in, tab, K, tab_rows, row_order, d_n_out, out_cap, weight, scale, shift, residual, relu, out, tab_tiles, st);   \
    }
    DZ_SB(8, 16) DZ_SB(16, 16) DZ_SB(16, 32) DZ_SB(32, 32) DZ_SB(32, 64) DZ_SB(64, 64) DZ_SB(64, 128) DZ_SB(128, 128)
#undef DZ_SB
    dz_set_error("dz_spconv_fwd_planes: (cin=%d, cout=%d) not instantiated", cin, cout);
    return DZ_ERR_UNSUPPORTED;
}
