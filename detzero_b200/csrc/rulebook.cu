// rulebook.cu -- rulebook (neighbour-table) build for submanifold and strided sparse convolution, sm_100a.
//
// Replaces spconv's generate_subm_conv_inds / generate_conv_inds_stage{1,2} (GPU hash table) used through
// SubMConv3d / SparseConv3d at detection/detzero_det/models/centerpoint_modules/backbone3d.py:68-71,93-100.
//
// Design: coordinates are looked up in the L2-resident grid index (bitmap + popcount prefix) -- two dependent
// loads whose cache lines are shared by x-adjacent probes -- instead of probing a hash table.  The output is the
// output-stationary neighbour table nbr[k][o] (k-major => coalesced writes here and coalesced reads in the conv
// kernel); strided-conv output sites come out of a bitmap rank scan already sorted by (b,z,y,x), so no sort.
#include "common.cuh"

struct ConvGeom {
    int k[3], s[3], p[3];
    int in_dhw[3], out_dhw[3];
};

// ---- table outputs + tile-schedule digest (see the schedule section at the end of this file) -----------------------------
static constexpr int SCHED_BINS = 1 << 12;          // 12-bit digest of the 27-bit neighbour mask
struct TableOut {
    int32_t* nbr;                                   // k-major (K, cap) table: the exact-fp32 kernel, tests     (or NULL)
    int32_t* tab;                                   // row-major (cap, 32) table: the tensor-core kernels         (or NULL)
    uint16_t* keys;                                 // [cap]        schedule digests                              (or NULL)
    int* masks;                                     // [cap]        neighbour bit masks (compact copy for the schedule pass)
    int* hist;                                      // [SCHED_BINS] digest histogram -> exclusive offsets (last block)
    int* ticket;                                    // block-completion counter
    int fb;                                         // frame bits of the schedule key (0 = digest only)
    int B;                                          // frames in the batch
};

// schedule key = (frame group, digest): frame-major order keeps the rows a CTA wave gathers inside ONE frame's feature map
// (L2-resident) instead of spreading every tile over the whole batch; the digest gives up its fb lowest-priority bits
__device__ __forceinline__ uint32_t sched_key(const TableOut& to, uint32_t digest, int frame) {
    if (to.fb == 0) return digest;
    const uint32_t fg = ((uint32_t)frame << to.fb) / (uint32_t)to.B;
    return (fg << (12 - to.fb)) | (digest >> to.fb);
}

// Rows are grouped by DESCENDING digest so that the tiles with many offsets come first (launch order ~ tile order).
__device__ __forceinline__ uint32_t sched_digest(uint32_t m, int K) {
    if (K != 27) return (~m) & (SCHED_BINS - 1);
    auto line = [&](int l) -> uint32_t { return ((m >> (3 * l)) & 7u) ? 1u : 0u; };
    auto bit = [&](int b) -> uint32_t { return (m >> b) & 1u; };
    uint32_t d = line(6);
    d = d << 1 | line(8); d = d << 1 | line(2); d = d << 1 | line(0); d = d << 1 | line(7);
    d = d << 1 | bit(12); d = d << 1 | bit(14); d = d << 1 | bit(9);  d = d << 1 | bit(11);
    d = d << 1 | bit(15); d = d << 1 | bit(17); d = d << 1 | line(1);
    return (~d) & (SCHED_BINS - 1);
}

// one row's schedule digest + mask.  s_hist: the block's digest histogram in shared memory (hot digests are shared by
// thousands of rows: per-row or per-warp global atomics on them serialise in L2)
__device__ __forceinline__ void sched_emit(const TableOut& to, bool valid, int i, uint32_t mask, int K, int* s_hist, int frame) {
    if (to.keys && valid) {
        const uint32_t key = sched_key(to, sched_digest(mask, K), frame);
        to.keys[i] = (uint16_t)key;
        to.masks[i] = (int)mask;
        atomicAdd(s_hist + key, 1);
    }
}

// one table row: v[0..K-1] neighbour rows (or -1)
__device__ __forceinline__ void table_emit(const TableOut& to, bool valid, int i, int cap, const int (&v)[27], int K, int* s_hist, int frame) {
    uint32_t mask = 0;
#pragma unroll
    for (int k = 0; k < 27; ++k) mask |= (k < K && v[k] >= 0 ? 1u : 0u) << k;
    if (valid) {
        if (to.nbr) {
#pragma unroll
            for (int k = 0; k < 27; ++k)
                if (k < K) to.nbr[(size_t)k * cap + i] = v[k];
        }
        if (to.tab) {                                // one 128-byte line per row: {nbr[0..26] (-1 beyond K), mask, 0, 0, 0, 0}
            int4* dst = reinterpret_cast<int4*>(to.tab + (size_t)i * 32);
#pragma unroll
            for (int q = 0; q < 6; ++q)
                dst[q] = make_int4(4 * q < K ? v[4 * q] : -1, 4 * q + 1 < K ? v[4 * q + 1] : -1, 4 * q + 2 < K ? v[4 * q + 2] : -1,
                                   4 * q + 3 < K ? v[4 * q + 3] : -1);
            dst[6] = make_int4(24 < K ? v[24] : -1, 25 < K ? v[25] : -1, 26 < K ? v[26] : -1, (int)mask);
            dst[7] = make_int4(0, 0, 0, 0);
        }
    }
    sched_emit(to, valid, i, mask, K, s_hist, frame);
}

// the last block to finish turns the digest histogram into exclusive offsets (block of 256 threads, 32 bins each)
__device__ __forceinline__ void table_finish(const TableOut& to, int* s_hist) {
    if (!to.keys) return;
    __shared__ int s_last;
    __syncthreads();
    for (int b = threadIdx.x; b < SCHED_BINS; b += blockDim.x) {            // flush this block's histogram
        const int c = s_hist[b];
        if (c) atomicAdd(to.hist + b, c);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(to.ticket, 1) == (int)gridDim.x - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    constexpr int PER = SCHED_BINS / 256;          // blockDim.x == 256
    int v[PER], sum = 0;
    int4* h4 = reinterpret_cast<int4*>(to.hist + threadIdx.x * PER);
#pragma unroll
    for (int j = 0; j < PER / 4; ++j) { int4 q = __ldcg(h4 + j); v[4 * j] = q.x; v[4 * j + 1] = q.y; v[4 * j + 2] = q.z; v[4 * j + 3] = q.w; sum += q.x + q.y + q.z + q.w; }
    int total;
    int run = block_exclusive_scan(sum, &total);
#pragma unroll
    for (int j = 0; j < PER / 4; ++j) {
        int4 q;
        q.x = run; run += v[4 * j]; q.y = run; run += v[4 * j + 1]; q.z = run; run += v[4 * j + 2]; q.w = run; run += v[4 * j + 3];
        h4[j] = q;
    }
}

__global__ void __launch_bounds__(256) k_subm_nbr(const int32_t* __restrict__ coords, const int* __restrict__ d_n, int cap,
                                                  GridIndex g, int KD, int KH, int KW, TableOut to) {
    __shared__ int s_hist[SCHED_BINS];
    if (to.keys) { for (int b = threadIdx.x; b < SCHED_BINS; b += blockDim.x) s_hist[b] = 0; __syncthreads(); }
    int n = min(*d_n, cap);
    int K = KD * KH * KW;
    int hz = (KD - 1) / 2, hy = (KH - 1) / 2, hx = (KW - 1) / 2;
    const int lane = threadIdx.x & 31;
    for (int base = blockIdx.x * blockDim.x + threadIdx.x - lane; base < n; base += gridDim.x * blockDim.x) {     // warp-uniform trip count
        const int i = base + lane;
        int v[27];
        int frame = 0;
#pragma unroll
        for (int k = 0; k < 27; ++k) v[k] = -1;
        if (i < n) {
            int4 c = __ldg(reinterpret_cast<const int4*>(coords) + i);    // b,z,y,x
            frame = c.x;
            int kz = 0, ky = 0, kx = 0;
#pragma unroll
            for (int k = 0; k < 27; ++k) {
                if (k < K) {
                    if (kz == hz && ky == hy && kx == hx) v[k] = i;         // centre tap is the site itself
                    else v[k] = grid_lookup(g, c.x, c.y + kz - hz, c.z + ky - hy, c.w + kx - hx);
                    if (++kx == KW) { kx = 0; if (++ky == KH) { ky = 0; ++kz; } }
                }
            }
        }
        table_emit(to, i < n, i, cap, v, K, s_hist, frame);
    }
    table_finish(to, s_hist);
}

// workspace layout shared by the rulebook kernels (which emit digests + histogram) and dz_rulebook_schedule:
// hist[SCHED_BINS] | tile_mask[tiles] | tickets[8] | masks[cap] | keys[cap] (u16)
static int sched_frame_bits(int B, int frame_major) {
    if (!frame_major || B <= 1) return 0;
    int fb = 1;
    while ((1 << fb) < B && fb < 4) ++fb;
    return fb;
}
static TableOut table_out(int32_t* nbr, int32_t* tab, void* sched_ws, int cap, int B = 1, int frame_major = 0) {
    TableOut to{nbr, tab, nullptr, nullptr, nullptr, nullptr, sched_frame_bits(B, frame_major), B};
    if (sched_ws) {
        to.hist = reinterpret_cast<int*>(sched_ws);
        to.ticket = to.hist + SCHED_BINS + dz_cdiv(cap, 128);
        to.masks = to.ticket + 8;
        to.keys = reinterpret_cast<uint16_t*>(to.masks + cap);
    }
    return to;
}
static size_t sched_zero_bytes(int cap) { return (size_t)(SCHED_BINS + dz_cdiv(cap, 128) + 8) * 4; }
extern "C" size_t dz_rulebook_schedule_ws_bytes(int cap) { return sched_zero_bytes(cap) + (size_t)cap * 4 + (((size_t)cap * 2 + 255) & ~(size_t)255); }

extern "C" int dz_rulebook_subm(const int32_t* coords, const int* d_n, int cap, int B, int D, int H, int W,
                                const int* ks, const uint32_t* bitmap, const uint32_t* prefix, const int32_t* perm,
                                int32_t* nbr, int32_t* tab, void* sched_ws, int sched_frame_major, dz_stream_t stream) {
    DZ_CHECK_ARG(coords && d_n && bitmap && prefix && (nbr || tab) && cap >= 1);
    DZ_CHECK_ARG(ks[0] % 2 == 1 && ks[1] % 2 == 1 && ks[2] % 2 == 1 && ks[0] * ks[1] * ks[2] <= 27);
    DZ_CHECK_ARG(!sched_ws || tab);
    TableOut to = table_out(nbr, tab, sched_ws, cap, B, sched_frame_major);
    if (sched_ws) DZ_CUDA(cudaMemsetAsync(sched_ws, 0, sched_zero_bytes(cap), (cudaStream_t)stream));
    GridIndex g{bitmap, prefix, perm, B, D, H, W, dz_cells_pad(D, H, W)};
    int blocks = max(1, min(dz_cdiv(cap, 256), DZ_NUM_SMS * 8));
    k_subm_nbr<<<blocks, 256, 0, (cudaStream_t)stream>>>(coords, d_n, cap, g, ks[0], ks[1], ks[2], to);
    DZ_LAUNCH_CHECK();
    return DZ_OK;
}

// mark every output cell reachable from an active input: o = (i + p - k) / s when divisible and in range
__global__ void __launch_bounds__(256) k_conv_mark(const int32_t* __restrict__ coords, const int* __restrict__ d_n, int cap,
                                                   ConvGeom cg, long long out_cells_pad, uint32_t* __restrict__ out_bitmap) {
    int n = min(*d_n, cap);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        int4 c = __ldg(reinterpret_cast<const int4*>(coords) + i);
        int iz[3] = {c.y, c.z, c.w};
        // per-dimension candidate outputs (at most ceil(k/s) each)
        int oz[3][3], cnt[3];
        for (int d = 0; d < 3; ++d) {
            cnt[d] = 0;
            for (int k = 0; k < cg.k[d]; ++k) {
                int num = iz[d] + cg.p[d] - k;
                if (num < 0 || num % cg.s[d]) continue;
                int o = num / cg.s[d];
                if (o >= cg.out_dhw[d]) continue;
                oz[d][cnt[d]++] = o;
            }
        }
        for (int a = 0; a < cnt[0]; ++a)
            for (int b = 0; b < cnt[1]; ++b)
                for (int e = 0; e < cnt[2]; ++e) {
                    long long cell = (long long)c.x * out_cells_pad +
                                     ((long long)oz[0][a] * cg.out_dhw[1] + oz[1][b]) * cg.out_dhw[2] + oz[2][e];
                    uint32_t bit = 1u << (cell & 31);
                    uint32_t* wp = out_bitmap + (cell >> 5);
                    if (!(*wp & bit)) atomicOr(wp, bit);        // plain read first: most cells are already set
                }
    }
}

// bitmap words -> sorted coordinate list
__global__ void __launch_bounds__(256) k_index_to_coords(const uint32_t* __restrict__ bitmap, const uint32_t* __restrict__ prefix,
                                                         size_t n_words, int D, int H, int W, long long cells_pad, int cap,
                                                         int32_t* __restrict__ coords) {
    for (size_t w = blockIdx.x * (size_t)blockDim.x + threadIdx.x; w < n_words; w += (size_t)gridDim.x * blockDim.x) {
        uint32_t word = __ldg(bitmap + w);
        if (!word) continue;
        int rank = (int)__ldg(prefix + w);
        // decompose the word's first cell once (64-bit divisions are slow), then walk the set bits with carries
        const long long cell0 = (long long)w << 5;
        const int b = (int)(cell0 / cells_pad);
        long long r = cell0 - (long long)b * cells_pad;
        const int x0 = (int)(r % W); r /= W;
        const int y0 = (int)(r % H);
        const int z0 = (int)(r / H);
        while (word) {
            int bit = __ffs(word) - 1;
            word &= word - 1;
            if (rank < cap) {
                int x = x0 + bit, y = y0, z = z0;
                while (x >= W) { x -= W; if (++y == H) { y = 0; ++z; } }
                reinterpret_cast<int4*>(coords)[rank] = make_int4(b, z, y, x);
            }
            ++rank;
        }
    }
}

__global__ void __launch_bounds__(256) k_conv_nbr(const int32_t* __restrict__ out_coords, const int* __restrict__ d_n_out, int out_cap,
                                                  ConvGeom cg, GridIndex gin, TableOut to) {
    __shared__ int s_hist[SCHED_BINS];
    if (to.keys) { for (int b = threadIdx.x; b < SCHED_BINS; b += blockDim.x) s_hist[b] = 0; __syncthreads(); }
    int n = min(*d_n_out, out_cap);
    const int lane = threadIdx.x & 31;
    const int K = cg.k[0] * cg.k[1] * cg.k[2];
    for (int base = blockIdx.x * blockDim.x + threadIdx.x - lane; base < n; base += gridDim.x * blockDim.x) {     // warp-uniform trip count
        const int o = base + lane;
        int v[27];
        int frame = 0;
#pragma unroll
        for (int k = 0; k < 27; ++k) v[k] = -1;
        if (o < n) {
            int4 c = __ldg(reinterpret_cast<const int4*>(out_coords) + o);
            frame = c.x;
            int kz = 0, ky = 0, kx = 0;
#pragma unroll
            for (int k = 0; k < 27; ++k) {
                if (k < K) {
                    v[k] = grid_lookup(gin, c.x, c.y * cg.s[0] - cg.p[0] + kz, c.z * cg.s[1] - cg.p[1] + ky, c.w * cg.s[2] - cg.p[2] + kx);
                    if (++kx == cg.k[2]) { kx = 0; if (++ky == cg.k[1]) { ky = 0; ++kz; } }
                }
            }
        }
        table_emit(to, o < n, o, out_cap, v, K, s_hist, frame);
    }
    table_finish(to, s_hist);
}

// ---- direct path: neighbour masks line by line, no table ------------------------------------------------------------
// With a dilation of 1 the KW x-taps of one (kz, ky) kernel line are KW <= 3 adjacent cells of one lattice row, so one or two
// bitmap words hold all of them: one dependent load per line instead of one bitmap -> prefix -> perm chain per tap.  The
// x range is clipped to [0, W) first, so bits of the neighbouring x-row, of the frame's cells_pad tail or of the next word
// never enter (the same per-dimension bounds as grid_lookup).  Tap (kz, ky, kx) of output site (z, y, x) reads input cell
// (z*s - p + kz, y*s - p + ky, x*s - p + kx); a submanifold conv is s = 1, p = (k-1)/2.
struct LineWords {
    long long c_lo;                                 // first in-range cell of the line
    uint32_t w_lo, w_hi;                            // bitmap words of the first / last in-range cell (equal if one word)
    int x_lo, n;                                    // first in-range tap index kx, number of in-range taps (0: line outside)
};
__device__ __forceinline__ LineWords line_words(const GridIndex& g, int b, int z, int y, int x0, int KW) {
    LineWords l{0, 0, 0, 0, 0};
    if ((unsigned)z >= (unsigned)g.D || (unsigned)y >= (unsigned)g.H) return l;
    const int xlo = max(x0, 0), xhi = min(x0 + KW - 1, g.W - 1);
    if (xlo > xhi) return l;
    l.c_lo = (long long)b * g.cells_pad + ((long long)z * g.H + y) * g.W + xlo;
    const long long c_hi = l.c_lo + (xhi - xlo);
    l.w_lo = __ldg(g.bitmap + (l.c_lo >> 5));
    l.w_hi = (c_hi >> 5) != (l.c_lo >> 5) ? __ldg(g.bitmap + (c_hi >> 5)) : l.w_lo;
    l.x_lo = xlo - x0;
    l.n = xhi - xlo + 1;
    return l;
}
// bits 0..n-1 = cells c_lo .. c_lo+n-1 are active (the 64-bit window w_hi:w_lo starts at c_lo's word)
__device__ __forceinline__ uint32_t line_bits(const LineWords& l) {
    const unsigned long long win = ((unsigned long long)l.w_hi << 32) | l.w_lo;
    return (uint32_t)(win >> (l.c_lo & 31)) & ((1u << l.n) - 1u);
}

// 27-bit neighbour mask of one output site (the centre tap of a submanifold conv is the site itself: always live)
__device__ __forceinline__ uint32_t site_mask(const GridIndex& g, const ConvGeom& cg, int4 c, int centre) {
    const int z0 = c.y * cg.s[0] - cg.p[0], y0 = c.z * cg.s[1] - cg.p[1], x0 = c.w * cg.s[2] - cg.p[2];
    uint32_t m = 0;
#pragma unroll
    for (int kz = 0; kz < 3; ++kz)
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
            if (kz < cg.k[0] && ky < cg.k[1]) {
                const LineWords l = line_words(g, c.x, z0 + kz, y0 + ky, x0, cg.k[2]);
                if (l.n) m |= line_bits(l) << ((kz * cg.k[1] + ky) * cg.k[2] + l.x_lo);
            }
    if (centre >= 0) m |= 1u << centre;
    return m;
}

// mask pass: masks[i], keys[i] and the digest histogram exactly as table_emit leaves them, no table.  perm_walk (a
// submanifold conv on an index with perm): thread r takes row perm[r], i.e. rows in lattice order, so the lanes of a warp
// probe neighbouring cells and share bitmap lines (the rows themselves are in the voxelizer's first-appearance order).
__device__ __forceinline__ void mask_rows(const int32_t* __restrict__ coords, int n, const ConvGeom& cg, const GridIndex& g, int centre,
                                          const int32_t* __restrict__ perm_walk, const TableOut& to, int* s_hist) {
    const int K = cg.k[0] * cg.k[1] * cg.k[2];
    for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < n; r += gridDim.x * blockDim.x) {
        const int i = perm_walk ? __ldg(perm_walk + r) : r;
        const int4 c = __ldg(reinterpret_cast<const int4*>(coords) + i);    // b,z,y,x
        sched_emit(to, true, i, site_mask(g, cg, c, centre), K, s_hist, c.x);
    }
}
__global__ void __launch_bounds__(256) k_subm_mask(const int32_t* __restrict__ coords, const int* __restrict__ d_n, int cap, ConvGeom cg,
                                                   GridIndex g, int centre, const int32_t* __restrict__ perm_walk, TableOut to) {
    __shared__ int s_hist[SCHED_BINS];
    for (int b = threadIdx.x; b < SCHED_BINS; b += blockDim.x) s_hist[b] = 0;
    __syncthreads();
    mask_rows(coords, min(*d_n, cap), cg, g, centre, perm_walk, to, s_hist);
    table_finish(to, s_hist);
}
__global__ void __launch_bounds__(256) k_conv_mask(const int32_t* __restrict__ out_coords, const int* __restrict__ d_n_out, int out_cap,
                                                   ConvGeom cg, GridIndex gin, TableOut to) {
    __shared__ int s_hist[SCHED_BINS];
    for (int b = threadIdx.x; b < SCHED_BINS; b += blockDim.x) s_hist[b] = 0;
    __syncthreads();
    mask_rows(out_coords, min(*d_n_out, out_cap), cg, gin, -1, nullptr, to, s_hist);
    table_finish(to, s_hist);
}

static ConvGeom subm_geom(int D, int H, int W, const int* ks) {
    ConvGeom cg;
    const int dhw[3] = {D, H, W};
    for (int d = 0; d < 3; ++d) { cg.k[d] = ks[d]; cg.s[d] = 1; cg.p[d] = (ks[d] - 1) / 2; cg.in_dhw[d] = cg.out_dhw[d] = dhw[d]; }
    return cg;
}

extern "C" int dz_rulebook_subm_masks(const int32_t* coords, const int* d_n, int cap, int B, int D, int H, int W, const int* ks,
                                      const uint32_t* bitmap, const uint32_t* prefix, const int32_t* perm, void* sched_ws,
                                      int sched_frame_major, int perm_walk, dz_stream_t stream) {
    DZ_CHECK_ARG(coords && d_n && bitmap && prefix && sched_ws && cap >= 1 && (perm || !perm_walk));
    DZ_CHECK_ARG(ks[0] % 2 == 1 && ks[1] % 2 == 1 && ks[2] % 2 == 1 && ks[0] <= 3 && ks[1] <= 3 && ks[2] <= 3);
    TableOut to = table_out(nullptr, nullptr, sched_ws, cap, B, sched_frame_major);
    DZ_CUDA(cudaMemsetAsync(sched_ws, 0, sched_zero_bytes(cap), (cudaStream_t)stream));
    GridIndex g{bitmap, prefix, perm, B, D, H, W, dz_cells_pad(D, H, W)};
    const int blocks = max(1, min(dz_cdiv(cap, 256), DZ_NUM_SMS * 8));
    k_subm_mask<<<blocks, 256, 0, (cudaStream_t)stream>>>(coords, d_n, cap, subm_geom(D, H, W, ks), g, (ks[0] * ks[1] * ks[2] - 1) / 2,
                                                           perm_walk ? perm : nullptr, to);
    DZ_LAUNCH_CHECK();
    return DZ_OK;
}

__global__ void k_clamp_count(int* d_n, int cap) {
    if (threadIdx.x == 0 && blockIdx.x == 0 && *d_n > cap) *d_n = cap;   // overflow is reported by the host wrapper
}

// the strided conv with a table (nbr / tab) or, masks_only, the direct path's mask pass (sched_ws, no table)
static int rulebook_conv(const int32_t* in_coords, const int* d_n_in, int in_cap, int B, const int* in_dhw,
                         const int* ks, const int* st_, const int* pd, const uint32_t* in_bitmap,
                         const uint32_t* in_prefix, const int32_t* in_perm, int32_t* out_coords, int* d_n_out,
                         int out_cap, uint32_t* out_bitmap, uint32_t* out_prefix, int32_t* nbr, int32_t* tab, void* ws,
                         size_t ws_bytes, void* sched_ws, int sched_frame_major, bool masks_only, dz_stream_t stream) {
    DZ_CHECK_ARG(in_coords && d_n_in && in_bitmap && in_prefix && out_coords && d_n_out && out_bitmap && out_prefix);
    DZ_CHECK_ARG(masks_only ? (sched_ws && !nbr && !tab) : ((nbr || tab) && (!sched_ws || tab)));
    DZ_CHECK_ARG(in_cap >= 1 && out_cap >= 1 && B >= 1);
    ConvGeom cg;
    for (int d = 0; d < 3; ++d) {
        DZ_CHECK_ARG(ks[d] >= 1 && ks[d] <= 3 && st_[d] >= 1 && pd[d] >= 0);
        cg.k[d] = ks[d]; cg.s[d] = st_[d]; cg.p[d] = pd[d]; cg.in_dhw[d] = in_dhw[d];
        cg.out_dhw[d] = (in_dhw[d] + 2 * pd[d] - (ks[d] - 1) - 1) / st_[d] + 1;       // SURVEY A.2
    }
    cudaStream_t st = (cudaStream_t)stream;
    size_t out_words = dz_grid_index_words(B, cg.out_dhw[0], cg.out_dhw[1], cg.out_dhw[2]);
    if (ws_bytes < dz_scan_ws_bytes(out_words)) { dz_set_error("dz_rulebook_conv: workspace too small"); return DZ_ERR_WORKSPACE; }
    long long out_cp = dz_cells_pad(cg.out_dhw[0], cg.out_dhw[1], cg.out_dhw[2]);
    int blocks_in = max(1, min(dz_cdiv(in_cap, 256), DZ_NUM_SMS * 8));
    k_conv_mark<<<blocks_in, 256, 0, st>>>(in_coords, d_n_in, in_cap, cg, out_cp, out_bitmap);
    int rc = dz_grid_index_scan(out_bitmap, out_prefix, out_words, nullptr, d_n_out, ws, ws_bytes, stream);
    if (rc) return rc;
    int blocks_w = max(1, min(dz_cdiv((long long)out_words, 256), DZ_NUM_SMS * 8));
    k_index_to_coords<<<blocks_w, 256, 0, st>>>(out_bitmap, out_prefix, out_words, cg.out_dhw[0], cg.out_dhw[1], cg.out_dhw[2],
                                                out_cp, out_cap, out_coords);
    GridIndex gin{in_bitmap, in_prefix, in_perm, B, in_dhw[0], in_dhw[1], in_dhw[2], dz_cells_pad(in_dhw[0], in_dhw[1], in_dhw[2])};
    int blocks_out = max(1, min(dz_cdiv(out_cap, 256), DZ_NUM_SMS * 8));
    TableOut to = table_out(nbr, tab, sched_ws, out_cap, B, sched_frame_major);
    if (sched_ws) DZ_CUDA(cudaMemsetAsync(sched_ws, 0, sched_zero_bytes(out_cap), st));
    if (masks_only) k_conv_mask<<<blocks_out, 256, 0, st>>>(out_coords, d_n_out, out_cap, cg, gin, to);
    else k_conv_nbr<<<blocks_out, 256, 0, st>>>(out_coords, d_n_out, out_cap, cg, gin, to);
    DZ_LAUNCH_CHECK();
    return DZ_OK;
}

extern "C" int dz_rulebook_conv(const int32_t* in_coords, const int* d_n_in, int in_cap, int B, const int* in_dhw,
                                const int* ks, const int* st_, const int* pd, const uint32_t* in_bitmap,
                                const uint32_t* in_prefix, const int32_t* in_perm, int32_t* out_coords, int* d_n_out,
                                int out_cap, uint32_t* out_bitmap, uint32_t* out_prefix, int32_t* nbr, int32_t* tab, void* ws,
                                size_t ws_bytes, void* sched_ws, int sched_frame_major, dz_stream_t stream) {
    return rulebook_conv(in_coords, d_n_in, in_cap, B, in_dhw, ks, st_, pd, in_bitmap, in_prefix, in_perm, out_coords, d_n_out, out_cap,
                         out_bitmap, out_prefix, nbr, tab, ws, ws_bytes, sched_ws, sched_frame_major, false, stream);
}

extern "C" int dz_rulebook_conv_masks(const int32_t* in_coords, const int* d_n_in, int in_cap, int B, const int* in_dhw,
                                      const int* ks, const int* st_, const int* pd, const uint32_t* in_bitmap,
                                      const uint32_t* in_prefix, const int32_t* in_perm, int32_t* out_coords, int* d_n_out,
                                      int out_cap, uint32_t* out_bitmap, uint32_t* out_prefix, void* ws, size_t ws_bytes,
                                      void* sched_ws, int sched_frame_major, dz_stream_t stream) {
    return rulebook_conv(in_coords, d_n_in, in_cap, B, in_dhw, ks, st_, pd, in_bitmap, in_prefix, in_perm, out_coords, d_n_out, out_cap,
                         out_bitmap, out_prefix, nullptr, nullptr, ws, ws_bytes, sched_ws, sched_frame_major, true, stream);
}


// =====================================================================================================================
// Tile schedule for the output-stationary tensor-core conv: group the output rows whose neighbour masks are alike.
//
// The conv kernel owns 128 output rows per CTA and skips a kernel offset k when NONE of its rows has a neighbour through
// k.  In coordinate order a tile touches ~21-23 of the 27 offsets although each row only has 4.6 (0.1 m level) to 14.7
// (0.8 m level) neighbours; after grouping rows by mask a tile touches 7-17 offsets, i.e. the gather and the MMA work
// drop 1.3-3x (synthetic Waymo frame, profiles/r01_spconv_notes.md).  spconv's implicit-GEMM path sorts by the full mask
// for the same reason; here a single-pass counting sort on a 12-bit digest of the mask is enough: the digest keeps the
// five "line present" bits of the z+-1 planes, the six x+-1 bits of the centre plane and one more (order found by greedy
// search on the frame statistics), most significant first.  The digest and its histogram are produced by the rulebook
// kernel itself and scanned by its last block (sched_ws), so the schedule costs ONE more pass:
//   order[p]            tile position -> output row (descending digest: heavy rows first)
//   order[cap + j]      tile launch order: the j-th CTA takes the tile with the j-th largest number of live offsets
//                       (longest-processing-time-first; launch order follows blockIdx)
// The table itself stays in canonical row order (row-major, one 128-byte line per row); the conv kernel reads row
// order[p].  Every row's accumulation order over k is unchanged, so results are bit-identical to the unscheduled launch.
// =====================================================================================================================
// rows per scatter block: each block zeroes, flushes and re-reads a SCHED_BINS histogram, so a block must own many more rows
// than bins for that fixed cost to vanish (at 512 rows it was 8 bins per row)
static constexpr int SCHED_CHUNK = 4096;
__device__ __forceinline__ int tile_bin(int tm) {
    const int m = tm & 0x7ffffff;
    return m ? ((tm >> 27) & 15) * 28 + (27 - __popc(m)) : 511;
}
__global__ void __launch_bounds__(256) k_sched_scatter(const int32_t* __restrict__ masks, int cap, const int* __restrict__ d_n,
                                                       const uint16_t* __restrict__ keys, int* __restrict__ offs, int* __restrict__ tile_mask,
                                                       int* __restrict__ ticket, int32_t* __restrict__ order, int fb) {
    // block-aggregated counting-sort scatter: count this block's rows per digest in shared memory, reserve one global range
    // per (block, digest) with a single atomic, then hand out positions from shared memory.  The grid is sized by the
    // capacity (no host read of the count); blocks past the count only take their ticket.
    __shared__ int s_cnt[SCHED_BINS];
    const int n = min(*d_n, cap);
    const int r0 = blockIdx.x * SCHED_CHUNK, r1 = min(n, r0 + SCHED_CHUNK);
    if (r0 < r1) {
        for (int b = threadIdx.x; b < SCHED_BINS; b += blockDim.x) s_cnt[b] = 0;
        __syncthreads();
        for (int i = r0 + threadIdx.x; i < r1; i += blockDim.x) atomicAdd(s_cnt + keys[i], 1);
        __syncthreads();
        for (int b = threadIdx.x; b < SCHED_BINS; b += blockDim.x) {
            const int c = s_cnt[b];
            if (c) s_cnt[b] = atomicAdd(offs + b, c);
        }
        __syncthreads();
        for (int i = r0 + threadIdx.x; i < r1; i += blockDim.x) {
            const int pos = atomicAdd(s_cnt + keys[i], 1);
            order[pos] = i;
            int m = __ldg(masks + i);
            int* tm = tile_mask + (pos >> 7);
            if (fb && (pos & 127) == 0) m |= (int)(keys[i] >> (12 - fb)) << 27;      // the tile's frame group = its first row's (bits 27..30)
            if ((__ldcg(tm) & m) != m) atomicOr(tm, m);              // plain read first: after a few rows the tile's mask is complete
        }
    }
    // ---- the last block orders the tiles by descending work (counting sort over popc(mask) = 0..27)
    // frame-major: bin = frame group * 28 + (27 - live offsets); empty capacity tiles (mask 0) go last (bin 511)
    __shared__ int s_last, bins[512];
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(ticket, 1) == (int)gridDim.x - 1);
    __syncthreads();
    if (!s_last) return;
    for (int b = threadIdx.x; b < 512; b += blockDim.x) bins[b] = 0;
    __threadfence();
    __syncthreads();
    const int tiles = (cap + 127) >> 7;
    int32_t* tile_order = order + cap;
    // warp-aggregated (28 bins, thousands of tiles: per-tile shared-memory atomics on the same few counters serialise)
    const int lane = threadIdx.x & 31;
    for (int t0 = threadIdx.x - lane; t0 < tiles; t0 += blockDim.x) {
        const int t = t0 + lane;
        const int bin = t < tiles ? tile_bin(__ldcg(tile_mask + t)) : 999;
        const unsigned peers = __match_any_sync(0xffffffffu, bin);
        if (t < tiles && lane == __ffs(peers) - 1) atomicAdd(bins + bin, __popc(peers));
    }
    __syncthreads();
    {                                                                      // exclusive scan of the 512 bins, 2 per thread
        const int c0 = bins[2 * threadIdx.x], c1 = bins[2 * threadIdx.x + 1];
        int total;
        const int run = block_exclusive_scan(c0 + c1, &total);
        bins[2 * threadIdx.x] = run;
        bins[2 * threadIdx.x + 1] = run + c0;
    }
    __syncthreads();
    for (int t0 = threadIdx.x - lane; t0 < tiles; t0 += blockDim.x) {
        const int t = t0 + lane;
        const int bin = t < tiles ? tile_bin(__ldcg(tile_mask + t)) : 999;
        const unsigned peers = __match_any_sync(0xffffffffu, bin);
        const int leader = __ffs(peers) - 1;
        int start = 0;
        if (t < tiles && lane == leader) start = atomicAdd(bins + bin, __popc(peers));
        start = __shfl_sync(0xffffffffu, start, leader);
        if (t < tiles) tile_order[start + __popc(peers & ((1u << lane) - 1u))] = t;
    }
}

// tile-major copy of the scheduled table for the persistent conv kernel: tile j = (K+1) x 128 ints, plane k < K = neighbour row of
// tile position p through offset k (-1: none), plane K = the output row order[j*128 + p] (-1 beyond the count).  One contiguous
// block per tile: the conv kernel fetches it with ONE bulk copy instead of 128 dependent (order -> table line) gathers.
__global__ void __launch_bounds__(256) k_sched_tiles(const int32_t* __restrict__ tab, int cap, const int* __restrict__ d_n, int K,
                                                     const int32_t* __restrict__ order, const int* __restrict__ tile_mask, int32_t* __restrict__ tab_tiles) {
    const int n = min(*d_n, cap);
    const int tiles_n = (n + 127) >> 7;
    const int tiles = (cap + 127) >> 7;
    int32_t* mask_out = const_cast<int32_t*>(order) + cap + tiles;                 // order[cap + tiles + j] = OR of tile j's row masks
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < tiles; j += gridDim.x * blockDim.x) mask_out[j] = __ldg(tile_mask + j) & 0x7ffffff;
    for (int pos = blockIdx.x * blockDim.x + threadIdx.x; pos < tiles_n * 128; pos += gridDim.x * blockDim.x) {
        const int i = pos < n ? __ldg(order + pos) : -1;
        int w[28];
        const int4* rowp = reinterpret_cast<const int4*>(tab) + (size_t)(i < 0 ? 0 : i) * 8;
#pragma unroll
        for (int q = 0; q < 7; ++q) {
            const int4 t4 = i >= 0 ? __ldg(rowp + q) : make_int4(-1, -1, -1, -1);
            w[4 * q] = t4.x; w[4 * q + 1] = t4.y; w[4 * q + 2] = t4.z; w[4 * q + 3] = t4.w;
        }
        int32_t* dst = tab_tiles + (size_t)(pos >> 7) * (K + 1) * 128 + (pos & 127);
#pragma unroll
        for (int k = 0; k < 27; ++k)
            if (k < K) dst[k * 128] = w[k];
        dst[K * 128] = i;
    }
}

// direct path's tile pass: the same tile-major table as k_sched_tiles, but the ranks are computed here from the grid index
// (no row-major table exists).  One thread per tile position p: row i = order[p], its coordinates and mask; for each LIVE
// kernel line one or two bitmap words + prefix words give every tap's rank = prefix + popc (grid_lookup's arithmetic),
// then perm.  Plane k is written coalesced across the warp.
__global__ void __launch_bounds__(256) k_tiles_direct(const int32_t* __restrict__ coords, int cap, const int* __restrict__ d_n, ConvGeom cg,
                                                      GridIndex g, int centre, const int* __restrict__ masks, const int32_t* __restrict__ order,
                                                      const int* __restrict__ tile_mask, int32_t* __restrict__ tab_tiles) {
    const int n = min(*d_n, cap);
    const int tiles_n = (n + 127) >> 7;
    const int tiles = (cap + 127) >> 7;
    const int K = cg.k[0] * cg.k[1] * cg.k[2];
    int32_t* mask_out = const_cast<int32_t*>(order) + cap + tiles;                 // order[cap + tiles + j] = OR of tile j's row masks
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < tiles; j += gridDim.x * blockDim.x) mask_out[j] = __ldg(tile_mask + j) & 0x7ffffff;
    for (int pos = blockIdx.x * blockDim.x + threadIdx.x; pos < tiles_n * 128; pos += gridDim.x * blockDim.x) {
        const int i = pos < n ? __ldg(order + pos) : -1;
        int4 c = make_int4(0, 0, 0, 0);
        uint32_t m = 0;                                                            // no live tap beyond the count
        if (i >= 0) { c = __ldg(reinterpret_cast<const int4*>(coords) + i); m = (uint32_t)__ldg(masks + i); }
        const int z0 = c.y * cg.s[0] - cg.p[0], y0 = c.z * cg.s[1] - cg.p[1], x0 = c.w * cg.s[2] - cg.p[2];
        int32_t* dst = tab_tiles + (size_t)(pos >> 7) * (K + 1) * 128 + (pos & 127);
#pragma unroll
        for (int kz = 0; kz < 3; ++kz)
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
                if (kz >= cg.k[0] || ky >= cg.k[1]) continue;
                const int line = kz * cg.k[1] + ky;
                const uint32_t lm = (m >> (line * cg.k[2])) & ((1u << cg.k[2]) - 1u);
                LineWords l{0, 0, 0, 0, 0};
                uint32_t p_lo = 0, p_hi = 0;
                if (lm) {                                                          // live line: its words and prefixes
                    l = line_words(g, c.x, z0 + kz, y0 + ky, x0, cg.k[2]);
                    const size_t wi = (size_t)(l.c_lo >> 5);
                    p_lo = __ldg(g.prefix + wi);
                    p_hi = (l.c_lo & 31) + l.n > 32 ? __ldg(g.prefix + wi + 1) : p_lo;      // the line spans two words
                }
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) {
                    if (kx >= cg.k[2]) continue;
                    const int k = line * cg.k[2] + kx;
                    int v = -1;
                    if ((lm >> kx) & 1u) {
                        if (k == centre) {
                            v = i;                                                 // the site itself
                        } else {
                            const int bit = (int)(l.c_lo & 31) + (kx - l.x_lo);    // live => inside the clipped range
                            const uint32_t word = bit < 32 ? l.w_lo : l.w_hi;
                            const int rank = (int)((bit < 32 ? p_lo : p_hi) + __popc(word & ((1u << (bit & 31)) - 1u)));
                            v = g.perm ? __ldg(g.perm + rank) : rank;
                        }
                    }
                    dst[k * 128] = v;
                }
            }
        dst[K * 128] = i;
    }
}

extern "C" int dz_rulebook_schedule_direct(const int32_t* coords, int cap, const int* d_n, int B, const int* in_dhw, const int* ks,
                                           const int* st_, const int* pd, int subm, const uint32_t* in_bitmap, const uint32_t* in_prefix,
                                           const int32_t* in_perm, int32_t* order, void* sched_ws, size_t ws_bytes, int sched_frame_major,
                                           int32_t* tab_tiles, dz_stream_t stream) {
    DZ_CHECK_ARG(coords && d_n && in_bitmap && in_prefix && order && sched_ws && tab_tiles && cap >= 1 && B >= 1);
    if (ws_bytes < dz_rulebook_schedule_ws_bytes(cap)) { dz_set_error("dz_rulebook_schedule_direct: workspace too small"); return DZ_ERR_WORKSPACE; }
    ConvGeom cg;
    if (subm) {
        DZ_CHECK_ARG(ks[0] % 2 == 1 && ks[1] % 2 == 1 && ks[2] % 2 == 1 && ks[0] <= 3 && ks[1] <= 3 && ks[2] <= 3);
        cg = subm_geom(in_dhw[0], in_dhw[1], in_dhw[2], ks);
    } else {
        for (int d = 0; d < 3; ++d) {
            DZ_CHECK_ARG(ks[d] >= 1 && ks[d] <= 3 && st_[d] >= 1 && pd[d] >= 0);
            cg.k[d] = ks[d]; cg.s[d] = st_[d]; cg.p[d] = pd[d]; cg.in_dhw[d] = in_dhw[d];
            cg.out_dhw[d] = (in_dhw[d] + 2 * pd[d] - (ks[d] - 1) - 1) / st_[d] + 1;
        }
    }
    const int K = cg.k[0] * cg.k[1] * cg.k[2];
    cudaStream_t st = (cudaStream_t)stream;
    TableOut to = table_out(nullptr, nullptr, sched_ws, cap);
    k_sched_scatter<<<dz_cdiv(cap, SCHED_CHUNK), 256, 0, st>>>(to.masks, cap, d_n, to.keys, to.hist, to.hist + SCHED_BINS, to.ticket + 1, order,
                                                                sched_frame_bits(B, sched_frame_major));
    DZ_LAUNCH_CHECK();
    GridIndex g{in_bitmap, in_prefix, in_perm, B, in_dhw[0], in_dhw[1], in_dhw[2], dz_cells_pad(in_dhw[0], in_dhw[1], in_dhw[2])};
    const int blocks = max(1, min(dz_cdiv(cap, 256), DZ_NUM_SMS * 8));
    k_tiles_direct<<<blocks, 256, 0, st>>>(coords, cap, d_n, cg, g, subm ? (K - 1) / 2 : -1, to.masks, order, to.hist + SCHED_BINS, tab_tiles);
    DZ_LAUNCH_CHECK();
    return DZ_OK;
}

extern "C" int dz_rulebook_schedule(const int32_t* tab, int cap, const int* d_n, int32_t* order, void* sched_ws, size_t ws_bytes,
                                    int B, int sched_frame_major, int K, int32_t* tab_tiles, dz_stream_t stream) {
    DZ_CHECK_ARG(tab && d_n && order && sched_ws && cap >= 1);
    if (ws_bytes < dz_rulebook_schedule_ws_bytes(cap)) { dz_set_error("dz_rulebook_schedule: workspace too small"); return DZ_ERR_WORKSPACE; }
    TableOut to = table_out(nullptr, const_cast<int32_t*>(tab), sched_ws, cap);
    k_sched_scatter<<<dz_cdiv(cap, SCHED_CHUNK), 256, 0, (cudaStream_t)stream>>>(to.masks, cap, d_n, to.keys, to.hist, to.hist + SCHED_BINS, to.ticket + 1, order,
                                                                                 sched_frame_bits(B, sched_frame_major));
    DZ_LAUNCH_CHECK();
    if (tab_tiles) {
        DZ_CHECK_ARG(K >= 1 && K <= 27);
        const int blocks = max(1, min(dz_cdiv(cap, 256), DZ_NUM_SMS * 8));
        k_sched_tiles<<<blocks, 256, 0, (cudaStream_t)stream>>>(tab, cap, d_n, K, order, to.hist + SCHED_BINS, tab_tiles);
        DZ_LAUNCH_CHECK();
    }
    return DZ_OK;
}
