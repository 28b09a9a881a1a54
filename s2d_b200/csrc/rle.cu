// f2: COCO run-length encoding of binary masks on the GPU, with area and bounding box - the step right
// after the path: annotations.py:94-106 (mask_util.encode / area / toBbox per keymask) and
// convert_results_to_annotations.py:70-81. pycocotools' maskApi.c rleEncode walks the mask in
// COLUMN-major order and emits run lengths starting with a run of zeros; rleArea sums the odd runs;
// rleToBbox is the tight box of the set pixels as (x, y, w, h).
//
// Two kernels per batch of N masks (u8 [N][H][W], row-major, non-zero = set):
//   rle_colbits_kernel  transposes to column-major BITS: a warp reads a 32 x 32 tile with one 32-byte
//                       row segment per lane (whole sectors), 32 ballots turn it into the 32 column
//                       words of the tile; area (popc) and bbox (min / max) fall out of the same words.
//   rle_runs_kernel     one CTA per mask walks the column-major bit sequence: transitions
//                       b ^ (b << 1 | carry), a block-wide exclusive scan of their popcounts (warp
//                       shuffles) gives every transition its run index, the edges are written in order
//                       and differenced into run lengths.
// The delta / base-48 string compression of the counts (rleToString) stays on the host: it is a
// sequential pass over a few hundred integers.
#include "common.cuh"

#include <limits.h>

namespace s2d {

// colbits [N][W][HW] u32 (HW = ceil(H / 32)): bit y & 31 of word (x, y >> 5) = mask[y][x] != 0
__global__ void __launch_bounds__(128)
rle_colbits_kernel(const uint8_t* __restrict__ masks, int H, int W, int HW, uint32_t* __restrict__ colbits,
                   int32_t* __restrict__ area, int32_t* __restrict__ bbox) {
    const int n = blockIdx.z, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x0 = blockIdx.x * 32, yw = blockIdx.y * 4 + warp;      // word row of this warp
    if (yw >= HW) return;
    const int y = yw * 32 + lane;
    const uint8_t* m = masks + (int64_t)n * H * W;
    uint32_t b[8] = {0, 0, 0, 0, 0, 0, 0, 0};                       // the lane's row segment, 32 pixels
    if (y < H) {
        const uint8_t* row = m + (int64_t)y * W + x0;
        if (x0 + 32 <= W && ((reinterpret_cast<uintptr_t>(row) & 15) == 0)) {
            const uint4 a = *reinterpret_cast<const uint4*>(row), c = *reinterpret_cast<const uint4*>(row + 16);
            b[0] = a.x; b[1] = a.y; b[2] = a.z; b[3] = a.w; b[4] = c.x; b[5] = c.y; b[6] = c.z; b[7] = c.w;
        } else {
#pragma unroll
            for (int i = 0; i < 32; ++i)
                if (x0 + i < W) b[i >> 2] |= (uint32_t)row[i] << (8 * (i & 3));
        }
    }
    uint32_t mine = 0;                                               // column word of column x0 + lane
#pragma unroll
    for (int i = 0; i < 32; ++i) {
        const uint32_t w = __ballot_sync(0xffffffffu, ((b[i >> 2] >> (8 * (i & 3))) & 255u) != 0);
        if (lane == i) mine = w;
    }
    const int x = x0 + lane;
    S2D_DEV_ASSERT(x >= W || (yw < HW && n < (int)gridDim.z));
    if (x < W) colbits[((int64_t)n * W + x) * HW + yw] = mine;
    // area and bounding box
    const int cnt = __reduce_add_sync(0xffffffffu, __popc(mine));
    const uint32_t any_rows = __reduce_or_sync(0xffffffffu, mine);
    const uint32_t cols = __ballot_sync(0xffffffffu, mine != 0);
    if (lane == 0 && cnt) {
        atomicAdd(&area[n], cnt);
        int32_t* bb = bbox + 4 * n;                                  // xmin, ymin, xmax, ymax
        atomicMin(&bb[0], x0 + __ffs(cols) - 1);
        atomicMax(&bb[2], x0 + 31 - __clz(cols));
        atomicMin(&bb[1], yw * 32 + __ffs(any_rows) - 1);
        atomicMax(&bb[3], yw * 32 + 31 - __clz(any_rows));
    }
}

__global__ void rle_init_kernel(int N, int32_t* __restrict__ area, int32_t* __restrict__ bbox) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) {
        area[i] = 0;
        bbox[4 * i] = INT_MAX; bbox[4 * i + 1] = INT_MAX; bbox[4 * i + 2] = -1; bbox[4 * i + 3] = -1;
    }
}

constexpr int RLE_THREADS = 256;

// counts [N][max_runs]: run lengths in column-major order starting with zeros; nruns[n] is the true
// number of runs (may exceed max_runs: then only the first max_runs were written).
__global__ void __launch_bounds__(RLE_THREADS)
rle_runs_kernel(const uint32_t* __restrict__ colbits, int H, int W, int HW, int max_runs,
                int32_t* __restrict__ edges, int32_t* __restrict__ counts, int32_t* __restrict__ nruns) {
    __shared__ int wsum[RLE_THREADS / 32];
    const int n = blockIdx.x, tid = threadIdx.x;
    const uint32_t* cb = colbits + (int64_t)n * W * HW;
    int32_t* ed = edges + (int64_t)n * max_runs;
    int32_t* ct = counts + (int64_t)n * max_runs;
    const int nwords = W * HW;
    const uint32_t tailmask = (H & 31) ? ((1u << (H & 31)) - 1u) : 0xFFFFFFFFu;   // valid rows of a column's last word
    int running = 0;
    for (int base = 0; base < nwords; base += RLE_THREADS) {
        const int i = base + tid;
        uint32_t t = 0;
        int x = 0, j = 0;
        if (i < nwords) {
            x = i / HW; j = i - x * HW;
            const uint32_t b = cb[i];
            // the bit before this word's first row: last valid row of the previous word in sequence
            uint32_t prev = 0;
            if (i > 0) {
                const uint32_t pw = cb[i - 1];
                prev = (j == 0) ? ((pw >> ((H - 1) & 31)) & 1u) : (pw >> 31);
            }
            t = (b ^ ((b << 1) | prev)) & (j == HW - 1 ? tailmask : 0xFFFFFFFFu);
        }
        int total;
        int idx = running + block_excl_scan<RLE_THREADS>(__popc(t), wsum, total);
        while (t) {                                   // edges: column-major position of every transition
            const int bit = __ffs(t) - 1;
            t &= t - 1;
            S2D_DEV_ASSERT(idx >= 0 && x * H + j * 32 + bit <= H * W);
            if (idx < max_runs) ed[idx] = x * H + j * 32 + bit;
            ++idx;
        }
        running += total;
    }
    // run k = edges[k] - edges[k-1] (edges[-1] = 0), the last run ends at H * W. A mask that starts with a
    // set pixel has a transition at position 0, i.e. a leading zero-length run, exactly like rleEncode.
    const int ntr = running;
    const int total_runs = ntr + 1;
    __threadfence_block();
    __syncthreads();
    for (int k = tid; k < total_runs && k < max_runs; k += RLE_THREADS) {
        const int lo = k == 0 ? 0 : ed[k - 1];
        const int hi = k < ntr ? ed[k] : H * W;
        S2D_DEV_ASSERT(hi >= lo && k < max_runs);
        ct[k] = hi - lo;
    }
    if (tid == 0) nruns[n] = total_runs;
}

}  // namespace s2d

using namespace s2d;

extern "C" int s2d_rle_work_ints(int N, int H, int W, int max_runs, int64_t* out) {
    S2D_CHECK_ARG(out && N > 0 && H > 0 && W > 0 && max_runs > 0, "s2d_rle_work_ints: bad arguments");
    *out = (int64_t)N * W * ((H + 31) / 32) + (int64_t)N * max_runs;
    return 0;
}

extern "C" int s2d_rle_encode(const uint8_t* masks, int N, int H, int W, int max_runs, int32_t* work,
                              int32_t* counts, int32_t* nruns, int32_t* area, int32_t* bbox, void* stream) {
    S2D_ENTER(stream);
    S2D_CHECK_ARG(masks && work && counts && nruns && area && bbox, "s2d_rle_encode: null pointer");
    S2D_CHECK_ARG(N > 0 && N <= 65535 && H > 0 && W > 0 && max_runs > 0, "s2d_rle_encode: bad sizes");
    S2D_CHECK_ARG((int64_t)H * W < INT_MAX, "s2d_rle_encode: mask too large");
    cudaStream_t st = (cudaStream_t)stream;
    const int HW = (H + 31) / 32;
    uint32_t* colbits = reinterpret_cast<uint32_t*>(work);
    int32_t* edges = work + (int64_t)N * W * HW;
    rle_init_kernel<<<(N + 255) / 256, 256, 0, st>>>(N, area, bbox);
    S2D_CHECK_LAUNCH("rle_init_kernel");
    dim3 grid((W + 31) / 32, (HW + 3) / 4, N);
    rle_colbits_kernel<<<grid, 128, 0, st>>>(masks, H, W, HW, colbits, area, bbox);
    S2D_CHECK_LAUNCH("rle_colbits_kernel");
    rle_runs_kernel<<<N, RLE_THREADS, 0, st>>>(colbits, H, W, HW, max_runs, edges, counts, nruns);
    S2D_CHECK_LAUNCH("rle_runs_kernel");
    return 0;
}

// ------------------------------------------------------------------------------------------
// RLE -> area and bounding box (maskApi.c rleArea / rleToBbox; convert_results_to_annotations.py:
// 70-81 recomputes both for every predicted segmentation). One warp per RLE: the lanes walk the
// counts 32 at a time with a warp-wide inclusive scan carrying the running pixel position.
// rleToBbox semantics are kept to the letter: with cc the inclusive prefix of the first
// m = 2 * floor(n / 2) counts, boundary j sits at t = cc - (j & 1) (first pixel of a set run for
// even j, last pixel for odd j), x = t / h, y = t % h; a set run that crosses into another column
// makes the box span all rows; an RLE without a complete set run gives (0, 0, 0, 0).
// ------------------------------------------------------------------------------------------
namespace s2d {

__global__ void __launch_bounds__(128)
rle_area_bbox_kernel(const int32_t* __restrict__ counts, const int64_t* __restrict__ offsets, int N, const int32_t* __restrict__ hs,
                     int32_t* __restrict__ area, int32_t* __restrict__ bbox) {
    const int n = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (n >= N) return;
    const int32_t* c = counts + offsets[n];
    const int nr = (int)(offsets[n + 1] - offsets[n]);
    const int m = (nr / 2) * 2;
    const unsigned h = (unsigned)hs[n];
    unsigned carry = 0, a = 0;
    unsigned xs = 0xFFFFFFFFu, ys = 0xFFFFFFFFu, xe = 0, ye = 0;
    unsigned xp_carry = 0;                        // x of the latest even boundary seen so far
    bool full_rows = false;
    for (int base = 0; base < m; base += 32) {
        const int j = base + lane;
        S2D_DEV_ASSERT(j >= m || j < nr);
        const unsigned v = j < m ? (unsigned)c[j] : 0u;
        const unsigned cc = carry + warp_incl_scan(v);
        const unsigned t = cc - (unsigned)(j & 1);
        const unsigned y = t % h, x = (t - y) / h;
        // x of the preceding even boundary: the previous lane's (or the previous chunk's last even one)
        unsigned xprev = __shfl_up_sync(0xffffffffu, x, 1);
        if (lane == 0) xprev = xp_carry;
        if (j < m) {
            if (j & 1) { a += v; if (xprev < x) full_rows = true; }
            xs = min(xs, x); xe = max(xe, x); ys = min(ys, y); ye = max(ye, y);
        }
        carry = __shfl_sync(0xffffffffu, cc, 31);
        xp_carry = __shfl_sync(0xffffffffu, x, 30);          // lane 30 holds an even j (base is a multiple of 32)
    }
    a = __reduce_add_sync(0xffffffffu, a);
    xs = __reduce_min_sync(0xffffffffu, xs); ys = __reduce_min_sync(0xffffffffu, ys);
    xe = __reduce_max_sync(0xffffffffu, xe); ye = __reduce_max_sync(0xffffffffu, ye);
    full_rows = __any_sync(0xffffffffu, full_rows);
    if (lane == 0) {
        area[n] = (int32_t)a;
        int32_t* bb = bbox + 4 * n;
        if (m == 0) { bb[0] = bb[1] = bb[2] = bb[3] = 0; }
        else {
            if (full_rows) { ys = 0; ye = h - 1; }
            bb[0] = (int32_t)xs; bb[1] = (int32_t)ys; bb[2] = (int32_t)(xe - xs + 1); bb[3] = (int32_t)(ye - ys + 1);
        }
    }
}

}  // namespace s2d

extern "C" int s2d_rle_area_bbox(const int32_t* counts, const int64_t* offsets, int N, const int32_t* heights,
                                 int32_t* area, int32_t* bbox, void* stream) {
    S2D_ENTER(stream);
    S2D_CHECK_ARG(counts && offsets && heights && area && bbox && N > 0, "s2d_rle_area_bbox: bad arguments");
    rle_area_bbox_kernel<<<(N + 3) / 4, 128, 0, (cudaStream_t)stream>>>(counts, offsets, N, heights, area, bbox);
    S2D_CHECK_LAUNCH("rle_area_bbox_kernel");
    return 0;
}
