// Stage E on the device: COCO RLE of every (frame, label) keymask straight from the u8 label maps, and the
// base-48 string packing of run lengths (maskApi.c rleEncode / rleToString; annotations.py:94-106 calls them
// through pycocotools once per keymask PNG).
//
// The cost does not depend on the number of objects in a frame. In column-major order a transition between
// pixel labels a -> b is an edge of mask a and of mask b and of nothing else, so the edges of every mask of a
// frame come from one walk over the frame's transitions. A warp owns a strip of S <= 32 columns of one frame:
// it stages the strip in shared memory (coalesced row segments), then walks it column by column, 32 rows of a
// column per step; the ballot of "label differs from the pixel before" is almost always zero, and the rare
// transitions are handed out in order to per-label counters in the warp's shared memory. Because the warp owns
// whole columns, the per-label order of the edges it finds is column-major.
//
//   pass 1  lr_strip_kernel<false>   edges per (frame, strip, label) of every keymask row
//   scan    lr_frame_scan_kernel     per frame and label: exclusive prefix over strips; runs per row = edges + 1
//           offsets_kernel           runs per row -> int64 offsets of the rows in one flat `counts` buffer
//   pass 2  lr_strip_kernel<true>    edge positions written in order at offsets[row] + strip prefix + rank
//   diff    lr_diff_kernel           a warp per row turns its edges into run lengths in place, bounding box
// Each frame's bytes are read from HBM twice (pass 1 and pass 2). Nothing is written at or past `capacity`.
#include "common.cuh"

#include <limits.h>

namespace s2d {

constexpr int LR_WARPS = 4;                    // warps (strips) per CTA, fewer when a whole column of a tall frame is staged
constexpr int LR_SMEM_MAX = 200 * 1024;
constexpr int LR_STAGE_BYTES = 26624;          // staged strip per warp: 32 columns of up to 739 rows (720p at full width)
constexpr int LR_NONE = 256;                   // the "pixel" before (0, 0): no label

// strip width for frames of H rows and its shared-memory row stride: an odd number of words, so that 32 lanes
// reading one column of 32 consecutive rows hit 32 different banks
__host__ __device__ inline int lr_strip_width(int H) {
    if (H * 36 <= LR_STAGE_BYTES) return 32;
    if (H * 20 <= LR_STAGE_BYTES) return 16;
    if (H * 12 <= LR_STAGE_BYTES) return 8;
    if (H * 4 <= LR_STAGE_BYTES) return 4;
    return 1;
}
__host__ __device__ inline int lr_row_stride(int S) { return S == 32 ? 36 : S == 16 ? 20 : S == 8 ? 12 : S == 4 ? 4 : 1; }
// staged bytes per warp for a batch whose tallest frame has max_H rows (S = 1 stages a whole column)
inline int lr_stage_bytes(int max_H) { return max_H > LR_STAGE_BYTES ? (max_H + 15) & ~15 : LR_STAGE_BYTES; }
// strip slots per frame in the pass-1 table (strip width only shrinks with H)
inline int64_t lr_max_strips(int max_H, int max_W) { return (max_W + lr_strip_width(max_H) - 1) / lr_strip_width(max_H); }

template <bool WRITE>
__global__ void __launch_bounds__(LR_WARPS * 32)
lr_strip_kernel(const s2d_video_desc* __restrict__ descs, const int32_t* __restrict__ vidinfo,
                const int32_t* __restrict__ gid_of, int stage_bytes, int64_t max_strips, int32_t* __restrict__ scnt,
                const int64_t* __restrict__ offsets, int64_t capacity, int32_t* __restrict__ counts) {
    extern __shared__ __align__(16) uint8_t lr_smem[];
    __shared__ int gidt[S2D_MAX_LABELS];
    const int v = blockIdx.z, t = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const s2d_video_desc d = descs[v];
    if (t >= d.T || vidinfo[v * S2D_VIDINFO_WORDS + 3] != 1) return;      // the reference annotates status-1 videos only
    const int H = d.H, W = d.W, S = lr_strip_width(H), stride = lr_row_stride(S);
    const int nstrip = (W + S - 1) / S;
    const int64_t f = d.frame0 + t;
    for (int l = threadIdx.x; l < S2D_MAX_LABELS; l += blockDim.x) {
        const int g = gid_of[f * S2D_MAX_LABELS + l];
        gidt[l] = (g >= 0 && g < d.Nm) ? g : -1;
    }
    __syncthreads();
    const int s = blockIdx.x * nw + warp;
    if (s >= nstrip) return;
    S2D_DEV_ASSERT(s < max_strips);
    uint8_t* stage = lr_smem + (int64_t)warp * (stage_bytes + S2D_MAX_LABELS * 8);
    int64_t* wpos = reinterpret_cast<int64_t*>(stage + stage_bytes);     // WRITE: next slot per label
    int32_t* wcnt = reinterpret_cast<int32_t*>(wpos);                    // count pass: edges per label
    int32_t* srow = scnt + (f * max_strips + s) * S2D_MAX_LABELS;
    for (int l = lane; l < S2D_MAX_LABELS; l += 32) {
        if (WRITE) {
            const int g = gidt[l];
            S2D_DEV_ASSERT(g < 0 || d.row0 + g < d.row0 + d.Nm);
            wpos[l] = g >= 0 ? offsets[d.row0 + g] + srow[l] : 0;
        } else {
            wcnt[l] = 0;
        }
    }
    // stage the strip: rows 0..H-1, columns x0 .. x0 + ws - 1
    const int x0 = s * S, ws = min(S, W - x0);
    const uint8_t* frame = d.labels + (int64_t)t * H * W;
    const uint8_t* src = frame + x0;
    S2D_DEV_ASSERT(H * stride <= stage_bytes);
    const bool vec = ws == S && (S == 32 || S == 16) && (W & 15) == 0 && ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
    if (vec && S == 32) {
        for (int y = lane; y < H; y += 128) {
            int4 a[4], b[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int yy = y + 32 * k;
                if (yy < H) {
                    a[k] = ld_stream(reinterpret_cast<const int4*>(src + yy * W));
                    b[k] = ld_stream(reinterpret_cast<const int4*>(src + yy * W + 16));
                }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int yy = y + 32 * k;
                if (yy < H) {
                    uint32_t* r = reinterpret_cast<uint32_t*>(stage + yy * stride);
                    r[0] = a[k].x; r[1] = a[k].y; r[2] = a[k].z; r[3] = a[k].w;
                    r[4] = b[k].x; r[5] = b[k].y; r[6] = b[k].z; r[7] = b[k].w;
                }
            }
        }
    } else if (vec) {
        for (int y = lane; y < H; y += 128) {
            int4 a[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) if (y + 32 * k < H) a[k] = ld_stream(reinterpret_cast<const int4*>(src + (y + 32 * k) * W));
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int yy = y + 32 * k;
                if (yy < H) {
                    uint32_t* r = reinterpret_cast<uint32_t*>(stage + yy * stride);
                    r[0] = a[k].x; r[1] = a[k].y; r[2] = a[k].z; r[3] = a[k].w;
                }
            }
        }
    } else {
        const int n = H * ws;
        for (int i = lane; i < n; i += 32) {
            const int y = i / ws, c = i - y * ws;
            S2D_DEV_ASSERT(y * stride + c < stage_bytes);
            stage[y * stride + c] = src[y * W + c];
        }
    }
    __syncwarp();
    // walk the strip in column-major order
    int carry = x0 > 0 ? (int)frame[(H - 1) * W + x0 - 1] : LR_NONE;    // the pixel before (0, x0)
    for (int c = 0; c < ws; ++c) {
        const int x = x0 + c;
        for (int y0 = 0; y0 < H; y0 += 32) {
            const int y = y0 + lane;
            const bool in = y < H;
            S2D_DEV_ASSERT(!in || y * stride + c < stage_bytes);
            const int cur = in ? (int)stage[y * stride + c] : 0;
            int prev = __shfl_up_sync(0xffffffffu, cur, 1);
            if (lane == 0) prev = carry;
            uint32_t bits = __ballot_sync(0xffffffffu, in && cur != prev);
            carry = __shfl_sync(0xffffffffu, cur, min(31, H - 1 - y0));
            while (bits) {                                               // warp-uniform: edges in column order
                const int j = __ffs(bits) - 1;
                bits &= bits - 1;
                const int a = __shfl_sync(0xffffffffu, prev, j), b = __shfl_sync(0xffffffffu, cur, j);
                if (lane == 0) {
                    const int pos = x * H + y0 + j;
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int l = e ? b : a;
                        if (l < S2D_MAX_LABELS && gidt[l] >= 0) {
                            if (WRITE) {
                                const int64_t idx = wpos[l]++;
                                S2D_DEV_ASSERT(idx >= 0);
                                if (idx < capacity) counts[idx] = pos;
                            } else {
                                ++wcnt[l];
                            }
                        }
                    }
                }
            }
        }
    }
    if (!WRITE) {
        __syncwarp();
        for (int l = lane; l < S2D_MAX_LABELS; l += 32)
            if (gidt[l] >= 0) srow[l] = wcnt[l];
    }
}

// per frame: exclusive prefix of the pass-1 counts over strips (in place), runs of each row = edges + 1
__global__ void __launch_bounds__(S2D_MAX_LABELS)
lr_frame_scan_kernel(const s2d_video_desc* __restrict__ descs, const int32_t* __restrict__ vidinfo,
                     const int32_t* __restrict__ gid_of, int64_t max_strips, int32_t* __restrict__ scnt,
                     int32_t* __restrict__ rowruns) {
    const int v = blockIdx.y, t = blockIdx.x, l = threadIdx.x;
    const s2d_video_desc d = descs[v];
    if (t >= d.T || vidinfo[v * S2D_VIDINFO_WORDS + 3] != 1) return;
    const int64_t f = d.frame0 + t;
    const int g = gid_of[f * S2D_MAX_LABELS + l];
    if (g < 0 || g >= d.Nm) return;
    const int S = lr_strip_width(d.H), nstrip = (d.W + S - 1) / S;
    int32_t* col = scnt + f * max_strips * S2D_MAX_LABELS + l;
    int run = 0;
    for (int s = 0; s < nstrip; ++s) {
        S2D_DEV_ASSERT(s < max_strips);
        const int c = col[(int64_t)s * S2D_MAX_LABELS];
        col[(int64_t)s * S2D_MAX_LABELS] = run;
        run += c;
    }
    rowruns[d.row0 + g] = run + 1;
}

// out[i] = in[0] + ... + in[i - 1] (int64) for i = 0 .. n, *total = out[n]. One CTA; the next step's inputs are
// loaded before the current step's scan, so the load latency overlaps the scan's barriers instead of adding to them.
constexpr int OFFSETS_THREADS = 1024;
__global__ void __launch_bounds__(OFFSETS_THREADS)
offsets_kernel(const int32_t* __restrict__ in, int64_t n, int64_t* __restrict__ out, int64_t* __restrict__ total) {
    __shared__ int64_t wsum[OFFSETS_THREADS / 32];
    int64_t carry = 0;
    int x = threadIdx.x < n ? in[threadIdx.x] : 0;
    for (int64_t base = 0; base < n; base += OFFSETS_THREADS) {
        const int64_t i = base + threadIdx.x, next = i + OFFSETS_THREADS;
        const int xn = next < n ? in[next] : 0;
        int64_t tot;
        const int64_t ex = block_excl_scan<OFFSETS_THREADS, int64_t>(x, wsum, tot);
        if (i < n) out[i] = carry + ex;
        carry += tot;
        x = xn;
    }
    if (threadIdx.x == 0) { out[n] = carry; *total = carry; }
}

int launch_offsets(const int32_t* in, int64_t n, int64_t* out, int64_t* total, cudaStream_t st) {
    offsets_kernel<<<1, OFFSETS_THREADS, 0, st>>>(in, n, out, total);
    S2D_CHECK_LAUNCH("offsets_kernel");
    return 0;
}

// A warp per keymask row: its edges e_0 < ... < e_{n-1} (column-major positions) become the run lengths
// e_0, e_1 - e_0, ..., H * W - e_{n-1} in place, chunk by chunk (a chunk is read before it is overwritten, the
// previous chunk's last edge is carried in a register). Set runs are [e_2k, e_2k+1) (e_n = H * W); a set run that
// crosses a column boundary covers row H - 1 and row 0, so the box spans all rows. bbox = xmin, ymin, xmax, ymax.
constexpr int LR_DIFF_WARPS = 8;
__global__ void __launch_bounds__(LR_DIFF_WARPS * 32)
lr_diff_kernel(const s2d_video_desc* __restrict__ descs, const int32_t* __restrict__ vidinfo,
               const int64_t* __restrict__ offsets, int64_t capacity, int32_t* __restrict__ counts,
               int32_t* __restrict__ bbox) {
    const int v = blockIdx.y, lane = threadIdx.x & 31;
    const s2d_video_desc d = descs[v];
    const int q = blockIdx.x * LR_DIFF_WARPS + (threadIdx.x >> 5);
    if (q >= d.Nm || vidinfo[v * S2D_VIDINFO_WORDS + 3] != 1) return;
    const int64_t r = d.row0 + q;
    const int64_t o0 = offsets[r], o1 = offsets[r + 1];
    if (o1 > capacity || o1 <= o0) return;                               // incomplete (caller re-runs) or no runs
    const int n = (int)(o1 - o0 - 1), H = d.H, HW = d.H * d.W;
    int32_t* e = counts + o0;
    int carry = 0;
    int xs = INT_MAX, xe = -1, ys = INT_MAX, ye = -1;
    for (int base = 0; base <= n; base += 32) {
        const int j = base + lane;
        S2D_DEV_ASSERT(j > n || o0 + j < capacity);
        const int ej = j < n ? e[j] : HW;                                // e_n = H * W closes the last run
        const int enext = __shfl_down_sync(0xffffffffu, ej, 1);         // lane 31 (odd j) never needs it
        int eprev = __shfl_up_sync(0xffffffffu, ej, 1);
        if (lane == 0) eprev = carry;
        carry = __shfl_sync(0xffffffffu, ej, 31);
        if (j < n && !(j & 1)) {                                         // set run [e_j, e_j+1)
            const int hi = (j + 1 < n ? enext : HW) - 1;
            const int x0 = ej / H, x1 = hi / H;
            xs = min(xs, x0); xe = max(xe, x1);
            if (x0 != x1) { ys = 0; ye = H - 1; }
            else { ys = min(ys, ej - x0 * H); ye = max(ye, hi - x1 * H); }
        }
        __syncwarp();
        if (j <= n) e[j] = ej - eprev;
    }
    xs = __reduce_min_sync(0xffffffffu, xs); ys = __reduce_min_sync(0xffffffffu, ys);
    xe = __reduce_max_sync(0xffffffffu, xe); ye = __reduce_max_sync(0xffffffffu, ye);
    if (lane == 0) {
        int32_t* bb = bbox + 4 * r;
        bb[0] = xs; bb[1] = ys; bb[2] = xe; bb[3] = ye;
    }
}

// ------------------------------------------------------------------------------------------
// rleToString: x = cnts[i] (minus cnts[i-2] for i > 2), then 5-bit groups low to high with the continuation bit
// 0x20 and +48; a group ends the value once the rest is 0 (or -1 for a set sign bit 0x10). Every count depends
// only on the value two places back, so lengths and digits are computed per count and placed by a scan.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ int rs_value(const int32_t* c, int i) { return i > 2 ? c[i] - c[i - 2] : c[i]; }
__device__ __forceinline__ int rs_len(int x) {
    int len = 0;
    bool more = true;
    while (more) {
        const int c = x & 0x1F;
        x >>= 5;
        more = (c & 0x10) ? x != -1 : x != 0;
        ++len;
    }
    return len;
}

constexpr int RS_WARPS = 8;
// warp per mask; WRITE = false: lens[n] = string length; WRITE = true: the characters at str_off[n]
template <bool WRITE>
__global__ void __launch_bounds__(RS_WARPS * 32)
rs_kernel(const int32_t* __restrict__ counts, const int64_t* __restrict__ offsets, int N, int64_t ncounts,
          int32_t* __restrict__ lens, const int64_t* __restrict__ str_off, int64_t capacity, char* __restrict__ chars) {
    const int n = blockIdx.x * RS_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (n >= N) return;
    const int64_t o0 = offsets[n], o1 = offsets[n + 1];
    const bool ok = o1 <= ncounts && o1 >= o0;                           // counts that were not all written: empty
    const int nc = ok ? (int)(o1 - o0) : 0;
    const int32_t* c = counts + o0;
    int64_t pos = WRITE ? str_off[n] : 0;
    int total = 0;
    for (int base = 0; base < nc; base += 32) {
        const int i = base + lane;
        S2D_DEV_ASSERT(i >= nc || o0 + i < ncounts);
        int x = i < nc ? rs_value(c, i) : 0;
        const int len = i < nc ? rs_len(x) : 0;
        if (WRITE) {
            const int incl = warp_incl_scan(len);
            int64_t p = pos + incl - len;
            for (int k = 0; k < len; ++k, ++p) {
                int ch = x & 0x1F;
                x >>= 5;
                if (k + 1 < len) ch |= 0x20;
                if (p < capacity) chars[p] = (char)(ch + 48);
            }
            pos += __shfl_sync(0xffffffffu, incl, 31);
        } else {
            total += __reduce_add_sync(0xffffffffu, len);
        }
    }
    if (!WRITE && lane == 0) lens[n] = total;
}

}  // namespace s2d

using namespace s2d;

extern "C" int s2d_label_rle_work_ints(int64_t total_frames, int64_t total_rows, int max_H, int max_W, int64_t* out) {
    S2D_CHECK_ARG(out && total_frames > 0 && total_rows >= 0 && max_H > 0 && max_W > 0, "s2d_label_rle_work_ints: bad arguments");
    *out = total_frames * lr_max_strips(max_H, max_W) * S2D_MAX_LABELS + total_rows;
    return 0;
}

extern "C" int s2d_label_rle(const s2d_video_desc* descs, int nvideos, int max_T, int max_H, int max_W, int max_Nm,
                             int64_t total_frames, int64_t total_rows, const int32_t* gid_of, const int32_t* vidinfo,
                             int32_t* work, int64_t capacity, int32_t* counts, int64_t* offsets, int32_t* bbox,
                             int64_t* needed, void* stream) {
    S2D_ENTER(stream);
    S2D_CHECK_ARG(descs && gid_of && vidinfo && work && counts && offsets && bbox && needed, "s2d_label_rle: null pointer");
    S2D_CHECK_ARG(nvideos > 0 && nvideos <= 65535 && max_T > 0 && max_T <= 65535 && max_H > 0 && max_W > 0 && max_Nm > 0 &&
                  total_frames > 0 && total_rows > 0 && capacity >= 0, "s2d_label_rle: bad sizes");
    S2D_CHECK_ARG((int64_t)max_H * max_W < INT_MAX, "s2d_label_rle: frame too large (H * W must be < 2^31)");
    S2D_CHECK_ARG(max_H <= 65535, "s2d_label_rle: H > 65535");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t max_strips = lr_max_strips(max_H, max_W);
    int32_t* scnt = work;
    int32_t* rowruns = work + total_frames * max_strips * S2D_MAX_LABELS;
    const int stage = lr_stage_bytes(max_H);
    const int per_warp = stage + S2D_MAX_LABELS * 8;
    const int nw = per_warp * LR_WARPS <= LR_SMEM_MAX ? LR_WARPS : LR_SMEM_MAX / per_warp;
    const int smem = nw * per_warp;
    static bool done0[S2D_MAX_DEVICES], done1[S2D_MAX_DEVICES];
    if (opt_in_smem(lr_strip_kernel<false>, LR_SMEM_MAX, done0) != cudaSuccess ||
        opt_in_smem(lr_strip_kernel<true>, LR_SMEM_MAX, done1) != cudaSuccess) {
        set_error("s2d_label_rle: shared memory opt-in failed");
        cudaGetLastError();
        return -2;
    }
    if (cudaMemsetAsync(rowruns, 0, total_rows * sizeof(int32_t), st) != cudaSuccess) {
        set_error("s2d_label_rle: memset failed");
        cudaGetLastError();
        return -2;
    }
    const dim3 grid((unsigned)((max_strips + nw - 1) / nw), max_T, nvideos);
    lr_strip_kernel<false><<<grid, nw * 32, smem, st>>>(descs, vidinfo, gid_of, stage, max_strips, scnt, nullptr,
                                                               capacity, counts);
    S2D_CHECK_LAUNCH("lr_strip_kernel<count>");
    lr_frame_scan_kernel<<<dim3(max_T, nvideos), S2D_MAX_LABELS, 0, st>>>(descs, vidinfo, gid_of, max_strips, scnt, rowruns);
    S2D_CHECK_LAUNCH("lr_frame_scan_kernel");
    if (const int rc = launch_offsets(rowruns, total_rows, offsets, needed, st)) return rc;
    lr_strip_kernel<true><<<grid, nw * 32, smem, st>>>(descs, vidinfo, gid_of, stage, max_strips, scnt, offsets,
                                                              capacity, counts);
    S2D_CHECK_LAUNCH("lr_strip_kernel<write>");
    lr_diff_kernel<<<dim3((max_Nm + LR_DIFF_WARPS - 1) / LR_DIFF_WARPS, nvideos), LR_DIFF_WARPS * 32, 0, st>>>(
        descs, vidinfo, offsets, capacity, counts, bbox);
    S2D_CHECK_LAUNCH("lr_diff_kernel");
    return 0;
}

extern "C" int s2d_rle_strings(const int32_t* counts, const int64_t* offsets, int N, int64_t ncounts, int32_t* work,
                               int64_t capacity, char* chars, int64_t* str_offsets, int64_t* needed, void* stream) {
    S2D_ENTER(stream);
    S2D_CHECK_ARG(counts && offsets && work && chars && str_offsets && needed, "s2d_rle_strings: null pointer");
    S2D_CHECK_ARG(N > 0 && ncounts >= 0 && capacity >= 0, "s2d_rle_strings: bad sizes");
    cudaStream_t st = (cudaStream_t)stream;
    const int blocks = (N + RS_WARPS - 1) / RS_WARPS;
    rs_kernel<false><<<blocks, RS_WARPS * 32, 0, st>>>(counts, offsets, N, ncounts, work, nullptr, capacity, chars);
    S2D_CHECK_LAUNCH("rs_kernel<length>");
    if (const int rc = launch_offsets(work, N, str_offsets, needed, st)) return rc;
    rs_kernel<true><<<blocks, RS_WARPS * 32, 0, st>>>(counts, offsets, N, ncounts, work, str_offsets, capacity, chars);
    S2D_CHECK_LAUNCH("rs_kernel<write>");
    return 0;
}
