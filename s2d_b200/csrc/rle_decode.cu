// COCO RLE back to masks on the device: the inverse of stage E's s2d_label_rle + s2d_rle_strings.
//
//   s2d_rle_from_strings (maskApi.c rleFrString for N strings back to back)
//     rp_count_kernel     warp per string: number of values = characters whose continuation bit 0x20 is clear
//     offsets_kernel      one CTA (launch_offsets): exclusive prefix -> count_offsets [N + 1], needed
//     rp_write_kernel     warp per string, 32 characters per step: a ballot of the value ends, a segmented OR scan
//                         assembles each value from its 5-bit groups, and two plain warp scans run the parity chains
//   s2d_rle_decode (maskApi.c rleDecode, each mask independently)
//     rd_scan_kernel      warp per mask: exclusive prefix of the run lengths = each run's column-major start (int64)
//     rd_tile_kernel      CTA per 64 x 128 tile of a mask (a fixed number of CTAs per mask stride over its tiles):
//                         per column a binary search finds the run that covers the tile's first row; a tile inside
//                         one run is stored straight from registers, any other is filled column by column into
//                         shared memory and stored row-major with 16-byte stores
//
// Value rules of rleFrString: c = byte - 48; a value ends at a character whose bit 0x20 is clear; groups are the low
// 5 bits, least significant first, sign-extended from bit 0x10 of the last; for m > 2, cnts[m] = x + cnts[m - 2]. So
// the counts are two interleaved prefix sums: odd indices from 1, even indices from 2, index 0 alone. A string is
// malformed (status 1) when its last character still has the continuation bit set (rleFrString reads past the end,
// from_string raises) or when a count falls outside [0, 2^31). Every value of a well-formed string lies in
// (-2^31, 2^31), so a value outside it marks the string, and within it the chains are exact in uint32: the first
// count that leaves [0, 2^31) reads as >= 2^31 there. Values longer than 12 groups are tracked as their low 60 bits and
// whether the groups above match the sign (anything else is at least 2^60 in magnitude).
#include <algorithm>

#include "common.cuh"

namespace s2d {

constexpr int RP_WARPS = 8;                    // strings per CTA
constexpr int RD_SCAN_WARPS = 8;               // masks per CTA of the run-start scan
constexpr int RD_TC = 128;                     // tile columns = threads of rd_tile_kernel
constexpr int RD_TR = 64;                      // tile rows
constexpr int RD_PITCH = RD_TC + 16;           // a row's bytes sit at its global address mod 16, so 16-byte chunks line up
constexpr int RD_CHUNKS = RD_PITCH / 16;

__device__ __forceinline__ int rp_char(const char* __restrict__ s, int64_t i) { return ((int)(uint8_t)s[i] - 48) & 0x3F; }

__global__ void __launch_bounds__(RP_WARPS * 32)
rp_count_kernel(const char* __restrict__ chars, const int64_t* __restrict__ str_off, int N, int32_t* __restrict__ nvals) {
    const int n = blockIdx.x * RP_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (n >= N) return;
    const int64_t s0 = str_off[n], s1 = str_off[n + 1];
    S2D_DEV_ASSERT(s0 >= 0 && s1 >= s0 && s1 - s0 < INT_MAX);
    int cnt = 0;
    for (int64_t base = s0; base < s1; base += 4 * 32) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int64_t i = base + 32 * k + lane;
            if (i < s1) cnt += !(rp_char(chars, i) & 0x20);
        }
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) nvals[n] = cnt;
}

__global__ void __launch_bounds__(RP_WARPS * 32)
rp_write_kernel(const char* __restrict__ chars, const int64_t* __restrict__ str_off, int N,
                const int64_t* __restrict__ count_off, int64_t capacity, int32_t* __restrict__ counts,
                int32_t* __restrict__ status) {
    const int n = blockIdx.x * RP_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (n >= N) return;
    const int64_t s0 = str_off[n], s1 = str_off[n + 1], c0 = count_off[n];
    [[maybe_unused]] const int64_t c1 = count_off[n + 1];
    S2D_DEV_ASSERT(s0 >= 0 && s1 >= s0 && c0 >= 0 && c1 >= c0);
    const unsigned lt = (1u << lane) - 1u;
    // the value in progress across steps: low 60 bits, groups so far, groups >= 12 not 0 / not 0x1F
    uint64_t xl = 0;
    int xk = 0, xhi = 0;
    uint32_t chain_odd = 0, chain_even = 0;
    int64_t j = 0;                                                         // values of the string so far
    bool bad = false;
    int cnext = s0 + lane < s1 ? rp_char(chars, s0 + lane) : 0;
    for (int64_t base = s0; base < s1; base += 32) {
        const bool valid = base + lane < s1;
        const int c = cnext;
        if (base + 32 + lane < s1) cnext = rp_char(chars, base + 32 + lane);
        const unsigned term = __ballot_sync(0xffffffffu, valid && !(c & 0x20));
        const unsigned lower = term & lt;
        const int head = lower ? 32 - __clz(lower) : 0;                   // first lane of this lane's value in the step
        const int k = lane - head + (lower ? 0 : xk);                     // group index of this character in its value
        const int g = c & 0x1F;
        uint64_t lo = k < 12 ? (uint64_t)g << (5 * k) : 0;
        int hi = k < 12 ? 0 : (g != 0) | ((g != 0x1F) << 1);
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {                                 // OR over the lanes [head, lane]
            const uint64_t ulo = __shfl_up_sync(0xffffffffu, lo, o);
            const int uhi = __shfl_up_sync(0xffffffffu, hi, o);
            if (lane - o >= head) { lo |= ulo; hi |= uhi; }
        }
        if (!lower) { lo |= xl; hi |= xhi; }                               // the value started in an earlier step
        const bool ends = (term >> lane) & 1u;
        const int64_t jl = j + __popc(lower);
        uint32_t u = 0;
        if (ends) {
            const bool neg = c & 0x10;
            const int64_t x = (int64_t)(neg ? lo | (~0ull << min(5 * (k + 1), 60)) : lo);
            bad |= (hi & (neg ? 2 : 1)) || x >= ((int64_t)1 << 31) || x <= -((int64_t)1 << 31);
            u = (uint32_t)x;
        }
        const uint32_t so = warp_incl_scan(ends && (jl & 1) ? u : 0u);
        const uint32_t se = warp_incl_scan(ends && !(jl & 1) && jl >= 2 ? u : 0u);
        if (ends) {
            const uint32_t cnt = jl == 0 ? u : (jl & 1) ? chain_odd + so : chain_even + se;
            bad |= cnt >= 0x80000000u;
            const int64_t q = c0 + jl;
            S2D_DEV_ASSERT(q < c1);
            if (q < capacity) counts[q] = (int32_t)cnt;
        }
        chain_odd += __shfl_sync(0xffffffffu, so, 31);
        chain_even += __shfl_sync(0xffffffffu, se, 31);
        j += __popc(term);
        const uint64_t l31 = __shfl_sync(0xffffffffu, lo, 31);
        const int h31 = __shfl_sync(0xffffffffu, hi, 31), k31 = __shfl_sync(0xffffffffu, k, 31);
        if (term >> 31) { xl = 0; xk = 0; xhi = 0; }
        else { xl = l31; xk = k31 + 1; xhi = h31; }
    }
    S2D_DEV_ASSERT(c0 + j == c1);
    bad = __any_sync(0xffffffffu, bad);
    if (lane == 0) status[n] = (bad || (s1 > s0 && (rp_char(chars, s1 - 1) & 0x20))) ? 1 : 0;
}

__device__ __forceinline__ bool rd_size_ok(int H, int W) { return H >= 0 && W >= 0 && H <= 65535 && W <= 65535 && (int64_t)H * W < INT_MAX; }

// warp per mask: starts[coff[n] + n + i] = sum of the first i runs (i = 0 .. nc); status |= 2 unless the sum is H * W
__global__ void __launch_bounds__(RD_SCAN_WARPS * 32)
rd_scan_kernel(const int32_t* __restrict__ counts, const int64_t* __restrict__ coff, int N, const int32_t* __restrict__ hs,
               const int32_t* __restrict__ ws, int64_t* __restrict__ starts, int32_t* __restrict__ status) {
    const int n = blockIdx.x * RD_SCAN_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (n >= N) return;
    const int64_t c0 = coff[n], nc = coff[n + 1] - c0;
    S2D_DEV_ASSERT(c0 >= 0 && nc >= 0);
    int64_t* st = starts + c0 + n;
    if (lane == 0) st[0] = 0;
    int64_t carry = 0;
    for (int64_t base = 0; base < nc; base += 32) {
        const int64_t i = base + lane;
        const int64_t incl = warp_incl_scan<int64_t>(i < nc ? (uint32_t)counts[c0 + i] : 0u);  // maskApi's counts are unsigned
        if (i < nc) st[i + 1] = carry + incl;
        carry += __shfl_sync(0xffffffffu, incl, 31);
    }
    const int H = hs[n], W = ws[n];
    if (lane == 0 && (!rd_size_ok(H, W) || carry != (int64_t)H * W)) status[n] |= 2;
}

__global__ void __launch_bounds__(RD_TC)
rd_tile_kernel(const int64_t* __restrict__ coff, int N, const int32_t* __restrict__ hs, const int32_t* __restrict__ ws,
               const int64_t* __restrict__ out_off, const int64_t* __restrict__ starts, int per_mask,
               uint8_t* __restrict__ out) {
    __shared__ __align__(16) uint8_t tile[RD_TR * RD_PITCH];
    const int n = blockIdx.x / per_mask, g = blockIdx.x % per_mask, tid = threadIdx.x;
    if (n >= N) return;
    const int H = hs[n], W = ws[n];
    if (!rd_size_ok(H, W)) return;
    const int64_t c0 = coff[n];
    const int nc = (int)(coff[n + 1] - c0);
    const int64_t* __restrict__ st = starts + c0 + n;                     // nc + 1 run starts, st[nc] = the sum
    const int64_t total = st[nc];
    uint8_t* const dst = out + out_off[n];
    const int tiles_x = (W + RD_TC - 1) / RD_TC, ntiles = tiles_x * ((H + RD_TR - 1) / RD_TR);
    for (int t = g; t < ntiles; t += per_mask) {
        const int y0 = t / tiles_x * RD_TR, x0 = t % tiles_x * RD_TC;
        const int rows = min(RD_TR, H - y0), cols = min(RD_TC, W - x0);
        const int64_t p0 = (int64_t)(x0 + tid) * H + y0;                  // column-major index of (y0, x0 + tid)
        int r = nc, v = 0;                                                 // run covering p0 (nc: past the runs, 0)
        bool uni = true;
        if (tid < cols) {
            if (p0 < total) {
                int lo = 0, hi = nc - 1;                                   // largest r with st[r] <= p0
                while (lo < hi) {
                    const int mid = (lo + hi + 1) >> 1;
                    if (st[mid] <= p0) lo = mid; else hi = mid - 1;
                }
                r = lo;
                v = r & 1;
                uni = st[r + 1] >= p0 + rows;
            }
        }
        const bool all0 = __syncthreads_and(tid >= cols || (uni && v == 0));
        const bool all1 = __syncthreads_and(tid >= cols || (uni && v == 1));
        const bool fast = all0 || all1;
        if (!fast && tid < cols) {
            int sh = (int)(((uintptr_t)dst + (int64_t)y0 * W + x0) & 15);
            const int wm = W & 15;
            for (int y = 0; y < rows; ++r) {
                const int end = r < nc ? (int)min(st[r + 1] - p0, (int64_t)rows) : rows;
                const uint8_t b = r < nc ? (uint8_t)(r & 1) : 0;
                for (; y < end; ++y) {
                    S2D_DEV_ASSERT(y * RD_PITCH + sh + tid < RD_TR * RD_PITCH);
                    tile[y * RD_PITCH + sh + tid] = b;
                    sh = (sh + wm) & 15;
                }
            }
        }
        __syncthreads();
        const uint32_t splat = all1 ? 0x01010101u : 0u;
        for (int q = tid; q < rows * RD_CHUNKS; q += RD_TC) {
            const int y = q / RD_CHUNKS, lo = 16 * (q % RD_CHUNKS);
            uint8_t* const row = dst + (int64_t)(y0 + y) * W + x0;
            const int sh = (int)((uintptr_t)row & 15);
            uint8_t* const al = row - sh;                                  // 16-byte aligned; only [sh, sh + cols) is ours
            const int a = max(lo, sh), b = min(lo + 16, sh + cols);
            if (a >= b) continue;
            S2D_DEV_ASSERT(a - sh >= 0 && b - sh <= cols && (int64_t)(y0 + y) * W + x0 + b - sh <= (int64_t)H * W);
            if (a == lo && b == lo + 16) {
                const uint4 w = fast ? make_uint4(splat, splat, splat, splat)
                                     : *reinterpret_cast<const uint4*>(tile + y * RD_PITCH + lo);
                *reinterpret_cast<uint4*>(al + lo) = w;
            } else {
                for (int i = a; i < b; ++i) al[i] = fast ? (uint8_t)splat : tile[y * RD_PITCH + i];
            }
        }
        __syncthreads();
    }
}

}  // namespace s2d

using namespace s2d;

extern "C" int s2d_rle_from_strings_work_ints(int N, int64_t nchars, int64_t* out) {
    S2D_CHECK_ARG(out && N > 0 && nchars >= 0, "s2d_rle_from_strings_work_ints: bad arguments");
    *out = N;
    return 0;
}

extern "C" int s2d_rle_from_strings(const char* chars, const int64_t* str_offsets, int N, int32_t* work, int64_t capacity,
                                    int32_t* counts, int64_t* count_offsets, int32_t* status, int64_t* needed,
                                    void* stream) {
    S2D_ENTER(stream);
    S2D_CHECK_ARG(chars && str_offsets && work && counts && count_offsets && status && needed,
                  "s2d_rle_from_strings: null pointer");
    S2D_CHECK_ARG(N > 0 && capacity >= 0, "s2d_rle_from_strings: bad sizes");
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned blocks = (unsigned)((N + RP_WARPS - 1) / RP_WARPS);
    rp_count_kernel<<<blocks, RP_WARPS * 32, 0, st>>>(chars, str_offsets, N, work);
    S2D_CHECK_LAUNCH("rp_count_kernel");
    if (const int rc = launch_offsets(work, N, count_offsets, needed, st)) return rc;
    rp_write_kernel<<<blocks, RP_WARPS * 32, 0, st>>>(chars, str_offsets, N, count_offsets, capacity, counts, status);
    S2D_CHECK_LAUNCH("rp_write_kernel");
    return 0;
}

extern "C" int s2d_rle_decode_work_ints(int N, int64_t ncounts, int64_t* out) {
    S2D_CHECK_ARG(out && N > 0 && ncounts >= 0, "s2d_rle_decode_work_ints: bad arguments");
    *out = 2 * (ncounts + N);
    return 0;
}

extern "C" int s2d_rle_decode(const int32_t* counts, const int64_t* count_offsets, int N, const int32_t* heights,
                              const int32_t* widths, const int64_t* out_offsets, int32_t* work, uint8_t* out,
                              int32_t* status, void* stream) {
    S2D_ENTER(stream);
    S2D_CHECK_ARG(counts && count_offsets && heights && widths && out_offsets && work && out && status,
                  "s2d_rle_decode: null pointer");
    S2D_CHECK_ARG(N > 0, "s2d_rle_decode: bad sizes");
    S2D_CHECK_ARG(reinterpret_cast<uintptr_t>(work) % 8 == 0, "s2d_rle_decode: work must be 8-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    int dev = 0, nsm = 148;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) { cudaGetLastError(); nsm = 148; }
    int64_t* starts = reinterpret_cast<int64_t*>(work);
    rd_scan_kernel<<<(unsigned)((N + RD_SCAN_WARPS - 1) / RD_SCAN_WARPS), RD_SCAN_WARPS * 32, 0, st>>>(
        counts, count_offsets, N, heights, widths, starts, status);
    S2D_CHECK_LAUNCH("rd_scan_kernel");
    // about 16 CTAs per SM in all, whatever the number of masks: the sizes are on the device
    const int per_mask = (int)std::max<int64_t>(1, std::min<int64_t>(1024, (int64_t)16 * nsm / N));
    S2D_CHECK_ARG((int64_t)N * per_mask < INT_MAX, "s2d_rle_decode: too many masks");
    rd_tile_kernel<<<(unsigned)(N * per_mask), RD_TC, 0, st>>>(count_offsets, N, heights, widths, out_offsets, starts,
                                                                per_mask, out);
    S2D_CHECK_LAUNCH("rd_tile_kernel");
    return 0;
}
