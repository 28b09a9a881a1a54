// K0 label statistics / object enumeration and K3a visibility reduce + binarise.
// HBM-bound streaming kernels: 128-bit loads, run-length aggregation into warp-private
// shared-memory histograms, one global atomic per (CTA, label).
#include "common.cuh"

namespace s2d {

// ------------------------------------------------------------------------------------------
// K0a: area[frame][256] += histogram of a chunk of the frame's label bytes.
// ------------------------------------------------------------------------------------------
constexpr int LH_THREADS = 256;
constexpr int LH_BYTES_PER_CTA = 64 * 1024;

// bit 7 of every byte of x that is non-zero
__device__ __forceinline__ uint32_t lh_nz7(uint32_t x) { return (((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) & 0x80808080u; }
// number of the 16 bytes of w that equal the byte replicated in s4
__device__ __forceinline__ int lh_count_eq(const int4 w, uint32_t s4) {
    const uint32_t m = (lh_nz7((uint32_t)w.x ^ s4) >> 7) | (lh_nz7((uint32_t)w.y ^ s4) >> 6) |
                       (lh_nz7((uint32_t)w.z ^ s4) >> 5) | (lh_nz7((uint32_t)w.w ^ s4) >> 4);
    return 16 - __popc(m);
}

// Label maps are piecewise constant: a 16-byte vector almost always holds one label (a) or two runs (a ... a z ... z), and
// the 32 vectors a warp reads side by side (512 consecutive pixels) mostly share them. Per warp step, branch-free: every
// lane counts the bytes equal to its first (a) and to its last (z) byte; the lanes whose a equals lane 0's are summed with
// one warp reduction and added by lane 0, the others add their own count, z likewise when the vector is not uniform.
// Only a vector with three or more labels (c_a + c_z < 16, rare) is counted byte by byte. The round-1 kernel kept a
// per-thread run and took a divergent per-byte path in every warp step that met an object border (ncu: 0.55 of HBM).
__global__ void __launch_bounds__(LH_THREADS)
label_hist_kernel(const s2d_video_desc* __restrict__ descs, int32_t* __restrict__ area) {
    const s2d_video_desc d = descs[blockIdx.z];
    const int t = blockIdx.y;
    if (t >= d.T) return;
    const int64_t npix = (int64_t)d.H * d.W;
    const int64_t beg = (int64_t)blockIdx.x * LH_BYTES_PER_CTA;
    if (beg >= npix) return;
    const int64_t end = min(npix, beg + (int64_t)LH_BYTES_PER_CTA);

    __shared__ int wh[LH_THREADS / 32][S2D_MAX_LABELS];
    for (int i = threadIdx.x; i < (LH_THREADS / 32) * S2D_MAX_LABELS; i += LH_THREADS) (&wh[0][0])[i] = 0;
    __syncthreads();
    int* mywh = wh[threadIdx.x >> 5];
    const int lane = threadIdx.x & 31;

    const uint8_t* base = d.labels + (int64_t)t * npix;
    // head / tail: bytes outside the 16-byte aligned body (thread 0 of the CTA; at most 15 each)
    const uintptr_t addr0 = (uintptr_t)(base + beg);
    const int64_t head = min((int64_t)((16 - (addr0 & 15)) & 15), end - beg);
    const int64_t vbeg = beg + head;
    const int64_t nvec = (end - vbeg) / 16;
    if (threadIdx.x == 0) {
        for (int64_t i = beg; i < vbeg; ++i) atomicAdd(&mywh[base[i]], 1);
        for (int64_t i = vbeg + nvec * 16; i < end; ++i) atomicAdd(&mywh[base[i]], 1);
    }
    const int4* vp = reinterpret_cast<const int4*>(base + vbeg);
    S2D_DEV_ASSERT(vbeg + nvec * 16 <= end && end <= npix);
    auto eat = [&](const int4 w, bool valid) {                 // warp-uniform call; `valid` false: the lane has no vector
        const uint32_t a = (uint32_t)w.x & 255u, z = (uint32_t)w.w >> 24;
        const int ca = valid ? lh_count_eq(w, a * 0x01010101u) : 0;
        const int cz = (valid && z != a) ? lh_count_eq(w, z * 0x01010101u) : 0;
        const uint32_t a0 = __shfl_sync(0xffffffffu, a, 0);
        const int sa = __reduce_add_sync(0xffffffffu, a == a0 ? ca : 0);
        if (lane == 0) atomicAdd(&mywh[a0], sa);
        else if (a != a0 && ca) atomicAdd(&mywh[a], ca);
        if (cz) atomicAdd(&mywh[z], cz);
        if (__any_sync(0xffffffffu, valid && ca + cz != 16)) {     // three or more labels in 16 pixels: byte by byte
            if (valid && ca + cz != 16) {
                const uint32_t ws[4] = {(uint32_t)w.x, (uint32_t)w.y, (uint32_t)w.z, (uint32_t)w.w};
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    const uint32_t v = (ws[k >> 2] >> (8 * (k & 3))) & 255u;
                    if (v != a && v != z) atomicAdd(&mywh[v], 1);
                }
            }
        }
    };
    // four independent 128-bit streaming loads in flight per thread
    const int64_t nfull = nvec - nvec % (4 * LH_THREADS);
    int64_t i = threadIdx.x;
    for (; i < nfull; i += 4 * LH_THREADS) {
        const int4 w0 = ld_stream(vp + i), w1 = ld_stream(vp + i + LH_THREADS);
        const int4 w2 = ld_stream(vp + i + 2 * LH_THREADS), w3 = ld_stream(vp + i + 3 * LH_THREADS);
        eat(w0, true); eat(w1, true); eat(w2, true); eat(w3, true);
    }
    for (int64_t j = nfull + (threadIdx.x & ~31); j < nvec; j += LH_THREADS) {       // warp-uniform trip count
        const bool valid = j + lane < nvec;
        eat(valid ? ld_stream(vp + j + lane) : make_int4(0, 0, 0, 0), valid);
    }
    __syncthreads();
    int32_t* out = area + (d.frame0 + t) * S2D_MAX_LABELS;
    for (int l = threadIdx.x; l < S2D_MAX_LABELS; l += LH_THREADS) {
        int s = 0;
#pragma unroll
        for (int w = 0; w < LH_THREADS / 32; ++w) s += wh[w][l];
        if (s) atomicAdd(&out[l], s);
    }
}

// ------------------------------------------------------------------------------------------
// K0b: object enumeration. One CTA (8 warps) per video. The only sequential quantity is the first global id of a
// frame (a prefix sum of the frames' object counts): pass 1 counts the objects of every frame (a warp per frame,
// lane = 8 labels, eight ballots), a block scan turns the counts into first ids, pass 2 writes the tables - the
// frames' loads are independent, so the kernel costs a few global-memory latencies instead of one per frame.
// ------------------------------------------------------------------------------------------
constexpr int FT_MAX_T = 1024;            // frames per video (s2d_windows has the same limit)

__device__ __forceinline__ void ft_presence(const int32_t* __restrict__ arow, int lane, uint32_t (&pres)[8]) {
    int a[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = arow[k * 32 + lane];          // label k * 32 + lane
#pragma unroll
    for (int k = 0; k < 8; ++k) pres[k] = __ballot_sync(0xffffffffu, a[k] > 0);
}

__global__ void __launch_bounds__(S2D_MAX_LABELS)
frame_tables_kernel(const s2d_video_desc* __restrict__ descs, const int32_t* __restrict__ area,
                    int32_t* __restrict__ gid_of, int32_t* __restrict__ frameinfo,
                    int32_t* __restrict__ qframe, int32_t* __restrict__ qlabel,
                    int32_t* __restrict__ vidinfo) {
    const s2d_video_desc d = descs[blockIdx.x];
    __shared__ int first[FT_MAX_T + 1];
    __shared__ int wsum[S2D_MAX_LABELS / 32];
    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
    const int T = min(d.T, FT_MAX_T);
    // pass 1: objects per frame (present labels minus the smallest one)
    for (int t = w; t < T; t += 8) {
        uint32_t pres[8];
        ft_presence(area + (d.frame0 + t) * S2D_MAX_LABELS, lane, pres);
        int total = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) total += __popc(pres[k]);
        if (lane == 0) first[t] = total > 0 ? total - 1 : 0;
    }
    __syncthreads();
    // exclusive scan of first[0..T) (T <= 1024: four values per thread)
    int v[4], s = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) { const int t = tid * 4 + k; v[k] = t < T ? first[t] : 0; s += v[k]; }
    int total_obj;
    int run = block_excl_scan<S2D_MAX_LABELS>(s, wsum, total_obj);
#pragma unroll
    for (int k = 0; k < 4; ++k) { const int t = tid * 4 + k; if (t < T) first[t] = run; run += v[k]; }
    __syncthreads();
    // pass 2: tables
    for (int t = w; t < T; t += 8) {
        const int64_t f = d.frame0 + t;
        uint32_t pres[8];
        ft_presence(area + f * S2D_MAX_LABELS, lane, pres);
        int total = 0, minlab = -1;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if (minlab < 0 && pres[k]) minlab = k * 32 + __ffs(pres[k]) - 1;
            total += __popc(pres[k]);
        }
        const int gid_base = first[t];
        int below = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int l = k * 32 + lane;
            const bool p = (pres[k] >> lane) & 1u;
            int gid = -1;
            if (p && l != minlab) {
                gid = gid_base + below + __popc(pres[k] & ((1u << lane) - 1u)) - 1;
                S2D_DEV_ASSERT(gid >= 0);
                if (gid < d.Nm) {
                    qframe[d.row0 + gid] = t;
                    qlabel[d.row0 + gid] = l;
                }
            }
            gid_of[f * S2D_MAX_LABELS + l] = gid;
            below += __popc(pres[k]);
        }
        if (lane == 0) reinterpret_cast<int4*>(frameinfo)[f] = make_int4(total > 0 ? total - 1 : 0, gid_base, minlab, total);
    }
    if (tid == 0) vidinfo[blockIdx.x * S2D_VIDINFO_WORDS + 5] = total_obj;
}

// ------------------------------------------------------------------------------------------
// K3a: visibility reduce. One warp per (row, frame): popcount of nonzero flag bytes.
// ------------------------------------------------------------------------------------------
constexpr int VR_WARPS = 8;

__global__ void __launch_bounds__(VR_WARPS * 32)
vis_reduce_kernel(const s2d_video_desc* __restrict__ descs, int32_t* __restrict__ cnt_out,
                  float* __restrict__ V) {
    const s2d_video_desc d = descs[blockIdx.y];
    const int64_t rt = (int64_t)blockIdx.x * VR_WARPS + (threadIdx.x >> 5);
    if (rt >= (int64_t)d.Nm * d.T) return;
    const int lane = threadIdx.x & 31;
    const int q = (int)(rt / d.T);
    const int n = d.npts ? min(max(d.npts[q], 0), d.P) : d.P;
    const uint8_t* row = d.vis + rt * d.P;
    int c = 0;
    if (d.flags & S2D_DESC_VIS_BITS) {
        // bit-packed flags: ceil(P / 32) words per row, only the first n bits count
        const int pw = (d.P + 31) >> 5;
        const uint32_t* wrow = reinterpret_cast<const uint32_t*>(d.vis) + rt * pw;
        const int nfull = n >> 5;                                   // whole words
        if ((pw & 3) == 0 && (((uintptr_t)wrow) & 15) == 0) {
            const int4* vp = reinterpret_cast<const int4*>(wrow);
            for (int i = lane; i < (nfull >> 2); i += 32) {
                const int4 a = ld_stream(vp + i);
                c += __popc((uint32_t)a.x) + __popc((uint32_t)a.y) + __popc((uint32_t)a.z) + __popc((uint32_t)a.w);
            }
            for (int i = (nfull & ~3) + lane; i < nfull; i += 32) c += __popc(wrow[i]);
        } else {
            for (int i = lane; i < nfull; i += 32) c += __popc(wrow[i]);
        }
        if (lane == 0 && (n & 31)) c += __popc(wrow[nfull] & ((1u << (n & 31)) - 1u));
    } else if (n == d.P && (d.P & 15) == 0 && (((uintptr_t)row) & 15) == 0) {
        const int4* vp = reinterpret_cast<const int4*>(row);
        const int nv = d.P >> 4;
        int i = lane;
        // two independent 128-bit loads in flight per lane
        for (; i + 32 < nv; i += 64) {
            int4 a = ld_stream(vp + i), b = ld_stream(vp + i + 32);
            c += __popc(__vsetne4((uint32_t)a.x, 0u)) + __popc(__vsetne4((uint32_t)a.y, 0u)) +
                 __popc(__vsetne4((uint32_t)a.z, 0u)) + __popc(__vsetne4((uint32_t)a.w, 0u));
            c += __popc(__vsetne4((uint32_t)b.x, 0u)) + __popc(__vsetne4((uint32_t)b.y, 0u)) +
                 __popc(__vsetne4((uint32_t)b.z, 0u)) + __popc(__vsetne4((uint32_t)b.w, 0u));
        }
        for (; i < nv; i += 32) {
            int4 a = ld_stream(vp + i);
            c += __popc(__vsetne4((uint32_t)a.x, 0u)) + __popc(__vsetne4((uint32_t)a.y, 0u)) +
                 __popc(__vsetne4((uint32_t)a.z, 0u)) + __popc(__vsetne4((uint32_t)a.w, 0u));
        }
    } else {
        for (int i = lane; i < n; i += 32) c += row[i] != 0;
    }
    c = warp_sum(c);
    if (lane == 0) {
        cnt_out[d.vt_off + rt] = c;
        // torch.mean(bool.float()) on CPU == float32(cnt) / float32(P), IEEE division; 0/0 = NaN
        V[d.vt_off + rt] = __fdiv_rn((float)c, (float)n);
    }
}

// K3 binarise: one thread per (row, word of 32 frames).
__global__ void binarize_kernel(const s2d_video_desc* __restrict__ descs, const float* __restrict__ V,
                                float thr, uint32_t* __restrict__ xbits) {
    const s2d_video_desc d = descs[blockIdx.y];
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)d.Nm * d.TW) return;
    const int q = (int)(i / d.TW), w = (int)(i % d.TW);
    const float* v = V + d.vt_off + (int64_t)q * d.T;
    uint32_t m = 0;
    for (int b = 0; b < 32; ++b) {
        const int t = w * 32 + b;
        if (t < d.T && v[t] > thr) m |= 1u << b;   // NaN compares false
    }
    xbits[d.xbits_off + i] = m;
}

}  // namespace s2d

using namespace s2d;

extern "C" int s2d_label_stats(const s2d_video_desc* descs, int nvideos, int max_T, int64_t max_npix,
                               int64_t total_frames, int32_t* area,
                               int32_t* gid_of, int32_t* frameinfo, int32_t* qframe, int32_t* qlabel,
                               int32_t* vidinfo, void* stream) {
    S2D_ENTER(stream);
    S2D_CHECK_ARG(descs && area && gid_of && frameinfo && qframe && qlabel && vidinfo,
                  "s2d_label_stats: null pointer");
    S2D_CHECK_ARG(nvideos > 0 && nvideos <= 65535 && max_T > 0 && max_T <= FT_MAX_T && max_npix > 0,
                  "s2d_label_stats: bad sizes nvideos=%d max_T=%d (videos of up to %d frames)", nvideos, max_T, FT_MAX_T);
    cudaStream_t st = (cudaStream_t)stream;
    cudaMemsetAsync(area, 0, (size_t)total_frames * S2D_MAX_LABELS * sizeof(int32_t), st);
    dim3 grid((unsigned)((max_npix + LH_BYTES_PER_CTA - 1) / LH_BYTES_PER_CTA), max_T, nvideos);
    label_hist_kernel<<<grid, LH_THREADS, 0, st>>>(descs, area);
    S2D_CHECK_LAUNCH("label_hist_kernel");
    frame_tables_kernel<<<nvideos, S2D_MAX_LABELS, 0, st>>>(descs, area, gid_of, frameinfo, qframe, qlabel, vidinfo);
    S2D_CHECK_LAUNCH("frame_tables_kernel");
    return 0;
}

extern "C" int s2d_vis_reduce(const s2d_video_desc* descs, int nvideos, int64_t max_rows_x_T,
                              int32_t* cnt, float* V, void* stream) {
    S2D_ENTER(stream);
    S2D_CHECK_ARG(descs && cnt && V, "s2d_vis_reduce: null pointer");
    S2D_CHECK_ARG(nvideos > 0 && nvideos <= 65535 && max_rows_x_T > 0, "s2d_vis_reduce: bad sizes");
    dim3 grid((unsigned)((max_rows_x_T + VR_WARPS - 1) / VR_WARPS), nvideos);
    vis_reduce_kernel<<<grid, VR_WARPS * 32, 0, (cudaStream_t)stream>>>(descs, cnt, V);
    S2D_CHECK_LAUNCH("vis_reduce_kernel");
    return 0;
}

extern "C" int s2d_binarize(const s2d_video_desc* descs, int nvideos, int64_t max_rows_x_TW,
                            const float* V, float visibility_threshold, uint32_t* xbits, void* stream) {
    S2D_ENTER(stream);
    S2D_CHECK_ARG(descs && V && xbits, "s2d_binarize: null pointer");
    S2D_CHECK_ARG(nvideos > 0 && nvideos <= 65535 && max_rows_x_TW > 0, "s2d_binarize: bad sizes");
    dim3 grid((unsigned)((max_rows_x_TW + 255) / 256), nvideos);
    binarize_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(descs, V, visibility_threshold, xbits);
    S2D_CHECK_LAUNCH("binarize_kernel");
    return 0;
}
