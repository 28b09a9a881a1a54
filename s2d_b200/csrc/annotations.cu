// Stage E's annotation layout on the device: which keymask rows become which YTVIS annotation, in the reference's
// order (annotations.py:8-140 walks `cluster_*` / `group_*` directories sorted as strings), packed into compact
// tables that a host copies back and slices into json objects without any per-row decision of its own.
//
//   al_sort_kernel   CTA per video: candidate clusters and their order, one 64-bit key per grouped row of a candidate
//                    cluster (cluster rank | decimal-string key of the group label | frame | label), bitonic sort of
//                    the keys (shared memory, or the video's slice of `work` for videos of many rows), counts
//   al_scan_kernel   one CTA: exclusive prefix of the per-video counts -> where each video's entries go, totals
//   al_write_kernel  CTA per video: annotation, member, cluster and range tables at the video's place; the members'
//                    strings gathered back to back
// Annotation a owns the sorted keys of one (cluster, group); of the keys of one frame, the last (largest label id)
// is the member. Nothing is written at or past `capacity` in `chars`.
#include "common.cuh"

namespace s2d {

constexpr int AL_THREADS = 1024;
constexpr int AL_SMEM_KEYS = 4096;             // videos of at most this many rows sort in shared memory
constexpr int AL_NCOUNT = 5;                   // per video: annotations, members, string bytes, clusters, range pairs
constexpr int AL_VWORDS = AL_NCOUNT + 1;       // ... and the number of sort keys
constexpr int AL_CLW = 3 * S2D_MAX_CLUSTERS;   // per video and cluster rank: cluster id, runs, annotated
constexpr uint64_t AL_PAD = ~0ull;

// Key that orders non-negative integers as their decimal strings order (Python's sorted() of "group_{l}"): the digits
// zero-padded on the right to 10, ties (one string a prefix of the other followed by zeros only) broken by length.
// < 2^38 for every int32.
__host__ __device__ inline uint64_t al_decimal_key(uint32_t x) {
    int d = 1;
    uint64_t p = 10, v = x;
    while (d < 10 && x >= p) { ++d; p *= 10; }
    for (int i = d; i < 10; ++i) v *= 10;
    return v * 16 + d;
}

// cluster rank (4 bits) | al_decimal_key(group label) (38) | frame (10) | label (8)
__device__ __forceinline__ uint64_t al_key(int rank, int group, int frame, int label) {
    return (uint64_t)rank << 56 | al_decimal_key((uint32_t)group) << 18 | (uint64_t)frame << 8 | (uint64_t)label;
}
__device__ __forceinline__ bool al_same_group(uint64_t a, uint64_t b) { return (a >> 18) == (b >> 18); }
__device__ __forceinline__ bool al_same_frame(uint64_t a, uint64_t b) { return (a >> 8) == (b >> 8); }

// set bits below T of a cluster's run-start (run-end) row
__device__ __forceinline__ uint32_t al_word(const uint32_t* row, int w, int T) {
    const int valid = T - 32 * w;
    return valid >= 32 ? row[w] : row[w] & ((1u << valid) - 1u);
}

__global__ void __launch_bounds__(AL_THREADS)
al_sort_kernel(const s2d_video_desc* __restrict__ descs, const int32_t* __restrict__ vidinfo,
               const int4* __restrict__ rowinfo, const uint32_t* __restrict__ winbits, const uint32_t* __restrict__ rsbits,
               const uint32_t* __restrict__ rebits, const int32_t* __restrict__ glabel, const int32_t* __restrict__ qframe,
               const int32_t* __restrict__ qlabel, const int32_t* __restrict__ gid_of, const int64_t* __restrict__ str_off,
               uint64_t* keys_work, int64_t* __restrict__ vcnt, int32_t* __restrict__ clw) {
    __shared__ uint64_t skeys[AL_SMEM_KEYS];
    __shared__ int nruns[S2D_MAX_CLUSTERS], cand[S2D_MAX_CLUSTERS], rank_of[S2D_MAX_CLUSTERS], annotated[S2D_MAX_CLUSTERS];
    __shared__ int nkeys, n_ann, n_mem;
    __shared__ unsigned long long n_chars;
    const int v = blockIdx.x, tid = threadIdx.x;
    const s2d_video_desc d = descs[v];
    int64_t* cnt = vcnt + (int64_t)v * AL_VWORDS;
    int32_t* cl = clw + (int64_t)v * AL_CLW;
    if (vidinfo[v * S2D_VIDINFO_WORDS + 3] != 1) {                      // the reference annotates status-1 videos only
        if (tid < AL_VWORDS) cnt[tid] = 0;
        return;
    }
    const int Nm = d.Nm, T = d.T, TW = d.TW;
    const int kc = max(0, min(vidinfo[v * S2D_VIDINFO_WORDS + 0], min(S2D_MAX_CLUSTERS, Nm)));
    // runs of cluster c: decode() pairs the set bits of rsbits and rebits (row c of the video's [Nm][TW] arrays)
    if (tid < S2D_MAX_CLUSTERS) {
        int ns = 0, ne = 0;
        if (tid < kc) {
            const uint32_t* rs = rsbits + d.xbits_off + (int64_t)tid * TW;
            const uint32_t* re = rebits + d.xbits_off + (int64_t)tid * TW;
            for (int w = 0; w < TW; ++w) { ns += __popc(al_word(rs, w, T)); ne += __popc(al_word(re, w, T)); }
        }
        nruns[tid] = min(ns, ne);
        cand[tid] = 0;
        annotated[tid] = 0;
    }
    if (tid == 0) { nkeys = 0; n_ann = 0; n_mem = 0; n_chars = 0; }
    __syncthreads();
    // a cluster counts when one of its rows is the candidate of run r: rowinfo.y == r and winner bit r set
    for (int q = tid; q < Nm; q += AL_THREADS) {
        const int4 ri = rowinfo[d.row0 + q];
        if (ri.x >= 0 && ri.x < kc && ri.y >= 0 && ri.y < nruns[ri.x] &&
            ((winbits[d.xbits_off + (int64_t)q * TW + (ri.y >> 5)] >> (ri.y & 31)) & 1u))
            cand[ri.x] = 1;
    }
    __syncthreads();
    // candidate clusters in the order of the strings cluster_{c}
    if (tid < kc && cand[tid]) {
        int r = 0;
        for (int c = 0; c < kc; ++c) r += cand[c] && al_decimal_key(c) < al_decimal_key(tid);
        rank_of[tid] = r;
        cl[r] = tid;
        cl[S2D_MAX_CLUSTERS + r] = nruns[tid];
    }
    __syncthreads();
    // one key per grouped row of a candidate cluster
    uint64_t* keys = Nm <= AL_SMEM_KEYS ? skeys : keys_work + 2 * d.row0;
    for (int q = tid; q < Nm; q += AL_THREADS) {
        const int c = rowinfo[d.row0 + q].x, l = glabel[d.row0 + q];
        if (c >= 0 && c < kc && cand[c] && l >= 0) {
            const int f = qframe[d.row0 + q], m = qlabel[d.row0 + q];
            S2D_DEV_ASSERT(l < Nm && f >= 0 && f < T && m >= 0 && m < S2D_MAX_LABELS);
            keys[atomicAdd(&nkeys, 1)] = al_key(rank_of[c], l, f, m);
        }
    }
    __syncthreads();
    const int n = nkeys;
    int N = 1;
    while (N < n) N <<= 1;
    S2D_DEV_ASSERT(Nm <= AL_SMEM_KEYS ? N <= AL_SMEM_KEYS : N <= 2 * Nm);
    for (int i = n + tid; i < N; i += AL_THREADS) keys[i] = AL_PAD;
    __syncthreads();
    for (int k = 2; k <= N; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = tid; i < N; i += AL_THREADS) {
                const int p = i ^ j;
                if (p > i) {
                    const uint64_t a = keys[i], b = keys[p];
                    if ((a > b) == ((i & k) == 0)) { keys[i] = b; keys[p] = a; }
                }
            }
            __syncthreads();
        }
    }
    // counts: a (cluster, group) per annotation, the last key of each of its frames per member
    int my_ann = 0, my_mem = 0;
    long long my_chars = 0;
    for (int j = tid; j < n; j += AL_THREADS) {
        const uint64_t key = keys[j];
        if (j == 0 || !al_same_group(keys[j - 1], key)) {
            ++my_ann;
            annotated[key >> 56] = 1;
        }
        if (j == n - 1 || !al_same_frame(keys[j + 1], key)) {
            const int f = (int)((key >> 8) & 1023), m = (int)(key & 255);
            const int g = gid_of[(d.frame0 + f) * S2D_MAX_LABELS + m];
            S2D_DEV_ASSERT(g >= 0 && g < Nm);
            ++my_mem;
            my_chars += str_off[d.row0 + g + 1] - str_off[d.row0 + g];
        }
        if (Nm > AL_SMEM_KEYS) continue;
        keys_work[2 * d.row0 + j] = key;                                  // al_write_kernel reads the sorted keys here
    }
    my_ann = warp_sum(my_ann);
    my_mem = warp_sum(my_mem);
    for (int o = 16; o > 0; o >>= 1) my_chars += __shfl_xor_sync(0xffffffffu, my_chars, o);
    if ((tid & 31) == 0) {
        atomicAdd(&n_ann, my_ann);
        atomicAdd(&n_mem, my_mem);
        atomicAdd(&n_chars, (unsigned long long)my_chars);
    }
    __syncthreads();
    if (tid == 0) {
        int ncl = 0, npairs = 0;
        for (int r = 0; r < S2D_MAX_CLUSTERS; ++r) {
            cl[2 * S2D_MAX_CLUSTERS + r] = annotated[r];
            if (annotated[r]) { ++ncl; npairs += cl[S2D_MAX_CLUSTERS + r]; }
        }
        cnt[0] = n_ann; cnt[1] = n_mem; cnt[2] = (int64_t)n_chars; cnt[3] = ncl; cnt[4] = npairs; cnt[5] = n;
    }
}

// exclusive prefix over videos of each count -> vfirst [nvideos][AL_NCOUNT], totals -> sizes; vann[v] = (count, first)
__global__ void __launch_bounds__(AL_THREADS)
al_scan_kernel(int nvideos, const int64_t* __restrict__ vcnt, int64_t* __restrict__ vfirst, int32_t* __restrict__ vann,
               int64_t* __restrict__ sizes) {
    __shared__ int64_t wsum[AL_THREADS / 32];
    for (int q = 0; q < AL_NCOUNT; ++q) {
        int64_t carry = 0;
        for (int base = 0; base < nvideos; base += AL_THREADS) {
            const int v = base + threadIdx.x;
            const int64_t x = v < nvideos ? vcnt[(int64_t)v * AL_VWORDS + q] : 0;
            int64_t tot;
            const int64_t ex = block_excl_scan<AL_THREADS>(x, wsum, tot);
            if (v < nvideos) {
                vfirst[(int64_t)v * AL_NCOUNT + q] = carry + ex;
                if (q == 0) { vann[2 * v] = (int32_t)x; vann[2 * v + 1] = (int32_t)(carry + ex); }
            }
            carry += tot;
        }
        if (threadIdx.x == 0) sizes[q] = carry;
    }
}

__global__ void __launch_bounds__(AL_THREADS)
al_write_kernel(const s2d_video_desc* __restrict__ descs, const int32_t* __restrict__ vidinfo,
                const uint32_t* __restrict__ rsbits, const uint32_t* __restrict__ rebits, const int32_t* __restrict__ glabel,
                const int32_t* __restrict__ grp_n, const int32_t* __restrict__ grp_one2x, const int32_t* __restrict__ area,
                const int32_t* __restrict__ gid_of, const int32_t* __restrict__ rle_bbox, const int64_t* __restrict__ str_off,
                const char* __restrict__ rle_chars, int64_t nchars, const uint64_t* __restrict__ keys_work,
                const int64_t* __restrict__ vcnt, const int64_t* __restrict__ vfirst, const int32_t* __restrict__ clw,
                int32_t* __restrict__ ann, int32_t* __restrict__ members, int64_t* __restrict__ member_off,
                int32_t* __restrict__ clusters, int32_t* __restrict__ pairs, int64_t capacity, char* __restrict__ chars) {
    __shared__ int64_t wsum[AL_THREADS / 32];
    __shared__ int cl_index[S2D_MAX_CLUSTERS];
    __shared__ int64_t s_src[AL_THREADS], s_dst[AL_THREADS];
    __shared__ int s_len[AL_THREADS];
    const int v = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (vidinfo[v * S2D_VIDINFO_WORDS + 3] != 1) return;
    const s2d_video_desc d = descs[v];
    const int Nm = d.Nm, T = d.T, TW = d.TW;
    const int n = (int)vcnt[(int64_t)v * AL_VWORDS + 5];
    const int64_t* first = vfirst + (int64_t)v * AL_NCOUNT;
    const int64_t A0 = first[0], M0 = first[1], C0 = first[2], CL0 = first[3], P0 = first[4];
    const int n_ann = (int)vcnt[(int64_t)v * AL_VWORDS + 0], n_mem = (int)vcnt[(int64_t)v * AL_VWORDS + 1];
    const int32_t* cl = clw + (int64_t)v * AL_CLW;
    // annotated clusters in rank order: their range lists
    if (tid < S2D_MAX_CLUSTERS) {
        int i = 0, p = 0;
        for (int r = 0; r < tid; ++r) if (cl[2 * S2D_MAX_CLUSTERS + r]) { ++i; p += cl[S2D_MAX_CLUSTERS + r]; }
        cl_index[tid] = (int)CL0 + i;
        if (cl[2 * S2D_MAX_CLUSTERS + tid]) {
            const int c = cl[tid], nr = cl[S2D_MAX_CLUSTERS + tid];
            int32_t* ci = clusters + 2 * (CL0 + i);
            ci[0] = (int32_t)(P0 + p);
            ci[1] = nr;
            int32_t* pr = pairs + 2 * (P0 + p);
            for (int e = 0; e < 2; ++e) {                                  // i-th set bit of run starts / ends
                const uint32_t* row = (e ? rebits : rsbits) + d.xbits_off + (int64_t)c * TW;
                int k = 0;
                for (int w = 0; w < TW && k < nr; ++w) {
                    for (uint32_t m = al_word(row, w, T); m && k < nr; m &= m - 1) pr[2 * k++ + e] = 32 * w + __ffs(m) - 1;
                }
            }
        }
    }
    __syncthreads();
    const uint64_t* keys = keys_work + 2 * d.row0;
    int64_t ann_carry = 0, mem_carry = 0, chr_carry = 0;
    for (int base = 0; base < n; base += AL_THREADS) {
        const int j = base + tid;
        const bool in = j < n;
        const uint64_t key = in ? keys[j] : 0;
        const bool gs = in && (j == 0 || !al_same_group(keys[j - 1], key));
        const bool mem = in && (j == n - 1 || !al_same_frame(keys[j + 1], key));
        const int f = (int)((key >> 8) & 1023), m = (int)(key & 255);
        const int64_t fl = (d.frame0 + f) * S2D_MAX_LABELS + m;
        const int g = in ? gid_of[fl] : 0;
        S2D_DEV_ASSERT(!in || (g >= 0 && g < Nm));
        const int64_t r = d.row0 + g;
        const int64_t src = in ? str_off[r] : 0;
        const int len = mem ? (int)(str_off[r + 1] - src) : 0;
        int64_t tot_a, tot_m, tot_c;
        const int64_t ea = block_excl_scan<AL_THREADS, int64_t>(gs, wsum, tot_a);
        const int64_t em = block_excl_scan<AL_THREADS, int64_t>(mem, wsum, tot_m);
        const int64_t ec = block_excl_scan<AL_THREADS, int64_t>(len, wsum, tot_c);
        const int64_t mi = M0 + mem_carry + em, dst = C0 + chr_carry + ec;
        if (gs) {
            const int rank = (int)(key >> 56), c = cl[rank], l = glabel[r];
            S2D_DEV_ASSERT(l >= 0 && l < Nm && A0 + ann_carry + ea < A0 + n_ann);
            const int64_t slot = 16 * d.row0 + (int64_t)c * Nm + l;
            int32_t* a = ann + 7 * (A0 + ann_carry + ea);
            a[0] = c; a[1] = l; a[2] = grp_n[slot]; a[3] = grp_one2x[slot]; a[4] = cl_index[rank]; a[5] = (int32_t)mi;
        }
        if (mem) {
            S2D_DEV_ASSERT(mi < M0 + n_mem);
            int32_t* me = members + 6 * mi;
            me[0] = f;
            me[1] = rle_bbox[4 * r]; me[2] = rle_bbox[4 * r + 1]; me[3] = rle_bbox[4 * r + 2]; me[4] = rle_bbox[4 * r + 3];
            me[5] = area[fl];
            member_off[mi] = dst;
        }
        s_src[tid] = src;
        s_dst[tid] = dst;
        s_len[tid] = len;
        __syncthreads();
        // string gather: a warp per member, bytes that lie outside either buffer are skipped (the caller re-runs
        // stage E and this call when a stage-E capacity was short)
        for (int i = warp; i < AL_THREADS; i += AL_THREADS / 32) {
            const int nb = s_len[i];
            if (nb == 0) continue;
            const int64_t s0 = s_src[i], d0 = s_dst[i];
            if (s0 < 0 || s0 + nb > nchars || d0 + nb > capacity) continue;
            const char* sp = rle_chars + s0;
            char* dp = chars + d0;
            int b = lane;
            for (; b + 96 < nb; b += 128) {
                const char c0 = sp[b], c1 = sp[b + 32], c2 = sp[b + 64], c3 = sp[b + 96];
                dp[b] = c0; dp[b + 32] = c1; dp[b + 64] = c2; dp[b + 96] = c3;
            }
            for (; b < nb; b += 32) dp[b] = sp[b];
        }
        ann_carry += tot_a; mem_carry += tot_m; chr_carry += tot_c;
        __syncthreads();
    }
    // member count of each annotation: up to the next annotation's first member
    for (int a = tid; a < n_ann; a += AL_THREADS) {
        int32_t* an = ann + 7 * (A0 + a);
        const int64_t next = a + 1 < n_ann ? (int64_t)an[7 + 5] : M0 + n_mem;
        an[6] = (int32_t)(next - an[5]);
    }
}

}  // namespace s2d

using namespace s2d;

extern "C" int s2d_annotation_layout_work_ints(int64_t total_rows, int nvideos, int64_t* out) {
    S2D_CHECK_ARG(out && total_rows >= 0 && nvideos > 0, "s2d_annotation_layout_work_ints: bad arguments");
    *out = 2 * (2 * total_rows + (int64_t)(AL_VWORDS + AL_NCOUNT) * nvideos) + (int64_t)AL_CLW * nvideos;
    return 0;
}

extern "C" int s2d_annotation_layout(const s2d_video_desc* descs, int nvideos, int64_t total_rows, const int32_t* vidinfo,
                                     const int32_t* rowinfo, const uint32_t* winbits, const uint32_t* rsbits,
                                     const uint32_t* rebits, const int32_t* glabel, const int32_t* qframe,
                                     const int32_t* qlabel, const int32_t* grp_n, const int32_t* grp_one2x,
                                     const int32_t* area, const int32_t* gid_of, const int32_t* rle_bbox,
                                     const int64_t* str_off, const char* rle_chars, int64_t nchars, int32_t* work,
                                     int32_t* vann, int32_t* ann, int32_t* members, int64_t* member_off,
                                     int32_t* clusters, int32_t* pairs, int64_t capacity, char* chars, int64_t* sizes,
                                     void* stream) {
    S2D_ENTER(stream);
    S2D_CHECK_ARG(descs && vidinfo && rowinfo && winbits && rsbits && rebits && glabel && qframe && qlabel && grp_n &&
                      grp_one2x && area && gid_of && rle_bbox && str_off && rle_chars && work && vann && ann && members &&
                      member_off && clusters && pairs && chars && sizes,
                  "s2d_annotation_layout: null pointer");
    S2D_CHECK_ARG(nvideos > 0 && nvideos <= 65535 && total_rows > 0 && nchars >= 0 && capacity >= 0,
                  "s2d_annotation_layout: bad sizes");
    S2D_CHECK_ARG(reinterpret_cast<uintptr_t>(work) % 8 == 0, "s2d_annotation_layout: work must be 8-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    uint64_t* keys = reinterpret_cast<uint64_t*>(work);
    int64_t* vcnt = reinterpret_cast<int64_t*>(keys + 2 * total_rows);
    int64_t* vfirst = vcnt + (int64_t)AL_VWORDS * nvideos;
    int32_t* clw = reinterpret_cast<int32_t*>(vfirst + (int64_t)AL_NCOUNT * nvideos);
    al_sort_kernel<<<nvideos, AL_THREADS, 0, st>>>(descs, vidinfo, reinterpret_cast<const int4*>(rowinfo), winbits, rsbits,
                                                   rebits, glabel, qframe, qlabel, gid_of, str_off, keys, vcnt, clw);
    S2D_CHECK_LAUNCH("al_sort_kernel");
    al_scan_kernel<<<1, AL_THREADS, 0, st>>>(nvideos, vcnt, vfirst, vann, sizes);
    S2D_CHECK_LAUNCH("al_scan_kernel");
    al_write_kernel<<<nvideos, AL_THREADS, 0, st>>>(descs, vidinfo, rsbits, rebits, glabel, grp_n, grp_one2x, area, gid_of,
                                                    rle_bbox, str_off, rle_chars, nchars, keys, vcnt, vfirst, clw, ann,
                                                    members, member_off, clusters, pairs, capacity, chars);
    S2D_CHECK_LAUNCH("al_write_kernel");
    return 0;
}
