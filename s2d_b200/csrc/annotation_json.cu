// Stage E's last layer on the device: the exact text of each video's YTVIS `annotations` list, byte for byte what
// `json.dumps(annotations_from_layout(...)[v])` prints, serialised from the tables of s2d_annotation_layout. The host
// only wraps the bytes in the file's `videos` / `categories` envelope.
//
//   aj_text_kernel<false>  warp per annotation: exact byte length of its text (+ 2 for the ", " or brackets around it)
//   aj_scan_kernel         one CTA: exclusive prefix of the annotation lengths, then per video its length (0 for a
//                          status other than 1, "[]" for a status-1 video without annotation) -> video_off, needed
//   aj_text_kernel<true>   warp per annotation: the text at video_off[v] + 1 + its offset in the video, with "[" before
//                          the first annotation of a video and ", " or "]" after each
// Both passes run the same emitter, so the lengths of pass 1 are the bytes of pass 2. Nothing is written at or past
// `capacity`, and nothing of the layout's strings is read at or past `nchars`, the capacity the layout had for them.
//
// Two details decide byte equality with Python's json.dumps:
//   - Escaping. RLE characters run from chr(48) to chr(111); of those only '\' (92) is escaped, as "\\". A string's
//     json length is its length plus its number of backslashes. Strings are copied 512 bytes per warp step: each lane
//     holds 16 bytes of 32-byte chunks, a ballot per chunk finds the backslashes and a popc prefix places each byte.
//   - one2x = repr(round(gs / gn, 2)), 0.0 when gn == 0. x = gs / gn is one IEEE double division, as in Python. Python
//     rounds the exact binary value of x to 2 decimals, ties to even (1/8 -> 0.12, 3/8 -> 0.38; the double of 1/200
//     lies above the tie -> 0.01). Here k = round_half_even(100 x) is computed exactly in integers from x's mantissa and
//     exponent, and printed as k / 100 with trailing zeros stripped and at least one decimal (0.0, 0.5, 0.33, 5.0).
//     For |gs|, |gn| < 2^31, k has at most 12 digits, so that decimal is the shortest that round-trips: Python's repr.
// Boxes print as Python prints float(int) ("12.0"; every coordinate is far below 1e16), areas and ranges as ints.
#include "common.cuh"

namespace s2d {

constexpr int AJ_WARPS = 8;                    // annotations per CTA
constexpr int AJ_SCAN_THREADS = 1024;
constexpr int AJ_CHUNKS = 16;                  // 32-byte chunks per lane step of the string copy (512 bytes per warp)

// A warp-uniform write cursor. Every lane runs the same calls, so `p` stays uniform; `one` writes on lane 0 only
// (small fixed text and numbers), `rep` and `str` write cooperatively. WRITE = false only counts.
template <bool WRITE>
struct AjOut {
    char* out;
    int64_t cap, p;
    int lane;
    __device__ __forceinline__ void put(int64_t q, char ch) const {
        if (WRITE && q < cap) out[q] = ch;
    }
    __device__ void lit(const char* s) {                                   // lane 0, serial
        for (; *s; ++s, ++p) if (lane == 0) put(p, *s);
    }
    __device__ void num(int64_t x) {                                       // decimal, lane 0
        if (x < 0) { if (lane == 0) put(p, '-'); ++p; x = -x; }
        int n = 1;
        for (int64_t t = x; t >= 10; t /= 10) ++n;
        if (WRITE && lane == 0)
            for (int i = n - 1; i >= 0; --i, x /= 10) put(p + i, (char)('0' + x % 10));
        p += n;
    }
    __device__ void rep(const char* s, int n, int64_t k) {                 // s (n bytes) k times, all lanes
        if (WRITE)
            for (int64_t b = lane; b < n * k; b += 32) put(p + b, s[b % n]);
        p += n * k;
    }
    // `k` frames without a member: "null, " each, except that the list's last frame has no separator (no byte is
    // written twice: the lanes of rep and lane 0 of the next lit store to disjoint addresses)
    __device__ void nulls(int64_t k, bool last) {
        if (k <= 0) return;
        if (last) {
            rep("null, ", 6, k - 1);
            rep("null", 4, 1);
        } else {
            rep("null, ", 6, k);
        }
    }
    // json string body of s[0, n): '\' -> "\\"
    __device__ void str(const char* __restrict__ s, int64_t n) {
        for (int64_t base = 0; base < n; base += 32 * AJ_CHUNKS) {
            char c[AJ_CHUNKS];
#pragma unroll
            for (int k = 0; k < AJ_CHUNKS; ++k) {
                const int64_t i = base + 32 * k + lane;
                c[k] = i < n ? s[i] : 0;
            }
            int before = 0;                                                // backslashes of earlier chunks
            if (WRITE) {
#pragma unroll
                for (int k = 0; k < AJ_CHUNKS; ++k) {
                    const unsigned bs = __ballot_sync(0xffffffffu, c[k] == '\\');
                    if (c[k]) {
                        const int64_t q = p + 32 * k + lane + before + __popc(bs & ((1u << lane) - 1u));
                        put(q, c[k]);
                        if (c[k] == '\\') put(q + 1, '\\');
                    }
                    before += __popc(bs);
                }
            } else {
#pragma unroll
                for (int k = 0; k < AJ_CHUNKS; ++k) before += c[k] == '\\';
                before = __reduce_add_sync(0xffffffffu, before);
            }
            p += min((int64_t)32 * AJ_CHUNKS, n - base) + before;
        }
    }
    // repr(round(gs / gn, 2)); 0.0 when gn == 0
    __device__ void one2x(int gs, int gn) {
        const double x = gn ? (double)gs / (double)gn : 0.0;
        if (signbit(x)) { if (lane == 0) put(p, '-'); ++p; }
        const uint64_t bits = __double_as_longlong(fabs(x));
        const int ex = (int)(bits >> 52);
        uint64_t m = bits & ((1ull << 52) - 1);
        int e;                                                             // |x| = m * 2^e
        if (ex == 0) e = -1074;
        else { m |= 1ull << 52; e = ex - 1075; }
        int64_t k;
        const uint64_t n100 = 100 * m;                                     // < 2^60
        if (e >= 0) k = (int64_t)(n100 << e);                              // |x| < 2^31: no overflow
        else if (-e > 62) k = 0;                                           // 100 |x| < 2^-2: rounds to 0
        else {
            const int s = -e;
            const uint64_t q = n100 >> s, r = n100 & ((1ull << s) - 1), half = 1ull << (s - 1);
            k = (int64_t)(q + (r > half || (r == half && (q & 1))));
        }
        num(k / 100);
        const int f = (int)(k % 100);
        if (lane == 0) put(p, '.');
        ++p;
        if (f % 10 == 0) {
            if (lane == 0) put(p, (char)('0' + f / 10));
            ++p;
        } else {
            if (lane == 0) { put(p, (char)('0' + f / 10)); put(p + 1, (char)('0' + f % 10)); }
            p += 2;
        }
    }
};

// the video of annotation a: the largest v with vann[v].first <= a (videos without annotation share the next one's
// first, and the last of such a tie is the one that owns a)
__device__ __forceinline__ int aj_video_of(const int32_t* __restrict__ vann, int nvideos, int64_t a) {
    int lo = 0, hi = nvideos - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (vann[2 * mid + 1] <= a) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// member m of annotation [m0, m0 + nm): frame, bbox, area, string start (lanes 0..5 load the row, shuffled out)
struct AjMember {
    int f, x0, y0, x1, y1, area;
};
__device__ __forceinline__ AjMember aj_member(const int32_t* __restrict__ members, int64_t m, int lane) {
    const int w = lane < 6 ? members[6 * m + lane] : 0;
    AjMember r;
    r.f = __shfl_sync(0xffffffffu, w, 0);
    r.x0 = __shfl_sync(0xffffffffu, w, 1);
    r.y0 = __shfl_sync(0xffffffffu, w, 2);
    r.x1 = __shfl_sync(0xffffffffu, w, 3);
    r.y1 = __shfl_sync(0xffffffffu, w, 4);
    r.area = __shfl_sync(0xffffffffu, w, 5);
    return r;
}

template <bool WRITE>
__global__ void __launch_bounds__(AJ_WARPS * 32, 1)
aj_text_kernel(const s2d_video_desc* __restrict__ descs, int nvideos, int64_t total_rows, const int32_t* __restrict__ vann,
               const int32_t* __restrict__ ann, const int32_t* __restrict__ members,
               const int64_t* __restrict__ member_off, const char* __restrict__ chars, int64_t nchars,
               const int32_t* __restrict__ clusters, const int32_t* __restrict__ pairs, const int64_t* __restrict__ sizes,
               int64_t* __restrict__ alen, const int64_t* __restrict__ video_off, int64_t capacity, char* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t a = (int64_t)blockIdx.x * AJ_WARPS + (threadIdx.x >> 5);
    const int64_t A = sizes[0], M = sizes[1], S = sizes[2];
    [[maybe_unused]] const int64_t K = sizes[3], R = sizes[4];
    if (a >= A) return;
    S2D_DEV_ASSERT(A <= total_rows && M <= total_rows);
    const int v = aj_video_of(vann, nvideos, a);
    const int nann = vann[2 * v], a0 = vann[2 * v + 1];
    S2D_DEV_ASSERT(v >= 0 && v < nvideos && a >= a0 && a < a0 + nann);
    const s2d_video_desc d = descs[v];
    const int T = d.T, H = d.H, W = d.W;
    const int32_t* an = ann + 7 * a;
    const int gn = an[2], gs = an[3], ci = an[4], nm = an[6];
    const int64_t m0 = an[5];
    S2D_DEV_ASSERT(m0 >= 0 && nm >= 0 && m0 + nm <= M && ci >= 0 && ci < K);
    AjOut<WRITE> o{out, capacity, 0, lane};
    if (WRITE) {
        const int64_t first = video_off[v] + 1;                            // after the video's "["
        o.p = first + alen[a] - alen[a0];
        if (a == a0) o.put(first - 1, '[');
    }
    o.lit("{\"video_id\": 1, \"iscrowd\": 0, \"height\": ");
    o.num(H);
    o.lit(", \"width\": ");
    o.num(W);
    o.lit(", \"length\": ");
    o.num(T);
    // segmentations, bboxes, areas: one entry per frame, null where the annotation has no member
    for (int sec = 0; sec < 3; ++sec) {
        o.lit(sec == 0 ? ", \"segmentations\": [" : sec == 1 ? "], \"bboxes\": [" : "], \"areas\": [");
        int prev = -1;
        for (int j = 0; j < nm; ++j) {
            const int64_t m = m0 + j;
            const AjMember me = aj_member(members, m, lane);
            S2D_DEV_ASSERT(me.f > prev && me.f < T);
            o.nulls(me.f - prev - 1, false);
            if (sec == 0) {
                // S > nchars when stage E's string capacity was short: the layout copied only what fits and the caller
                // re-runs stage E, so the text is discarded; reads stay inside the nchars bytes the buffer holds
                const int64_t s0 = min(member_off[m], nchars), s1 = min(m + 1 < M ? member_off[m + 1] : S, nchars);
                S2D_DEV_ASSERT(s0 >= 0 && s0 <= s1 && s1 <= nchars && s1 <= S);
                o.lit("{\"size\": [");
                o.num(H);
                o.lit(", ");
                o.num(W);
                o.lit("], \"counts\": \"");
                o.str(chars + s0, s1 - s0);
                o.lit("\"}");
            } else if (sec == 1) {
                o.lit("[");
                o.num(me.x0);
                o.lit(".0, ");
                o.num(me.y0);
                o.lit(".0, ");
                o.num((int64_t)me.x1 - me.x0 + 1);
                o.lit(".0, ");
                o.num((int64_t)me.y1 - me.y0 + 1);
                o.lit(".0]");
            } else {
                o.num(me.area);
            }
            if (me.f < T - 1) o.lit(", ");
            prev = me.f;
        }
        o.nulls(T - 1 - prev, true);
    }
    o.lit("], \"category_id\": 1, \"id\": ");
    o.num(a - a0 + 1);
    o.lit(", \"one2x\": ");
    o.one2x(gs, gn);
    o.lit(", \"visibility_ranges\": [");
    const int32_t* cl = clusters + 2 * ci;
    const int64_t p0 = cl[0];
    const int np = cl[1];
    S2D_DEV_ASSERT(p0 >= 0 && np >= 0 && p0 + np <= R);
    for (int i = 0; i < np; ++i) {
        o.lit(i ? ", [" : "[");
        o.num(pairs[2 * (p0 + i)]);
        o.lit(", ");
        o.num(pairs[2 * (p0 + i) + 1]);
        o.lit("]");
    }
    o.lit("]}");
    if (WRITE) o.lit(a + 1 < a0 + nann ? ", " : "]");
    else if (lane == 0) alen[a] = o.p + 2;                                 // with its ", " or the video's brackets
}

// in place: alen[0, A) -> exclusive prefix, alen[A] = total; per video its text length -> video_off [nvideos + 1],
// needed = the total; "[]" for a status-1 video without annotation
__global__ void __launch_bounds__(AJ_SCAN_THREADS)
aj_scan_kernel(int nvideos, int64_t total_rows, const int32_t* __restrict__ vidinfo, const int32_t* __restrict__ vann,
               const int64_t* __restrict__ sizes, int64_t* __restrict__ alen, int64_t* __restrict__ video_off,
               int64_t* __restrict__ needed, int64_t capacity, char* __restrict__ out) {
    __shared__ int64_t wsum[AJ_SCAN_THREADS / 32];
    const int tid = threadIdx.x;
    const int64_t A = sizes[0];
    S2D_DEV_ASSERT(A >= 0 && A <= total_rows);
    int64_t carry = 0;
    for (int64_t base = 0; base < A; base += AJ_SCAN_THREADS) {
        const int64_t i = base + tid;
        const int64_t x = i < A ? alen[i] : 0;
        int64_t tot;
        const int64_t ex = block_excl_scan<AJ_SCAN_THREADS>(x, wsum, tot);
        if (i < A) alen[i] = carry + ex;
        carry += tot;
    }
    if (tid == 0) alen[A] = carry;
    __syncthreads();
    carry = 0;
    for (int base = 0; base < nvideos; base += AJ_SCAN_THREADS) {
        const int v = base + tid;
        int64_t len = 0;
        bool empty = false;
        if (v < nvideos && vidinfo[v * S2D_VIDINFO_WORDS + 3] == 1) {
            const int n = vann[2 * v], a0 = vann[2 * v + 1];
            S2D_DEV_ASSERT(n >= 0 && a0 >= 0 && a0 + n <= A);
            empty = n == 0;
            len = empty ? 2 : alen[a0 + n] - alen[a0];
        }
        int64_t tot;
        const int64_t ex = carry + block_excl_scan<AJ_SCAN_THREADS>(len, wsum, tot);
        if (v < nvideos) {
            video_off[v] = ex;
            if (empty) {
                if (ex < capacity) out[ex] = '[';
                if (ex + 1 < capacity) out[ex + 1] = ']';
            }
        }
        carry += tot;
    }
    if (tid == 0) { video_off[nvideos] = carry; *needed = carry; }
}

}  // namespace s2d

using namespace s2d;

extern "C" int s2d_annotation_json_work_ints(int64_t total_rows, int nvideos, int64_t* out) {
    S2D_CHECK_ARG(out && total_rows >= 0 && nvideos > 0, "s2d_annotation_json_work_ints: bad arguments");
    *out = 2 * (total_rows + 1);
    return 0;
}

extern "C" int s2d_annotation_json(const s2d_video_desc* descs, int nvideos, int64_t total_rows, const int32_t* vidinfo,
                                   const int32_t* vann, const int32_t* ann, const int32_t* members,
                                   const int64_t* member_off, const char* chars, int64_t nchars,
                                   const int32_t* clusters,
                                   const int32_t* pairs, const int64_t* sizes, int32_t* work, int64_t capacity, char* out,
                                   int64_t* video_off, int64_t* needed, void* stream) {
    S2D_ENTER(stream);
    S2D_CHECK_ARG(descs && vidinfo && vann && ann && members && member_off && chars && clusters && pairs && sizes && work &&
                      out && video_off && needed,
                  "s2d_annotation_json: null pointer");
    S2D_CHECK_ARG(nvideos > 0 && nvideos <= 65535 && total_rows > 0 && nchars >= 0 && capacity >= 0,
                  "s2d_annotation_json: bad sizes");
    S2D_CHECK_ARG(reinterpret_cast<uintptr_t>(work) % 8 == 0, "s2d_annotation_json: work must be 8-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    int64_t* alen = reinterpret_cast<int64_t*>(work);
    const unsigned blocks = (unsigned)((total_rows + AJ_WARPS - 1) / AJ_WARPS);
    aj_text_kernel<false><<<blocks, AJ_WARPS * 32, 0, st>>>(descs, nvideos, total_rows, vann, ann, members, member_off,
                                                            chars, nchars, clusters, pairs, sizes, alen, nullptr, capacity,
                                                            out);
    S2D_CHECK_LAUNCH("aj_text_kernel<length>");
    aj_scan_kernel<<<1, AJ_SCAN_THREADS, 0, st>>>(nvideos, total_rows, vidinfo, vann, sizes, alen, video_off, needed,
                                                  capacity, out);
    S2D_CHECK_LAUNCH("aj_scan_kernel");
    aj_text_kernel<true><<<blocks, AJ_WARPS * 32, 0, st>>>(descs, nvideos, total_rows, vann, ann, members, member_off,
                                                           chars, nchars, clusters, pairs, sizes, alen, video_off, capacity,
                                                           out);
    S2D_CHECK_LAUNCH("aj_text_kernel<write>");
    return 0;
}
