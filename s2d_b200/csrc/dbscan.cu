// Batched Hamming DBSCAN: XOR + popc neighbour tests on bit rows, lock-free union-find over the
// core-core graph (root = lowest core index of the component, which is exactly the order in
// which sklearn's sequential expansion numbers clusters), border rows take the minimum label
// among their core neighbours.
#include "dbscan.cuh"

#include <limits.h>

#include <algorithm>

namespace s2d {

constexpr int DB_THREADS = 256;
constexpr int DB_ROWS_I = 32;     // rows i per CTA: 8 warps x 4 rows
constexpr int DB_NWC = 64;        // word chunk staged in shared memory
constexpr int DB_JT = 1;          // 32-row tiles of rows j staged per barrier pair (4 was measured: no gain)

__device__ __forceinline__ int uf_find(int32_t* parent, int i) {
    while (true) {
        int p = parent[i];
        S2D_DEV_ASSERT(p >= 0 && p <= i);          // roots are component minima: parents never point upwards
        if (p == i) return i;
        int gp = parent[p];
        if (gp != p) parent[i] = gp;   // path halving (benign race)
        i = p;
    }
}

// hook the larger root under the smaller one: the root of a component is its minimum index.
// Returns the root the two rows shared when the call returned.
__device__ __forceinline__ int uf_unite(int32_t* parent, int a, int b) {
    while (true) {
        a = uf_find(parent, a);
        b = uf_find(parent, b);
        if (a == b) return a;
        if (a < b) { int t = a; a = b; b = t; }
        if (atomicCAS(&parent[a], a, b) == a) return b;
    }
}

// carry-save adder on 32 bit lanes: (carry, sum) = a + b + c. POPC issues at a quarter of the LOP3 rate, so the
// distance loops count four words with one POPC instead of four.
__device__ __forceinline__ void csa(uint32_t& carry, uint32_t& sum, uint32_t a, uint32_t b, uint32_t c) {
    const uint32_t u = a ^ b;
    carry = (a & b) | (u & c);
    sum = u ^ c;
}

// Work list of a batch of problems: wl[0 .. n] = exclusive prefix of the problems' 32-row blocks nb(p) = ceil(N / 32),
// wl[n + 1 .. 2n + 1] = exclusive prefix of their block PAIRS nb (nb + 1) / 2. Most problems of a batch are empty (a
// video has 16 cluster slots and uses one or two): the passes below run as persistent CTAs over the non-empty work only
// instead of launching - and immediately retiring - a CTA per (problem, block) slot (round 1: 23 k CTAs per pass on the
// C2 batch, 2 944 of them with work).
__global__ void __launch_bounds__(1024) db_worklist_kernel(const DbProblem* __restrict__ problems, int n, int32_t* __restrict__ wl) {
    __shared__ int wsum[32];
    const int tid = threadIdx.x;
    int run0 = 0, run1 = 0;
    for (int base = 0; base < n; base += 1024) {
        const int i = base + tid;
        const int nb = i < n ? (problems[i].N + DB_ROWS_I - 1) / DB_ROWS_I : 0;
        int t0, t1;
        const int e0 = block_excl_scan<1024>(nb, wsum, t0);
        const int e1 = block_excl_scan<1024>(nb * (nb + 1) / 2, wsum, t1);
        if (i < n) { wl[i] = run0 + e0; wl[n + 1 + i] = run1 + e1; }
        run0 += t0; run1 += t1;
    }
    if (tid == 0) { wl[n] = run0; wl[2 * n + 1] = run1; }
}

// MODE 0: neighbour counts -> core   1: unions   2: border -> min core root. One work item = a 32-row block bi of a
// problem against every row j (MODE 1: every row j < i). Measured and rejected: one item per PAIR of blocks in MODE 1
// (critical path of one tile step instead of N / 32) - a block that walks its j tiles in turn remembers which rows it
// already united (imember) and issues ~N unions per problem; independent pairs issue one per neighbouring pair of rows
// (~20 x more atomicCAS / find chains): dbscan1 0.17 -> 0.31 ms, group 0.64 -> 0.95 ms on the C2 batch.
template <int MODE>
__device__ __forceinline__ void db_item(const DbProblem& p, int bi, int bj, uint32_t (&xi)[DB_ROWS_I][DB_NWC],
                                        uint32_t (&xjT)[DB_NWC][32 * DB_JT + 1]) {
    const int N = p.N;
    const int i0 = bi * DB_ROWS_I;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    int irow[4];
    bool icore[4];
    int acc[4];   // MODE0: neighbour count; MODE2: min root
    int imember[4];   // MODE1: a row of irow[r]'s component (lane-private view)
    bool mine = false;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        irow[r] = i0 + warp * 4 + r;
        imember[r] = irow[r];
        icore[r] = false;
        acc[r] = (MODE == 2) ? INT_MAX : 0;
        if (MODE != 0 && irow[r] < N) icore[r] = p.core[irow[r]] != 0;
        if (irow[r] < N) mine |= (MODE == 1) ? icore[r] : (MODE == 2 ? !icore[r] : true);
    }
    if (!__syncthreads_or(mine)) return;   // CTA-uniform: nothing to do for these 32 rows

    constexpr int JROWS = 32 * DB_JT;            // rows j staged per round: DB_JT tiles of 32, one barrier pair for all
    const int jbeg = 0;
    (void)bj;
    const int jend = (MODE == 1) ? min(N, i0 + DB_ROWS_I) : N;   // unions only need j < i
    const bool single_chunk = p.nw <= DB_NWC;
    // Gram mode (large problems): the caller computed G = X X^T of the 0/1 rows on the tensor cores; the Hamming distance
    // of two rows is |a| + |b| - 2 a.b with |a| = G[a][a]; rows that are not valid are all-zero rows
    int ipop[4] = {0, 0, 0, 0};
    bool ival[4] = {false, false, false, false};
    if (p.gram) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            ival[r] = irow[r] < N && (!p.valid || p.valid[irow[r]]);
            ipop[r] = ival[r] ? p.gram[(int64_t)irow[r] * p.gstride + irow[r]] : 0;
        }
    }
    for (int j0 = jbeg; j0 < jend; j0 += JROWS) {
        int dist[DB_JT][4];
        uint32_t ones[DB_JT][4], twos[DB_JT][4];   // carry-save partial counts (weights 1 and 2)
#pragma unroll
        for (int jt = 0; jt < DB_JT; ++jt)
#pragma unroll
            for (int r = 0; r < 4; ++r) { dist[jt][r] = 0; ones[jt][r] = 0; twos[jt][r] = 0; }
        const int jrows = min(JROWS, ((jend - j0 + 31) >> 5) << 5);
        if (p.gram) {
            const int j = j0 + lane;
            const bool vj = j < N && (!p.valid || p.valid[j]);
            const int jpop = vj ? p.gram[(int64_t)j * p.gstride + j] : 0;
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int g = (ival[r] && vj) ? p.gram[(int64_t)irow[r] * p.gstride + j] : 0;
                dist[0][r] = ipop[r] + jpop - 2 * g;
            }
        } else {
        for (int c0 = 0; c0 < p.nw; c0 += DB_NWC) {
            const int cw = min(DB_NWC, p.nw - c0);
            __syncthreads();
            if (!(single_chunk && j0 > jbeg)) {
                const int cwp = (cw + 3) & ~3;
                for (int idx = tid; idx < DB_ROWS_I * cwp; idx += DB_THREADS) {
                    const int r = idx / cwp, w = idx - r * cwp, row = i0 + r;
                    uint32_t v = 0;
                    if (w < cw && row < N && (!p.valid || p.valid[row])) v = p.bits[(int64_t)row * p.stride + p.w0 + c0 + w];
                    S2D_DEV_ASSERT(r < DB_ROWS_I && w < DB_NWC);
                    xi[r][w] = v;
                }
            }
            const int cw4 = (cw + 3) & ~3;           // the distance loop eats 4 words at a time: pad with zeros
            for (int idx = tid; idx < jrows * cw4; idx += DB_THREADS) {
                const int r = idx / cw4, w = idx - r * cw4, row = j0 + r;
                uint32_t v = 0;
                if (w < cw && row < N && (!p.valid || p.valid[row])) v = p.bits[(int64_t)row * p.stride + p.w0 + c0 + w];
                S2D_DEV_ASSERT(w < DB_NWC && r < 32 * DB_JT);
                xjT[w][r] = v;
            }
            __syncthreads();
            for (int w = 0; w < cw4; w += 4) {
                uint32_t x[4][4];
#pragma unroll
                for (int r = 0; r < 4; ++r)
#pragma unroll
                    for (int k = 0; k < 4; ++k) x[r][k] = xi[warp * 4 + r][w + k];
#pragma unroll
                for (int jt = 0; jt < DB_JT; ++jt) {
                    if (jt * 32 < jrows) {
                        uint32_t xj[4];
#pragma unroll
                        for (int k = 0; k < 4; ++k) xj[k] = xjT[w + k][jt * 32 + lane];
#pragma unroll
                        for (int r = 0; r < 4; ++r) {
                            uint32_t ta, tb, f;
                            csa(ta, ones[jt][r], ones[jt][r], x[r][0] ^ xj[0], x[r][1] ^ xj[1]);
                            csa(tb, ones[jt][r], ones[jt][r], x[r][2] ^ xj[2], x[r][3] ^ xj[3]);
                            csa(f, twos[jt][r], twos[jt][r], ta, tb);
                            dist[jt][r] += __popc(f);                 // in units of 4
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int jt = 0; jt < DB_JT; ++jt)
#pragma unroll
            for (int r = 0; r < 4; ++r) dist[jt][r] = 4 * dist[jt][r] + 2 * __popc(twos[jt][r]) + __popc(ones[jt][r]);
        }
#pragma unroll
        for (int jt = 0; jt < DB_JT; ++jt) {
            if (jt * 32 >= jrows) break;
            const int j = j0 + jt * 32 + lane;
            const bool jv = j < N;
            bool jcore = false;
            if (MODE != 0 && jv) jcore = p.core[j] != 0;
            int jroot = INT_MAX;
            if (MODE == 2 && jcore) jroot = uf_find(p.parent, j);
            // MODE 1: a row of j's component (its parent when read). Equal to a row known to be in i's component =>
            // already united; components never split, so a stale value only costs a redundant find.
            int jmember = -1;
            if (MODE == 1 && jcore) jmember = p.parent[j];
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const bool nb = jv && irow[r] < N && dist[jt][r] <= p.kmax;
                if (MODE == 0) {
                    acc[r] += __popc(__ballot_sync(0xffffffffu, nb));
                } else if (MODE == 1) {
                    if (nb && icore[r] && jcore && j < irow[r] && jmember != imember[r])
                        imember[r] = jmember = uf_unite(p.parent, irow[r], j);
                } else {
                    const int cand = (nb && !icore[r] && jcore) ? jroot : INT_MAX;
                    acc[r] = min(acc[r], __reduce_min_sync(0xffffffffu, cand));
                }
            }
        }
        if (MODE == 0) {
            // only "count >= min_samples" is ever read: stop scanning once every row of the CTA has got there
            // (rows of one object are mutual neighbours, so a handful of frames' worth of rows j is usually enough)
            bool done = true;
#pragma unroll
            for (int r = 0; r < 4; ++r) done &= irow[r] >= N || acc[r] >= p.min_samples;
            if (__syncthreads_and(done)) break;
        }
    }
    if (lane == 0) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            if (irow[r] >= N) continue;
            if (MODE == 0) {
                p.core[irow[r]] = acc[r] >= p.min_samples;
                p.parent[irow[r]] = irow[r];
            } else if (MODE == 2) {
                if (!icore[r]) p.aux[irow[r]] = acc[r];
            }
        }
    }
}

template <int MODE>
__global__ void __launch_bounds__(DB_THREADS) db_pass_kernel(const DbProblem* __restrict__ problems, int n, const int32_t* __restrict__ wl) {
    __shared__ uint32_t xi[DB_ROWS_I][DB_NWC];
    __shared__ uint32_t xjT[DB_NWC][32 * DB_JT + 1];
    const int32_t* pref = wl;
    const int total = pref[n];
    for (int w = blockIdx.x; w < total; w += gridDim.x) {
        int lo = 0, hi = n;                              // last problem with pref[pr] <= w (CTA-uniform)
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(pref + mid) <= w) lo = mid; else hi = mid;
        }
        const DbProblem p = problems[lo];
        const int bi = w - __ldg(pref + lo), bj = 0;
        S2D_DEV_ASSERT(bi * DB_ROWS_I < p.N);
        db_item<MODE>(p, bi, bj, xi, xjT);
        __syncthreads();                                 // the next item restages xi / xjT
    }
}

// cluster numbering by ascending root index + final labels; one CTA per problem
__global__ void __launch_bounds__(1024) db_label_kernel(const DbProblem* __restrict__ problems) {
    const DbProblem p = problems[blockIdx.x];
    const int N = p.N, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    __shared__ int wsum[32];
    __shared__ int running;
    if (tid == 0) running = 0;
    for (int i = tid; i < N; i += 1024)
        if (p.core[i]) p.aux[i] = uf_find(p.parent, i);
    __syncthreads();
    for (int base = 0; base < N; base += 1024) {
        const int i = base + tid;
        const bool flag = i < N && p.core[i] && p.aux[i] == i;
        const uint32_t b = __ballot_sync(0xffffffffu, flag);
        if (lane == 0) wsum[warp] = __popc(b);
        __syncthreads();
        int before = 0, total = 0;
        for (int w = 0; w < 32; ++w) {
            const int s = wsum[w];
            if (w < warp) before += s;
            total += s;
        }
        const int pos = running + before + __popc(b & ((1u << lane) - 1u));
        if (flag) p.parent[i] = pos;     // parent[] of a root now holds its cluster id
        __syncthreads();
        if (tid == 0) running += total;
        __syncthreads();
    }
    for (int i = tid; i < N; i += 1024) {
        const int a = p.aux[i];
        int lab = -1;
        S2D_DEV_ASSERT(!(p.core[i] || a != INT_MAX) || (a >= 0 && a < N));
        if (p.core[i] || a != INT_MAX) lab = p.parent[a];
        p.labels[i] = lab;
    }
    if (tid == 0 && p.nclusters) *p.nclusters = running;
}

int launch_dbscan(const DbProblem* problems, int nproblems, int max_N, int max_nw, int32_t* wl, cudaStream_t st) {
    (void)max_nw;
    if (nproblems <= 0 || max_N <= 0) return 0;
    db_worklist_kernel<<<1, 1024, 0, st>>>(problems, nproblems, wl);
    S2D_CHECK_LAUNCH("db_worklist_kernel");
    int dev = 0, nsm = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
    const int64_t nb = (max_N + DB_ROWS_I - 1) / DB_ROWS_I;
    const int64_t cap = (int64_t)nsm * (2048 / DB_THREADS);                      // resident CTAs
    const unsigned g02 = (unsigned)std::min<int64_t>(cap, nb * nproblems);
    db_pass_kernel<0><<<g02, DB_THREADS, 0, st>>>(problems, nproblems, wl);
    S2D_CHECK_LAUNCH("db_pass_kernel<0>");
    db_pass_kernel<1><<<g02, DB_THREADS, 0, st>>>(problems, nproblems, wl);
    S2D_CHECK_LAUNCH("db_pass_kernel<1>");
    db_pass_kernel<2><<<g02, DB_THREADS, 0, st>>>(problems, nproblems, wl);
    S2D_CHECK_LAUNCH("db_pass_kernel<2>");
    db_label_kernel<<<nproblems, 1024, 0, st>>>(problems);
    S2D_CHECK_LAUNCH("db_label_kernel");
    return 0;
}

// ------------------------------------------------------------------------------------------
__global__ void db1_setup_kernel(const s2d_video_desc* __restrict__ descs, int nvideos,
                                 const uint32_t* __restrict__ xbits, double eps, int min_samples,
                                 int32_t* __restrict__ work, int32_t* __restrict__ labels1,
                                 int32_t* __restrict__ vidinfo, DbProblem* __restrict__ problems) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= nvideos) return;
    const s2d_video_desc d = descs[v];
    DbProblem p;
    p.bits = xbits + d.xbits_off;
    p.valid = nullptr;
    p.core = work + 3 * d.row0;
    p.parent = p.core + d.Nm;
    p.aux = p.parent + d.Nm;
    p.labels = labels1 + d.row0;
    p.gram = nullptr; p.gstride = 0; p.pad = 0;
    p.nclusters = vidinfo + (int64_t)v * S2D_VIDINFO_WORDS + 0;
    p.stride = d.TW;
    p.w0 = 0;
    p.nw = d.TW;
    p.N = d.Nm;
    p.kmax = hamming_kmax(d.T, eps);
    p.min_samples = min_samples;
    problems[v] = p;
}

__global__ void db_single_setup_kernel(const uint32_t* bits, int N, int stride, int D, double eps,
                                       int min_samples, int32_t* work, int32_t* labels,
                                       DbProblem* problems) {
    DbProblem p;
    p.bits = bits;
    p.valid = nullptr;
    p.core = work;
    p.parent = work + N;
    p.aux = work + 2 * N;
    p.labels = labels;
    p.gram = nullptr; p.gstride = 0; p.pad = 0;
    p.nclusters = nullptr;
    p.stride = stride;
    p.w0 = 0;
    p.nw = (D + 31) / 32;
    p.N = N;
    p.kmax = hamming_kmax(D, eps);
    p.min_samples = min_samples;
    problems[0] = p;
}

}  // namespace s2d

using namespace s2d;

static_assert(sizeof(DbProblem) % 8 == 0, "DbProblem must keep 8-byte alignment in the work buffer");

extern "C" int s2d_dbscan_work_ints(int64_t total_rows, int nproblems, int64_t* out) {
    if (!out) return -1;
    *out = 3 * total_rows + 2 + (int64_t)nproblems * (int64_t)(sizeof(DbProblem) / 4) + db_worklist_ints(nproblems);
    return 0;
}

extern "C" int s2d_dbscan_visibility(const s2d_video_desc* descs, int nvideos, int max_Nm, int max_TW,
                                     int64_t total_rows, const uint32_t* xbits, double eps,
                                     int min_samples, int32_t* work, int32_t* labels1,
                                     int32_t* vidinfo, void* stream) {
    S2D_ENTER(stream);
    S2D_CHECK_ARG(descs && xbits && work && labels1 && vidinfo, "s2d_dbscan_visibility: null pointer");
    S2D_CHECK_ARG(nvideos > 0 && nvideos <= 65535 && max_Nm > 0, "s2d_dbscan_visibility: bad sizes");
    cudaStream_t st = (cudaStream_t)stream;
    // problem descriptors live behind the 3*total_rows ints of union-find scratch (8-byte aligned)
    int64_t off = 3 * total_rows;
    off += off & 1;
    DbProblem* problems = reinterpret_cast<DbProblem*>(work + off);
    S2D_CHECK_ARG((((uintptr_t)problems) & 7) == 0, "s2d_dbscan_visibility: work must be 8-byte aligned");
    db1_setup_kernel<<<(nvideos + 127) / 128, 128, 0, st>>>(descs, nvideos, xbits, eps, min_samples, work,
                                                            labels1, vidinfo, problems);
    S2D_CHECK_LAUNCH("db1_setup_kernel");
    return launch_dbscan(problems, nvideos, max_Nm, max_TW, reinterpret_cast<int32_t*>(problems + nvideos), st);
}

extern "C" int s2d_hamming_dbscan(const uint32_t* bits, int N, int stride, int D, double eps,
                                  int min_samples, int32_t* work, int32_t* labels, void* stream) {
    S2D_ENTER(stream);
    S2D_CHECK_ARG(bits && work && labels, "s2d_hamming_dbscan: null pointer");
    S2D_CHECK_ARG(N > 0 && D > 0 && stride >= (D + 31) / 32, "s2d_hamming_dbscan: bad sizes N=%d D=%d stride=%d", N, D, stride);
    cudaStream_t st = (cudaStream_t)stream;
    int64_t off = 3 * (int64_t)N;
    off += off & 1;
    DbProblem* problems = reinterpret_cast<DbProblem*>(work + off);
    S2D_CHECK_ARG((((uintptr_t)problems) & 7) == 0, "s2d_hamming_dbscan: work must be 8-byte aligned");
    db_single_setup_kernel<<<1, 1, 0, st>>>(bits, N, stride, D, eps, min_samples, work, labels, problems);
    S2D_CHECK_LAUNCH("db_single_setup_kernel");
    return launch_dbscan(problems, 1, N, (D + 31) / 32, reinterpret_cast<int32_t*>(problems + 1), st);
}
