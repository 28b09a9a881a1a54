// PNG label maps on the device: N zlib streams (each file's IDAT payloads joined) -> packed RGB frames, the pixels
// cv2.imread(path, IMREAD_COLOR) returns (in RGB order), for non-interlaced files.
//
//   png_inflate_kernel   warp per stream. All lanes decode the same symbols from one uniform 64-bit bit buffer, so no
//                        broadcast is needed. Dynamic blocks build their tables cooperatively in the warp's shared
//                        memory: __match_any_sync over the code lengths counts each length and ranks every symbol
//                        within it (canonical codes), a 9-bit (literal/length) or 6-bit (distance) primary table takes
//                        the short codes, and each primary slot with longer codes points to a sub-table sized by its
//                        longest code (a warp scan places them; zlib's ENOUGH bounds 852 / 592 entries hold). Literals
//                        are collected 32 at a time and stored by the warp at once. Matches run across the warp:
//                        dist < 32 is periodic, so every lane writes its bytes from the dist source bytes at once;
//                        otherwise steps of dist (>= 32) bytes, a __syncwarp between dependent steps. The window is the
//                        file's own output, read back through L1 / L2: a 32 KB shared window would hold a warp to 7 per
//                        SM, and the tables alone allow about 30.
//   png_unfilter_kernel  one warp per file, rows in order, the previous unfiltered row kept in shared memory (filtered
//                        in place). None / Up are lane-parallel, Sub is a stride-bpp warp scan with a carry from the
//                        previous 32 bytes, Avg / Paeth run lane-parallel over the bpp bytes of a pixel and serially
//                        along the row. Each finished row is converted straight to RGB; the adler32 of the stream is
//                        accumulated from the filtered bytes on the way and checked at the end.
//
// Conversion rules (libpng as cv2 sets it up for IMREAD_COLOR): palette lookup, gray replicated to R = G = B (1/2/4-bit
// gray scaled by 255, 85, 17), 1/2/4-bit indices unpacked MSB first, 16-bit samples reduced to their high byte, alpha
// (and tRNS) dropped.
#include "common.cuh"

namespace s2d {

constexpr int PI_WARPS = 4;             // streams per CTA of the inflate kernel
constexpr int PI_LROOT = 9, PI_DROOT = 6, PI_CROOT = 7;
constexpr int PI_LENOUGH = 852, PI_DENOUGH = 592;   // zlib's ENOUGH_LENS / ENOUGH_DISTS for these roots
constexpr uint32_t PI_PTR = 1u << 24;

struct __align__(16) InflateSmem {
    uint32_t lit[PI_LENOUGH];           // literal/length table; the code-length table (128 entries) while lengths are read
    uint32_t dist[PI_DENOUGH];
    uint16_t code[320];                 // canonical code of each symbol of the table being built
    uint8_t lens[320];                  // code lengths: literal/length [0, nlen), distance [nlen, nlen + ndist)
    uint8_t sub[1 << PI_LROOT];         // per primary slot: bits of its sub-table (0: none)
    int32_t cnt[16], next[16];
};

__constant__ uint16_t c_len_base[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31,
                                        35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
__constant__ uint8_t c_len_extra[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
__constant__ uint16_t c_dist_base[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769,
                                         1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
__constant__ uint8_t c_dist_extra[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
__constant__ uint8_t c_clen_order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};

__device__ __forceinline__ int png_channels(int ct) { return ct == 2 ? 3 : ct == 4 ? 2 : ct == 6 ? 4 : 1; }

// -1 for a (colour type, depth) pair PNG does not define or a frame the kernels do not take, else the row bytes
__device__ __forceinline__ int png_rowbytes(const s2d_png_desc& d) {
    const int ct = d.color_type, bd = d.bit_depth;
    const bool ok = (ct == 0 && (bd == 1 || bd == 2 || bd == 4 || bd == 8 || bd == 16)) ||
                    (ct == 3 && (bd == 1 || bd == 2 || bd == 4 || bd == 8)) ||
                    ((ct == 2 || ct == 4 || ct == 6) && (bd == 8 || bd == 16));
    if (!ok || d.width < 1 || d.height < 1 || d.width > S2D_PNG_MAX_ROWBYTES || (ct == 3 && (d.palette_size < 1 || d.palette_size > 256)))
        return -1;
    const int64_t rb = ((int64_t)d.width * png_channels(ct) * bd + 7) / 8;
    if (rb > S2D_PNG_MAX_ROWBYTES || (int64_t)d.height * (rb + 1) > S2D_PNG_MAX_RAW_BYTES) return -1;
    return (int)rb;
}

__device__ __forceinline__ uint32_t rev_bits(uint32_t x, int n) { return n ? __brev(x) >> (32 - n) : 0u; }

// Canonical Huffman table of n symbols (lengths lens[0, n), <= 15) at tab: primary slots [0, 2^root) indexed by the
// next root bits of the stream (LSB first); entry = symbol | length << 16 (length 0: no code), or a pointer
// offset | bits << 16 | PI_PTR to a sub-table indexed by the following `bits` bits. Returns false for an oversubscribed
// code or an incomplete one (zlib accepts incomplete only for a single code of length 1, or none at all). Warp-uniform.
__device__ bool build_table(InflateSmem& s, const uint8_t* lens, int n, uint32_t* tab, int root, int cap, int lane) {
    const unsigned lt = (1u << lane) - 1u;
    if (lane < 16) s.cnt[lane] = 0;
    for (int i = lane; i < (1 << root); i += 32) { tab[i] = 0; s.sub[i] = 0; }
    __syncwarp();
    for (int base = 0; base < n; base += 32) {              // symbols per length
        const int sym = base + lane;
        const int l = sym < n ? lens[sym] : 0;
        const unsigned peers = __match_any_sync(0xffffffffu, l);
        if (l > 0 && (peers & lt) == 0) s.cnt[l] += __popc(peers);
        __syncwarp();
    }
    int ok = 1;
    if (lane == 0) {
        int left = 1, code = 0, maxl = 0;
        s.next[0] = 0;
        for (int l = 1; l < 16; ++l) {
            left = (left << 1) - s.cnt[l];
            if (left < 0) ok = 0;
            code = (code + s.cnt[l - 1]) << 1;
            s.next[l] = code;
            if (s.cnt[l]) maxl = l;
        }
        if (ok && left > 0 && maxl > 1) ok = 0;
    }
    ok = __shfl_sync(0xffffffffu, ok, 0);
    __syncwarp();
    if (!ok) return false;
    for (int base = 0; base < n; base += 32) {              // canonical codes; short codes fill their primary slots
        const int sym = base + lane;
        const int l = sym < n ? lens[sym] : 0;
        const unsigned peers = __match_any_sync(0xffffffffu, l);
        const int c = l > 0 ? s.next[l] + __popc(peers & lt) : 0;
        __syncwarp();
        if (l > 0 && (peers & lt) == 0) s.next[l] += __popc(peers);
        if (l > 0) {
            S2D_DEV_ASSERT(sym < 320);
            s.code[sym] = (uint16_t)c;
            if (l <= root) {
                const uint32_t r = rev_bits((uint32_t)c, l);
                for (uint32_t k = 0; k < (1u << (root - l)); ++k) {
                    S2D_DEV_ASSERT((r | (k << l)) < (1u << root));
                    tab[r | (k << l)] = (uint32_t)sym | ((uint32_t)l << 16);
                }
            } else {
                const uint32_t p = rev_bits((uint32_t)c >> (l - root), root);
                S2D_DEV_ASSERT(p < (1u << root));
                // byte-wide max over the codes of one prefix: a CAS loop on the containing word
                unsigned* w = reinterpret_cast<unsigned*>(s.sub) + (p >> 2);
                const int sh = 8 * (p & 3);
                unsigned old = *w, assumed;
                do {
                    assumed = old;
                    if ((int)((assumed >> sh) & 0xFF) >= l - root) break;
                    old = atomicCAS_block(w, assumed, (assumed & ~(0xFFu << sh)) | ((unsigned)(l - root) << sh));
                } while (old != assumed);
            }
        }
        __syncwarp();
    }
    // place the sub-tables after the primary slots: exclusive warp scan of 2^bits over the slots
    int off = 1 << root;
    for (int base = 0; base < (1 << root); base += 32) {
        const int p = base + lane;
        const int b = s.sub[p];
        const int sz = b ? 1 << b : 0, incl = warp_incl_scan(sz);
        if (b) { S2D_DEV_ASSERT(p < (1 << root)); tab[p] = (uint32_t)(off + incl - sz) | ((uint32_t)b << 16) | PI_PTR; }
        off += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (off > cap) return false;                              // cannot happen for a complete code (zlib's ENOUGH)
    __syncwarp();
    for (int base = 0; base < n; base += 32) {              // long codes fill their sub-tables
        const int sym = base + lane;
        const int l = sym < n ? lens[sym] : 0;
        if (l > root) {
            const uint32_t c = s.code[sym];
            const uint32_t e = tab[rev_bits(c >> (l - root), root)];
            const int b = (e >> 16) & 0xFF, o = (int)(e & 0xFFFF), ls = l - root;
            const uint32_t r = rev_bits(c & ((1u << ls) - 1u), ls);
            for (uint32_t k = 0; k < (1u << (b - ls)); ++k) {
                S2D_DEV_ASSERT(o + (r | (k << ls)) < (uint32_t)cap);
                tab[o + (r | (k << ls))] = (uint32_t)sym | ((uint32_t)l << 16);
            }
        }
    }
    __syncwarp();
    return true;
}

// uniform bit reader: every lane holds the same state
struct BitIn {
    const uint8_t* __restrict__ src;
    int64_t pos, end;          // next byte to load, end of the stream
    uint64_t buf;
    int cnt;
    __device__ __forceinline__ void refill() {
        if (cnt < 32) {
            uint32_t w = 0;
#pragma unroll
            for (int k = 0; k < 4; ++k) w |= (pos + k < end ? (uint32_t)src[pos + k] : 0u) << (8 * k);
            buf |= (uint64_t)w << cnt;
            cnt += 32;
            pos += 4;
        }
    }
    __device__ __forceinline__ uint32_t bits(int n) { return (uint32_t)buf & ((1u << n) - 1u); }
    __device__ __forceinline__ void drop(int n) { buf >>= n; cnt -= n; }
    __device__ __forceinline__ uint32_t take(int n) { const uint32_t v = bits(n); drop(n); return v; }
    __device__ __forceinline__ bool overrun() const { return pos * 8 - cnt > end * 8; }
    __device__ __forceinline__ int64_t consumed_bytes() const { return pos - cnt / 8; }
};

__device__ __forceinline__ int decode_sym(BitIn& in, const uint32_t* tab, int root, int cap) {
    uint32_t e = tab[in.bits(root)];
    if (e & PI_PTR) {
        const int b = (e >> 16) & 0xFF;
        const uint32_t i = (e & 0xFFFF) + (((uint32_t)(in.buf >> root)) & ((1u << b) - 1u));
        S2D_DEV_ASSERT(i < (uint32_t)cap);
        e = tab[i];
    }
    const int l = (e >> 16) & 0xFF;
    if (l == 0) return -1;
    in.drop(l);
    return (int)(e & 0xFFFF);
}

__global__ void __launch_bounds__(PI_WARPS * 32)
png_inflate_kernel(const uint8_t* __restrict__ zdata, const int64_t* __restrict__ z_off, const s2d_png_desc* __restrict__ descs,
                   int N, uint8_t* __restrict__ raw_base, uint32_t* __restrict__ adler_out, int32_t* __restrict__ status) {
    __shared__ InflateSmem smem[PI_WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = blockIdx.x * PI_WARPS + warp;
    if (n >= N) return;
    InflateSmem& s = smem[warp];
    const s2d_png_desc& d = descs[n];
    const int rb = png_rowbytes(d);
    if (rb < 0) { if (lane == 0) status[n] = S2D_PNG_BAD_DESC; return; }
    const int64_t rawsize = (int64_t)d.height * (rb + 1);
    uint8_t* __restrict__ out = raw_base + d.raw_offset;
    BitIn in{zdata, z_off[n], z_off[n + 1], 0ull, 0};
    int err = 0;
    int64_t opos = 0;
    // zlib header: method 8, window <= 32 KB, no preset dictionary, check bits
    in.refill();
    const uint32_t cmf = in.take(8), flg = in.take(8);
    const int64_t window = (int64_t)1 << ((cmf >> 4) + 8);
    if ((cmf & 15) != 8 || (cmf >> 4) > 7 || (flg & 0x20) || ((cmf << 8) | flg) % 31 != 0) err = S2D_PNG_BAD_DEFLATE;
    // pending literals: lane k holds byte opos + k
    uint32_t pend = 0;
    int npend = 0;
    auto flush = [&]() {
        if (npend) {
            if (lane < npend) { S2D_DEV_ASSERT(opos + lane < rawsize); out[opos + lane] = (uint8_t)pend; }
            opos += npend;
            npend = 0;
        }
        __syncwarp();
    };
    bool last = false;
    while (!err && !last) {
        in.refill();
        last = in.take(1);
        const int type = (int)in.take(2);
        if (type == 0) {                                                   // stored
            in.drop(in.cnt & 7);
            in.refill();
            const uint32_t len = in.take(16), nlen = in.take(16);
            if ((len ^ 0xFFFFu) != nlen) { err = S2D_PNG_BAD_DEFLATE; break; }
            const int64_t p0 = in.consumed_bytes();                        // whole bytes left in the buffer go back
            in.pos = p0; in.buf = 0; in.cnt = 0;
            if (p0 + len > in.end) { err = S2D_PNG_BAD_DEFLATE; break; }
            if (opos + npend + len > rawsize) { err = S2D_PNG_BAD_SIZE; break; }
            flush();
            for (uint32_t i = lane; i < len; i += 32) { S2D_DEV_ASSERT(opos + i < rawsize); out[opos + i] = zdata[p0 + i]; }
            opos += len;
            in.pos += len;
            __syncwarp();
            continue;
        }
        if (type == 3) { err = S2D_PNG_BAD_DEFLATE; break; }
        int nlen = 288, ndist = 32;
        if (type == 1) {
            for (int i = lane; i < 320; i += 32) s.lens[i] = i < 144 ? 8 : i < 256 ? 9 : i < 280 ? 7 : i < 288 ? 8 : 5;
            __syncwarp();
        } else {                                                           // dynamic: code lengths, then the two codes
            nlen = (int)in.take(5) + 257;
            ndist = (int)in.take(5) + 1;
            const int ncl = (int)in.take(4) + 4;
            if (nlen > 286 || ndist > 30) { err = S2D_PNG_BAD_DEFLATE; break; }
            in.refill();
            if (lane < 19) s.lens[lane] = 0;
            __syncwarp();
            for (int i = 0; i < ncl; ++i) {
                in.refill();
                const uint32_t l = in.take(3);
                if (lane == 0) s.lens[c_clen_order[i]] = (uint8_t)l;
            }
            __syncwarp();
            if (!build_table(s, s.lens, 19, s.lit, PI_CROOT, 1 << PI_CROOT, lane)) { err = S2D_PNG_BAD_DEFLATE; break; }
            // the code-length table lives in lit; decode the lengths into lens[0, nlen + ndist)
            int i = 0;
            while (i < nlen + ndist) {
                in.refill();
                const int sym = decode_sym(in, s.lit, PI_CROOT, 1 << PI_CROOT);
                if (sym < 0) { err = S2D_PNG_BAD_DEFLATE; break; }
                if (sym < 16) {
                    if (lane == 0) { S2D_DEV_ASSERT(i < 320); s.lens[i] = (uint8_t)sym; }
                    ++i;
                    continue;
                }
                int rep, v = 0;
                if (sym == 16) {
                    if (i == 0) { err = S2D_PNG_BAD_DEFLATE; break; }
                    __syncwarp();
                    v = s.lens[i - 1];
                    rep = 3 + (int)in.take(2);
                } else if (sym == 17) rep = 3 + (int)in.take(3);
                else rep = 11 + (int)in.take(7);
                if (i + rep > nlen + ndist) { err = S2D_PNG_BAD_DEFLATE; break; }
                __syncwarp();
                for (int k = lane; k < rep; k += 32) { S2D_DEV_ASSERT(i + k < 320); s.lens[i + k] = (uint8_t)v; }
                i += rep;
            }
            __syncwarp();
            if (err) break;
            if (s.lens[256] == 0) { err = S2D_PNG_BAD_DEFLATE; break; }   // no end-of-block code
        }
        if (!build_table(s, s.lens, nlen, s.lit, PI_LROOT, PI_LENOUGH, lane) ||
            !build_table(s, s.lens + nlen, ndist, s.dist, PI_DROOT, PI_DENOUGH, lane)) { err = S2D_PNG_BAD_DEFLATE; break; }
        for (;;) {                                                         // symbols of the block
            in.refill();
            if (in.overrun()) { err = S2D_PNG_BAD_DEFLATE; break; }
            const int sym = decode_sym(in, s.lit, PI_LROOT, PI_LENOUGH);
            if (sym < 0 || sym > 285) { err = S2D_PNG_BAD_DEFLATE; break; }
            if (sym < 256) {
                if (opos + npend >= rawsize) { err = S2D_PNG_BAD_SIZE; break; }
                if (lane == npend) pend = (uint32_t)sym;
                if (++npend == 32) flush();
                continue;
            }
            if (sym == 256) break;
            const int li = sym - 257;
            const int len = c_len_base[li] + (int)in.take(c_len_extra[li]);
            in.refill();
            const int ds = decode_sym(in, s.dist, PI_DROOT, PI_DENOUGH);
            if (ds < 0 || ds > 29) { err = S2D_PNG_BAD_DEFLATE; break; }
            const int dist = c_dist_base[ds] + (int)in.take(c_dist_extra[ds]);
            flush();
            if (dist > opos || dist > window) { err = S2D_PNG_BAD_DEFLATE; break; }
            if (opos + len > rawsize) { err = S2D_PNG_BAD_SIZE; break; }
            uint8_t* __restrict__ dst = out + opos;
            const uint8_t* src = dst - dist;
            if (dist < 32) {                                               // periodic: every lane reads the dist source bytes
                const int step = 32 % dist;
                int j = lane % dist;
                for (int k = lane; k < len; k += 32) {
                    S2D_DEV_ASSERT(opos + k < rawsize && opos - dist + j >= 0 && j < dist);
                    dst[k] = src[j];
                    j += step; if (j >= dist) j -= dist;
                }
            } else {
                for (int b = 0; b < len; b += dist) {                      // dist >= 32 bytes per dependent step
                    const int e = min(len, b + dist);
                    for (int k = b + lane; k < e; k += 32) { S2D_DEV_ASSERT(opos + k < rawsize && opos - dist + k >= 0); dst[k] = src[k]; }
                    __syncwarp();
                }
            }
            opos += len;
            __syncwarp();
        }
        flush();
    }
    uint32_t adler = 0;
    if (!err) {                                                            // byte-aligned big-endian adler32, then the end
        in.drop(in.cnt & 7);
        in.refill();
        for (int k = 0; k < 4; ++k) adler = (adler << 8) | in.take(8);
        if (in.consumed_bytes() != in.end) err = S2D_PNG_BAD_DEFLATE;
        else if (opos != rawsize) err = S2D_PNG_BAD_SIZE;
    }
    if (lane == 0) { status[n] = err; adler_out[n] = adler; }
}

__global__ void __launch_bounds__(32)
png_unfilter_kernel(const s2d_png_desc* __restrict__ descs, int N, const uint8_t* __restrict__ raw_base,
                    const uint32_t* __restrict__ adler_in, uint8_t* __restrict__ rgb_out, int32_t* __restrict__ status) {
    __shared__ __align__(16) uint8_t row[S2D_PNG_MAX_ROWBYTES];
    __shared__ uint8_t pal[768];
    const int n = blockIdx.x, lane = threadIdx.x;
    if (n >= N || status[n] != 0) return;
    const s2d_png_desc& d = descs[n];
    const int rb = png_rowbytes(d);
    if (rb < 0) return;
    const int W = d.width, H = d.height, ct = d.color_type, bd = d.bit_depth;
    const int bpp = max(1, png_channels(ct) * bd / 8);
    const int64_t rawsize = (int64_t)H * (rb + 1);
    const uint8_t* __restrict__ raw = raw_base + d.raw_offset;
    uint8_t* __restrict__ dst = rgb_out + d.rgb_offset;
    for (int i = lane; i < rb; i += 32) row[i] = 0;
    if (ct == 3) for (int i = lane; i < 768; i += 32) pal[i] = i < 3 * d.palette_size ? d.palette[i] : 0;
    __syncwarp();
    uint64_t sa = 0, sb = 0;                                               // adler32 parts of this lane's bytes
    bool bad_index = false;
    int err = 0;
    for (int y = 0; y < H; ++y) {
        const int64_t r0 = (int64_t)y * (rb + 1);
        const int f = raw[r0];
        if (lane == 0) { sa += f; sb += (uint64_t)(rawsize - r0) * f; }
        if (f > 4) { err = S2D_PNG_BAD_FILTER; break; }
        if (f <= 2) {
            uint32_t prev_out = 0;
            for (int x0 = 0; x0 < rb; x0 += 32) {
                const int x = x0 + lane;
                const uint32_t v = x < rb ? raw[r0 + 1 + x] : 0u;
                sa += v; sb += (uint64_t)(rawsize - (r0 + 1 + x)) * v;
                uint32_t o = v;
                if (f == 1) {                                              // Sub: stride-bpp scan + carry
#pragma unroll 1
                    for (int k = bpp; k < 32; k <<= 1) { const uint32_t u = __shfl_up_sync(0xffffffffu, o, k); if (lane >= k) o += u; }
                    const uint32_t c = __shfl_sync(0xffffffffu, prev_out, 32 - bpp + lane % bpp);
                    o += x0 ? c : 0u;
                } else if (f == 2 && x < rb) {
                    S2D_DEV_ASSERT(x < S2D_PNG_MAX_ROWBYTES);
                    o += row[x];
                }
                o &= 0xFF;
                prev_out = o;
                if (x < rb) { S2D_DEV_ASSERT(x < S2D_PNG_MAX_ROWBYTES); row[x] = (uint8_t)o; }
            }
        } else if (lane < bpp) {                                           // Avg / Paeth: serial along the row
            uint32_t a = 0, c = 0;
            for (int x = lane; x < rb; x += bpp) {
                S2D_DEV_ASSERT(x < S2D_PNG_MAX_ROWBYTES);
                const uint32_t v = raw[r0 + 1 + x], b = row[x];
                sa += v; sb += (uint64_t)(rawsize - (r0 + 1 + x)) * v;
                uint32_t pred;
                if (f == 3) pred = (a + b) >> 1;
                else {
                    const int p = (int)a + (int)b - (int)c, pa = abs(p - (int)a), pb = abs(p - (int)b), pc = abs(p - (int)c);
                    pred = (pa <= pb && pa <= pc) ? a : pb <= pc ? b : c;
                }
                const uint32_t o = (v + pred) & 0xFF;
                row[x] = (uint8_t)o;
                a = o; c = b;
            }
        }
        sa %= 65521u; sb %= 65521u;
        __syncwarp();
        uint8_t* __restrict__ drow = dst + (int64_t)y * W * 3;
        for (int x = lane; x < W; x += 32) {                                // convert the row
            uint32_t r, g, b;
            if (bd < 8) {
                const int bit = x * bd;
                S2D_DEV_ASSERT((bit >> 3) < rb);
                const uint32_t v = (row[bit >> 3] >> (8 - bd - (bit & 7))) & ((1u << bd) - 1u);
                if (ct == 3) {
                    bad_index |= (int)v >= d.palette_size;
                    r = pal[3 * v]; g = pal[3 * v + 1]; b = pal[3 * v + 2];
                } else r = g = b = v * (bd == 1 ? 255u : bd == 2 ? 85u : 17u);
            } else {
                const int sbytes = bd / 8, px = x * png_channels(ct) * sbytes;   // high byte of each sample
                S2D_DEV_ASSERT(px + (ct == 2 || ct == 6 ? 2 * sbytes : 0) < rb);
                if (ct == 3) {
                    const uint32_t v = row[px];
                    bad_index |= (int)v >= d.palette_size;
                    r = pal[3 * v]; g = pal[3 * v + 1]; b = pal[3 * v + 2];
                } else if (ct == 0 || ct == 4) r = g = b = row[px];
                else { r = row[px]; g = row[px + sbytes]; b = row[px + 2 * sbytes]; }
            }
            S2D_DEV_ASSERT((int64_t)y * W * 3 + 3 * x + 2 < (int64_t)H * W * 3);
            drow[3 * x] = (uint8_t)r; drow[3 * x + 1] = (uint8_t)g; drow[3 * x + 2] = (uint8_t)b;
        }
        __syncwarp();
    }
    if (!err) {
        const uint32_t A = (1u + __reduce_add_sync(0xffffffffu, (uint32_t)sa)) % 65521u;
        const uint32_t B = (uint32_t)((rawsize % 65521 + __reduce_add_sync(0xffffffffu, (uint32_t)sb)) % 65521u);
        if (((B << 16) | A) != adler_in[n]) err = S2D_PNG_BAD_ADLER;
    }
    if (__any_sync(0xffffffffu, bad_index)) err |= S2D_PNG_BAD_INDEX;
    if (lane == 0 && err) status[n] = err;
}

}  // namespace s2d

using namespace s2d;

static int64_t png_scratch_base_ints(int N) { return ((int64_t)N + 3) / 4 * 4; }   // adler32 words, then 16-byte aligned bytes

extern "C" int s2d_png_decode_work_ints(int N, int64_t raw_bytes, int64_t* out) {
    S2D_CHECK_ARG(out && N > 0 && raw_bytes >= 0, "s2d_png_decode_work_ints: bad arguments");
    *out = png_scratch_base_ints(N) + (raw_bytes + 3) / 4;
    return 0;
}

extern "C" int s2d_png_decode(const uint8_t* zdata, const int64_t* z_offsets, const s2d_png_desc* descs, int N,
                              int32_t* work, uint8_t* rgb_out, int32_t* status, void* stream) {
    S2D_ENTER(stream);
    S2D_CHECK_ARG(zdata && z_offsets && descs && work && rgb_out && status, "s2d_png_decode: null pointer");
    S2D_CHECK_ARG(N > 0, "s2d_png_decode: bad sizes");
    S2D_CHECK_ARG(reinterpret_cast<uintptr_t>(work) % 16 == 0 && reinterpret_cast<uintptr_t>(descs) % 8 == 0,
                  "s2d_png_decode: work must be 16-byte and descs 8-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    uint32_t* adler = reinterpret_cast<uint32_t*>(work);
    uint8_t* raw = reinterpret_cast<uint8_t*>(work + png_scratch_base_ints(N));
    png_inflate_kernel<<<(unsigned)((N + PI_WARPS - 1) / PI_WARPS), PI_WARPS * 32, 0, st>>>(zdata, z_offsets, descs, N, raw,
                                                                                           adler, status);
    S2D_CHECK_LAUNCH("png_inflate_kernel");
    png_unfilter_kernel<<<(unsigned)N, 32, 0, st>>>(descs, N, raw, adler, rgb_out, status);
    S2D_CHECK_LAUNCH("png_unfilter_kernel");
    return 0;
}
