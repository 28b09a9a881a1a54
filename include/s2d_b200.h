/* s2d_b200 - C ABI of the B200-native keymask-discovery hot path.
 *
 * Drop-in boundary for the arithmetic underneath the reference's per-video loop
 * (leonsick/s2d keymask_ident/main_keymask_ident.py:81-139). The reference has no FFI of its own
 * (it is pure Python); each entry point below names the reference code it replaces. A Python
 * maintainer binds these with ctypes (see INTEGRATION.md and s2d_b200/_lib.py).
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error; s2d_last_error() gives the message
 *     (thread-local). No exceptions cross the boundary, nothing is allocated inside: all
 *     buffers are caller-owned DEVICE pointers unless the name says `host`.
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing syncs.
 *   - work is batched over videos: `descs` is a DEVICE array of `nvideos` s2d_video_desc that
 *     places each video inside the batch-wide buffers (layout below). Videos may differ in every
 *     dimension.
 *
 * Inputs are referenced per video by absolute device pointers in the descriptor (the producer's
 * own buffers: nothing is concatenated or copied). Workspace and outputs are batch-wide buffers;
 * the descriptor holds each video's element offset into them:
 *   per-(row,frame) arrays  [Nm][T]   cnt i32, V f32, uniq i32                @ vt_off
 *   hits     i32  [Nm][T][L]                                                  @ hits_off
 *   xbits / winbits / majbits / rsbits / rebits   u32 [Nm][TW]                @ xbits_off
 *   mbits    u32  [Nm][NW]            match matrix rows (bit g = target gid)  @ mbits_off
 *   per-row arrays [row0 + q]         qframe, qlabel, labels1, rowinfo (int4), one2x, glabel ...
 *   per-frame arrays [frame0 + t]     area i32 [256], gid_of i32 [256], frameinfo (int4)
 *   per-video arrays [v]              vidinfo i32 [S2D_VIDINFO_WORDS]
 *   per-(video,cluster) arrays        [v][S2D_MAX_CLUSTERS] clusterinfo i32 [S2D_CLINFO_WORDS]
 */
#ifndef S2D_B200_H
#define S2D_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define S2D_MAX_LABELS 256      /* label ids are u8 */
#define S2D_MAX_CLUSTERS 16     /* visibility clusters carried into stage D (>=11 fails the video) */
#define S2D_VIDINFO_WORDS 8
#define S2D_CLINFO_WORDS 16

#define S2D_DESC_VIS_BITS 1     /* desc.flags: `vis` is bit-packed by the producer (1/8 of the flag bytes on the wire) */

typedef struct s2d_video_desc {
    int32_t T, H, W, P;
    int32_t Nm;          /* rows = (frame,label) queries of this video                      */
    int32_t L;           /* histogram bins kept per (q,t): max label + 1, <= 256            */
    int32_t TW;          /* words per frame-bit row  = ceil(T / 32)                         */
    int32_t NW;          /* words per match-bit row  = ceil(Nm / 32)                        */
    int64_t row0;        /* first row in batch-wide per-row arrays                          */
    int64_t frame0;      /* first frame in batch-wide per-frame arrays                      */
    const uint8_t* labels;  /* device, u8  [T][H][W]      label maps, 0 = background          */
    const float*   tracks;  /* device, f32 [Nm][T][P][2]  CoTracker pred_tracks (x, y)        */
    const uint8_t* vis;     /* device, u8  [Nm][T][P]     CoTracker pred_visibility bytes; with     */
                            /* S2D_DESC_VIS_BITS: u32 [Nm][T][ceil(P/32)], bit p%32 of word p/32 = flag p */
    const int32_t* npts;    /* device, i32 [Nm] valid points per query (<= P) or NULL = all P  */
    const int32_t* tstart;  /* device, i32 [Nm] first frame stored in `tracks` per query, NULL = 0:  */
    int32_t Ttr;            /* tracks is [Nm][Ttr][P][2]; Ttr == T unless only the window is stored */
    int32_t flags;          /* S2D_DESC_* bits (long videos: SA-V-shaped configs keep Tw <= 64 frames per query) */
    int64_t vt_off;      /* elements of [Nm][T] arrays                                       */
    int64_t hits_off;    /* int32 elements                                                   */
    int64_t xbits_off;   /* u32 words of [Nm][TW] arrays                                     */
    int64_t mbits_off;   /* u32 words of [Nm][NW] arrays                                     */
} s2d_video_desc;

/* rowinfo int4: x = visibility cluster id (-1 noise), y = candidate run index (-1 = not a
 * candidate), z = v0, w = v1 (merged window of the cluster, cotracker_matching.py:1033-1038) */
/* frameinfo int4: x = number of objects (present labels minus the smallest), y = first gid of
 * the frame, z = smallest present label (dropped, cotracker_matching.py:294), w = #present   */
/* vidinfo: [0] nclusters (DBSCAN #1), [1] status after stage B (1 ok, -1 fail),
 *          [2] max matched gid (cotracker_matching.py:770-773), [3] final status (1 / -1),
 *          [4] number of candidate queries, [5] number of rows (check)                     */
/* clusterinfo: [0] size, [1] #candidates, [2] v0, [3] v1, [4] #runs, [5] row_min, [6] row_max,
 *          [7] col_min, [8] col_max, [9] kmax, [10] min_samples, [11] factor,
 *          [12] matched rows (coverage numerator), [13] one2x sum over queries, [14] #queries */

const char* s2d_last_error(void);
int s2d_version(void);
int s2d_desc_size(void);            /* sizeof(s2d_video_desc), for binding self-checks */
int s2d_device_sm_count(int device);

/* Host-side helpers of the end-to-end path (host buffers -> device -> results). s2d_host_register page-locks a
 * caller-allocated host range (e.g. an mmap'ed, huge-page backed staging pool placed on the GPU's NUMA node) so that
 * cudaMemcpyAsync from it is a true asynchronous DMA; s2d_device_pci_bus_id writes "dddd:bb:dd.f" of a device (its sysfs
 * node gives the NUMA node: /sys/bus/pci/devices/<id>/numa_node). The reference has no counterpart: it copies per call
 * from pageable memory (cotracker_occlusions.py:346-356). */
int s2d_host_register(void* ptr, int64_t bytes);
int s2d_host_unregister(void* ptr);
int s2d_device_pci_bus_id(int device, char* out, int len);

/* All `max_*` / `total_*` arguments are host-side bounds over the batch (grid sizing and memset
 * extents): max_T = max frames, max_npix = max H*W, max_rows_x_T = max Nm*T, total_rows = sum Nm,
 * total_frames = sum T, total_vt = sum Nm*T ... */

/* K0. Per-frame label histogram + object enumeration + global ids.
 * Replaces torch.unique(label[t])[1:] (cotracker_occlusions.py:337-338, cotracker_matching.py:
 * 294-295, 682-683) and contruct_frameid_maskid_lookup (cotracker_matching.py:289-306).
 * Outputs area[frame][256], gid_of[frame][256] (-1 = not an object), frameinfo[frame] (int4),
 * qframe/qlabel[row]; vidinfo[5] receives the enumerated row count (must equal desc.Nm). */
int s2d_label_stats(const s2d_video_desc* descs, int nvideos, int max_T, int64_t max_npix,
                    int64_t total_frames, int32_t* area, int32_t* gid_of,
                    int32_t* frameinfo, int32_t* qframe, int32_t* qlabel, int32_t* vidinfo,
                    void* stream);

/* K3a. Visibility reduce: cnt[q,t] = #nonzero flags, V = float32(cnt) / float32(P) (IEEE
 * division), replaces torch.mean(pred_visibility.float(), dim=2) (cotracker_occlusions.py:359).
 * Videos flagged S2D_DESC_VIS_BITS hand the flags over bit-packed (u32 words, 4-byte aligned rows of ceil(P/32)
 * words; bits at positions >= P of a row's last word are ignored): same counts from 1/8 of the bytes. */
int s2d_vis_reduce(const s2d_video_desc* descs, int nvideos, int64_t max_rows_x_T,
                   int32_t* cnt, float* V, void* stream);

/* K3 binarise: xbits[row] bit t = V[row,t] > thr (float32 compare,
 * identify_visibility_windows.py:114,119). */
int s2d_binarize(const s2d_video_desc* descs, int nvideos, int64_t max_rows_x_TW, const float* V,
                 float visibility_threshold, uint32_t* xbits, void* stream);

/* K3b. Hamming DBSCAN #1 over the rows of xbits, eps 0.2 / min_samples 5 in the reference
 * (identify_visibility_windows.py:114; sklearn.cluster.DBSCAN(metric="hamming")).
 * work: int32 scratch of s2d_dbscan_work_ints(total_rows, nvideos) elements, 8-byte aligned.
 * labels1[row] = cluster id or -1; vidinfo[0] = number of clusters. */
int s2d_dbscan_work_ints(int64_t total_rows, int nproblems, int64_t* out);
int s2d_dbscan_visibility(const s2d_video_desc* descs, int nvideos, int max_Nm, int max_TW,
                          int64_t total_rows, const uint32_t* xbits, double eps, int min_samples,
                          int32_t* work, int32_t* labels1, int32_t* vidinfo, void* stream);

/* K3c. Majority vote, run-length windows, highly-visible rows, candidates
 * (identify_visibility_windows.py:134-203; get_visible_ranges :65-88;
 * get_highly_visible_rows :90-105). Per cluster c (slot c of the video's [Nm][TW] arrays):
 * majbits, rsbits (run starts), rebits (run ends); clrow[row0+c] int4 = (size, #runs, v0, v1).
 * Per row: winbits (bit r = winner of run r), rowinfo. Per video: vidinfo[1..4], clusterinfo
 * for the first S2D_MAX_CLUSTERS clusters. ccount: int32 scratch [Nm][T] @ vt_off. T <= 1024. */
int s2d_windows(const s2d_video_desc* descs, int nvideos, int64_t max_rows_x_TW, int max_TW,
                int64_t total_rows, int64_t total_vt, const uint32_t* xbits,
                const int32_t* labels1, const int32_t* qframe, float winner_fraction,
                int32_t* ccount, int32_t* clrow, uint32_t* majbits, uint32_t* rsbits,
                uint32_t* rebits, uint32_t* winbits, int32_t* rowinfo, int32_t* vidinfo,
                int32_t* clusterinfo, void* stream);

/* K2. Point-in-mask voting for every candidate query q and every frame t of its window:
 *   uniq[q,t]      = # distinct in-bounds pixels of round-half-even(tracks[q,t])
 *   hits[q,t,lab]  = # of those pixels whose label is lab
 * Replaces pred_tracks_to_binary_masks + compute_point_mask_intersection for all masks of the
 * frame (cotracker_matching.py:453-503, 640-662, 665-692). Rows whose rowinfo.y < 0, frames
 * outside [v0,v1] and videos whose vidinfo[1] < 0 are skipped (hits/uniq left untouched).
 * rowinfo == NULL votes every (q,t); vidinfo == NULL ignores the stage-B status.
 * vec4_ok != 0 promises P even and 16-byte aligned tracks for every video (128-bit loads).
 * work: int32 scratch of s2d_point_votes_work_ints(total_rows) elements, 16-byte aligned; with it
 * (and vec4_ok, P <= 16384) a persistent kernel runs: a device-side plan lists the (row, frame)
 * tiles and 2-4 CTAs per SM stream them through cp.async.bulk. Variant 0 (default) pulls the
 * tile's bounding box of the label map into shared memory and resolves de-duplication and label
 * lookup with one shared-memory atomic per point; variant 2 (also used when work == NULL or the promises above
 * do not hold) is the one-CTA-per-tile kernel. All variants give identical results.
 * H, W <= 65535; P <= 32768.
 * Alignment / slack: when a video's label maps are fetched row by row (no descriptors: W or the base address
 * not a multiple of 16) each row copy is widened to whole 16-byte blocks, so up to 15 bytes before `labels` and
 * after its last byte are READ (never used): the buffer must sit inside an allocation that extends to the
 * enclosing 16-byte boundaries on both sides (any cudaMalloc / framework allocation does; an exact-size
 * sub-allocation at the very edge of a mapping does not).
 * Device: every entry point makes the device of `stream` current for the duration of the call (and restores the
 * caller's afterwards), so a caller may drive several GPUs from one thread; descs and all buffers must live on
 * that device.
 * label_tmaps (optional, may be NULL): DEVICE copy (64-byte aligned) of the buffer that
 * s2d_point_votes_tmaps fills on the HOST from a host copy of the descriptors - S2D_PV_TMAP_BYTES
 * per video: TMA descriptors of the video's label maps, so that variant 0 fetches a tile's table
 * as a few 2D boxes instead of one bulk copy per row. Videos whose W or label base address is not
 * a multiple of 16 get no descriptors and keep the row-by-row fetch. */
#define S2D_PV_TMAPS 32                            /* box widths 16, 32, ... 512 pixels, 16 rows each */
#define S2D_PV_TMAP_BYTES (S2D_PV_TMAPS * 128 + 128)
int s2d_point_votes_variant(int variant);   /* process-wide, for tests and A/B runs; 0 product dispatch, 2 one CTA per tile,
                                             * 3 label table for every P, 4 one warp per tile for every frame size (P <= 1024)
                                             * (1, the superseded bitmap kernel, only exists in the experiments build: make exp) */
int s2d_point_votes_work_ints(int64_t total_rows, int64_t* out);
int s2d_point_votes_tmaps(const s2d_video_desc* host_descs, int nvideos, void* host_out);
int s2d_point_votes(const s2d_video_desc* descs, int nvideos, int max_T, int max_Nm, int max_P,
                    int vec4_ok, int64_t total_rows, const int32_t* rowinfo, const int32_t* vidinfo,
                    int32_t* work, const void* label_tmaps, int32_t* hits, int32_t* uniq, void* stream);

/* s2d_point_votes with the size of the largest frame of the batch (H * W pixels; 0 = unknown = s2d_point_votes): batches of
 * <= 1024 tracked points per query on frames of up to 512 Ki pixels (480 x 854) run the one-warp-per-tile kernel instead of
 * the label-table kernel (measured: 40 % instead of 31 % of the HBM copy peak on 480p videos; larger frames keep the table
 * kernel, whose cost does not grow with the bounding box). Results are identical either way. */
int s2d_point_votes_sized(const s2d_video_desc* descs, int nvideos, int max_T, int max_Nm, int max_P,
                          int vec4_ok, int64_t total_rows, const int32_t* rowinfo, const int32_t* vidinfo,
                          int32_t* work, const void* label_tmaps, int64_t max_frame_pixels, int32_t* hits, int32_t* uniq,
                          void* stream);

/* K3d. Appearance events of visibility curves V f32 [N][T] (device): moving average of odd length
 * smoothing_window (reflect padding), `>= thresh`, morphological opening with window
 * min_run_length (erosion then dilation as reflect-padded min / max pooling; for even windows each
 * pooling shortens the signal by one sample, like the reference), then the 0->1 / 1->0 transitions
 * of the opened signal compacted per row with warp ballots: nstart[row], nend[row] and the first
 * max_events frame indices of each kind in starts / ends [N][max_events]. opened (optional,
 * u8 [N][T], first T2 columns written) receives the opened signal. Replaces
 * extract_appearance_events (cotracker_occlusions.py:166-223 == cotracker_matching.py:212-269);
 * bit-exact for smoothing_window == 1 (the default), float32 fma accumulation otherwise.
 * s2d_boolean_visibility: out[i] = V[i] >= threshold (cotracker_occlusions.py:226-240). */
int s2d_appearance_events(const float* V, int N, int T, int smoothing_window, float thresh,
                          int min_run_length, int max_events, int32_t* nstart, int32_t* nend,
                          int32_t* starts, int32_t* ends, uint8_t* opened, void* stream);
int s2d_boolean_visibility(const float* V, int64_t n, float threshold, uint8_t* out, void* stream);

/* f2. COCO run-length encoding of N binary masks (u8 [N][H][W] row-major, non-zero = set) with area
 * and bounding box: what annotations.py:94-106 and convert_results_to_annotations.py:70-81 obtain from
 * pycocotools (maskApi.c rleEncode / rleArea / rleToBbox). counts [N][max_runs] receives the run
 * lengths in COLUMN-major order starting with a run of zeros (possibly of length 0); nruns[n] is the
 * true number of runs - when it exceeds max_runs only the first max_runs were written and the caller
 * repeats the call with a larger bound. area[n] = set pixels; bbox[n] = (xmin, ymin, xmax, ymax)
 * inclusive, (INT_MAX, INT_MAX, -1, -1) for an empty mask. work: s2d_rle_work_ints() int32. The
 * base-48 string packing of the counts (rleToString) is a host-side pass over the short count list. */
int s2d_rle_work_ints(int N, int H, int W, int max_runs, int64_t* out);
int s2d_rle_encode(const uint8_t* masks, int N, int H, int W, int max_runs, int32_t* work,
                   int32_t* counts, int32_t* nruns, int32_t* area, int32_t* bbox, void* stream);

/* Area and bounding box of N run-length encodings without decoding them (maskApi.c rleArea /
 * rleToBbox, as convert_results_to_annotations.py:70-81 calls them per predicted segmentation).
 * counts: the RLEs' run lengths back to back (device int32), offsets [N+1] (device int64) the start
 * of each, heights [N] the mask heights. area[n] = sum of the odd runs, bbox[n] = (x, y, w, h). */
int s2d_rle_area_bbox(const int32_t* counts, const int64_t* offsets, int N, const int32_t* heights,
                      int32_t* area, int32_t* bbox, void* stream);

/* Stage E on the device: COCO RLE of every keymask row straight from the label maps, without materialising a mask
 * plane per keymask. Replaces the per-keymask mask_util.encode / toBbox of annotations.py:94-106 (maskApi.c rleEncode)
 * for a whole batch. Row g = (frame, label) as K0 enumerates them in gid_of; only videos whose vidinfo[3] (final
 * status) is 1 are encoded - the reference writes no annotation for the others, and their rows get no runs.
 *   counts   int32, the rows' run lengths back to back: column-major, starting with a run of zeros (of length 0
 *            when pixel (0, 0) is set), exactly what rleEncode produces for labels[f] == l
 *   offsets  int64 [total_rows + 1]: row g's runs are counts[offsets[g] .. offsets[g + 1])
 *   bbox     int32 [total_rows][4] = xmin, ymin, xmax, ymax (inclusive) of the mask; the area is K0's area[f][l]
 *   needed   int64 [1] = offsets[total_rows], the counts the batch needs. Nothing is written at or past `capacity`;
 *            when *needed > capacity the caller re-runs with a larger buffer (rows past the capacity are incomplete).
 * Each frame's label bytes are read twice whatever the number of objects (a transition a -> b in column-major order is
 * an edge of mask a and of mask b). Needs K0's gid_of and the final status of K4 (vidinfo) on the device: no host
 * round trip, so the call can be captured in a CUDA graph. H * W < 2^31, H <= 65535. work: int32 scratch of
 * s2d_label_rle_work_ints(total_frames, total_rows, max_H, max_W) elements. */
int s2d_label_rle_work_ints(int64_t total_frames, int64_t total_rows, int max_H, int max_W, int64_t* out);
int s2d_label_rle(const s2d_video_desc* descs, int nvideos, int max_T, int max_H, int max_W, int max_Nm,
                  int64_t total_frames, int64_t total_rows, const int32_t* gid_of, const int32_t* vidinfo,
                  int32_t* work, int64_t capacity, int32_t* counts, int64_t* offsets, int32_t* bbox,
                  int64_t* needed, void* stream);

/* COCO compressed-RLE strings of N run-length lists on the device (maskApi.c rleToString, as annotations.py:100 gets
 * them through mask_util.encode): counts / offsets [N + 1] in the layout above (lists that end past `ncounts`, the
 * valid length of counts, give empty strings). chars receives the strings back to back, str_offsets [N + 1] (int64)
 * where each starts, *needed the total length; nothing is written at or past `capacity` (re-run when *needed >
 * capacity). Byte-identical to the reference's packing. work: int32 scratch of N elements. */
int s2d_rle_strings(const int32_t* counts, const int64_t* offsets, int N, int64_t ncounts, int32_t* work,
                    int64_t capacity, char* chars, int64_t* str_offsets, int64_t* needed, void* stream);

/* The inverse of s2d_rle_strings: run-length lists of N COCO compressed-RLE strings on the device (maskApi.c rleFrString,
 * which every consumer of the annotations calls through mask_util.decode before it has a mask; annotations.py:94-106 and
 * convert_results_to_annotations.py:70-81 produce and read these strings). chars: the strings back to back, string n at
 * chars[str_offsets[n] .. str_offsets[n + 1]) (str_offsets int64 [N + 1], on the device). A value ends at a character
 * whose bit 0x20 is clear (c = byte - 48, for every byte as maskApi computes it); its 5-bit groups are sign-extended from
 * bit 0x10 of the last; count m > 2 is the value plus count m - 2.
 *   counts         int32, the lists back to back, list n at counts[count_offsets[n] .. count_offsets[n + 1])
 *   count_offsets  int64 [N + 1];  *needed = count_offsets[N], the total number of counts (at most the number of
 *                  characters). Nothing is written at or past `capacity` (re-run with a larger buffer when *needed >
 *                  capacity)
 *   status         int32 [N]: 0, or 1 for a malformed string: its last character still has the continuation bit set (the
 *                  unfinished value is dropped), or a count falls outside [0, 2^31). Other strings are not affected.
 * No host round trip: the call can be captured in a CUDA graph. work: int32 scratch of
 * s2d_rle_from_strings_work_ints(N, nchars) elements. */
int s2d_rle_from_strings_work_ints(int N, int64_t nchars, int64_t* out);
int s2d_rle_from_strings(const char* chars, const int64_t* str_offsets, int N, int32_t* work, int64_t capacity,
                         int32_t* counts, int64_t* count_offsets, int32_t* status, int64_t* needed, void* stream);

/* Binary masks of N run-length lists (maskApi.c rleDecode, what mask_util.decode returns per segmentation), each on its
 * own: counts / count_offsets [N + 1] as s2d_rle_from_strings writes them (counts are read as unsigned, as maskApi does),
 * heights / widths int32 [N], out_offsets int64 [N] (all on the device). Mask n is written to
 * out + out_offsets[n] as H * W bytes, row-major, value 0 or 1 (runs are column-major, the first a run of zeros); the
 * offsets may leave gaps (frames of an [A, T, H, W] tensor without a segmentation), which are not touched. Sizes may
 * differ within one call; H, W <= 65535 and H * W < 2^31. status int32 [N] is OR-ed with 2 when the runs do not sum to
 * H * W (or the size is out of range, then nothing is written for that mask): pixels past the sum are 0 and runs past
 * H * W are ignored. No byte outside a mask's own H * W bytes is written. No host round trip: the call can be captured
 * in a CUDA graph. work: int32 scratch of s2d_rle_decode_work_ints(N, count_offsets[N]) elements, 8-byte aligned. */
int s2d_rle_decode_work_ints(int N, int64_t ncounts, int64_t* out);
int s2d_rle_decode(const int32_t* counts, const int64_t* count_offsets, int N, const int32_t* heights,
                   const int32_t* widths, const int64_t* out_offsets, int32_t* work, uint8_t* out, int32_t* status,
                   void* stream);

/* PNG label maps (the colour-coded mask frames every video starts from) decoded to packed RGB on the device: what
 * cv2.imread(path, IMREAD_COLOR) returns in load_masks / load_image_robust (crw_utils.py:310-346, 714-767,
 * cotracker_occlusions.py:22-85, cotracker_matching.py:22-84), in RGB order, for non-interlaced files. The host parses
 * the chunks; this call inflates each file's zlib stream (a warp per file: stored, fixed- and dynamic-Huffman blocks),
 * undoes the row filters and converts each row: palette lookup, gray replicated to R = G = B (1/2/4-bit gray scaled to
 * 0-255), 1/2/4-bit samples unpacked, 16-bit samples reduced to their high byte, alpha and tRNS dropped.
 *   zdata       the files' IDAT payloads joined, file n at zdata[z_offsets[n] .. z_offsets[n + 1]) (z_offsets int64
 *               [N + 1]), the 2-byte zlib header and the adler32 trailer included
 *   descs       s2d_png_desc [N] (on the device, 8-byte aligned): the IHDR fields, the palette, and where the file's
 *               filtered scanlines (H * (1 + rowbytes) bytes, in the work area) and its RGB frame (H * W * 3 bytes,
 *               row-major, at rgb_out + rgb_offset) go. Ranges of different files must not overlap; sizes may differ.
 *   status      int32 [N], written for every file: 0, or an OR of the S2D_PNG_BAD_* bits. A flagged file's RGB range
 *               holds no defined pixels; other files are not affected. No byte outside a file's own ranges is written.
 * No host round trip: the call can be captured in a CUDA graph. work: int32 scratch of
 * s2d_png_decode_work_ints(N, raw_bytes) elements, 16-byte aligned, where raw_bytes covers every file's
 * raw_offset + H * (1 + rowbytes). */
#define S2D_PNG_MAX_ROWBYTES 16384            /* wider rows (and frames above S2D_PNG_MAX_RAW_BYTES) get S2D_PNG_BAD_DESC */
#define S2D_PNG_MAX_RAW_BYTES (1 << 30)
#define S2D_PNG_BAD_DEFLATE 1                 /* zlib header, block type, code, symbol 286/287, distance 30/31 or one
                                                 reaching before the stream's start or past its window; data short of
                                                 the final block or left after the adler32 */
#define S2D_PNG_BAD_SIZE 2                    /* the stream ends short of, or would run past, H * (1 + rowbytes) bytes */
#define S2D_PNG_BAD_FILTER 4                  /* a filter byte greater than 4 */
#define S2D_PNG_BAD_ADLER 8                   /* adler32 mismatch */
#define S2D_PNG_BAD_DESC 16                   /* (colour type, bit depth) pair, size or palette size out of range */
#define S2D_PNG_BAD_INDEX 32                  /* a palette index at or past the palette's entries */
typedef struct s2d_png_desc {
    int32_t width, height, bit_depth, color_type;   /* IHDR; colour type 0, 2, 3, 4 or 6 */
    int64_t raw_offset;                             /* byte offset of the filtered scanlines in the work area */
    int64_t rgb_offset;                             /* byte offset of the RGB frame in rgb_out */
    int32_t palette_size;                           /* PLTE entries (colour type 3), 1-256 */
    int32_t reserved;
    uint8_t palette[768];                           /* PLTE, RGB */
} s2d_png_desc;                                     /* 808 bytes */
int s2d_png_decode_work_ints(int N, int64_t raw_bytes, int64_t* out);
int s2d_png_decode(const uint8_t* zdata, const int64_t* z_offsets, const s2d_png_desc* descs, int N, int32_t* work,
                   uint8_t* rgb_out, int32_t* status, void* stream);

/* Annotation layout of stage E: which keymask rows become which YTVIS annotation, in the reference's order
 * (annotations.py:8-140 walks `cluster_*` and `group_*` directories sorted as strings), as compact tables. Reads the
 * tables of stages L, B, D and E already on the device; only videos whose vidinfo[3] (final status) is 1 get entries.
 *   - a cluster c (< S2D_MAX_CLUSTERS) counts when one of its rows (rowinfo.x == c) is the candidate of a run r: rowinfo.y
 *     == r, r below the cluster's number of runs and winner bit r of the row set. Counted clusters are ordered as the
 *     strings cluster_{c};
 *   - its groups are the distinct glabel >= 0 of its rows, ordered as the strings group_{l} (group_10 before group_2);
 *     one annotation per group, numbered from 1 across the video;
 *   - the members of a group are its rows; of two on one frame the one with the larger label id is kept.
 * Outputs (caller-sized from host numbers; A <= total_rows annotations, M <= total_rows members, S <= the string bytes
 * s2d_rle_strings reported, K <= S2D_MAX_CLUSTERS * nvideos clusters, R <= S2D_MAX_CLUSTERS / 2 * (total_frames +
 * nvideos) range pairs; sizes int64 [5] receives A, M, S, K, R):
 *   vann        int32 [nvideos][2]  number of annotations of the video, index of its first
 *   ann         int32 [A][7]        cluster c, group l, grp_n and grp_one2x of (c, l) (the host divides them), index of the
 *                                   cluster's range list in `clusters`, first member, number of members
 *   members     int32 [M][6]        frame, bbox (xmin, ymin, xmax, ymax), area;  member_off int64 [M]: start of the member's
 *                                   string in `chars` (it ends where the next member's starts, the last at S)
 *   chars       the members' strings back to back, in (video, annotation, frame) order; nothing is written at or past
 *               `capacity`, and a string that does not lie inside rle_chars [0, nchars) is not copied (when stage E's
 *               own capacities were short the caller re-runs stage E and this call)
 *   clusters    int32 [K][2]        first pair in `pairs`, number of pairs: [start, end] of every visibility run
 *   pairs       int32 [R][2]
 * The host only slices: no decision per row is left to it. rle_bbox / str_off / rle_chars as s2d_label_rle and
 * s2d_rle_strings left them, area / gid_of of K0. No host round trip: the call can be captured in a CUDA graph.
 * work: int32 scratch of s2d_annotation_layout_work_ints(total_rows, nvideos) elements, 8-byte aligned. */
int s2d_annotation_layout_work_ints(int64_t total_rows, int nvideos, int64_t* out);
int s2d_annotation_layout(const s2d_video_desc* descs, int nvideos, int64_t total_rows, const int32_t* vidinfo,
                          const int32_t* rowinfo, const uint32_t* winbits, const uint32_t* rsbits, const uint32_t* rebits,
                          const int32_t* glabel, const int32_t* qframe, const int32_t* qlabel, const int32_t* grp_n,
                          const int32_t* grp_one2x, const int32_t* area, const int32_t* gid_of, const int32_t* rle_bbox,
                          const int64_t* str_off, const char* rle_chars, int64_t nchars, int32_t* work, int32_t* vann,
                          int32_t* ann, int32_t* members, int64_t* member_off, int32_t* clusters, int32_t* pairs,
                          int64_t capacity, char* chars, int64_t* sizes, void* stream);

/* The annotation json of stage E: for every video whose vidinfo[3] (final status) is 1, the exact text of its YTVIS
 * `annotations` list - the bytes of Python's json.dumps of the list annotations_from_layout (s2d_b200/pipeline.py)
 * builds from the same tables: default separators ", " and ": ", keys in the order video_id, iscrowd, height, width,
 * length, segmentations, bboxes, areas, category_id, id, one2x, visibility_ranges; null for a frame without a member;
 * segmentations {"size": [H, W], "counts": "..."}; boxes [x0.0, y0.0, w.0, h.0] as Python prints float(int); areas
 * and range pairs as ints; "[]" for a video without annotation. Two rules decide byte equality:
 *   - '\' (92), the only character of the RLE alphabet chr(48)..chr(111) that json escapes, is written as "\\";
 *   - one2x = repr(round(gs / gn, 2)) (0.0 when gn == 0): x = gs / gn is one IEEE double division, k = 100 x rounded
 *     half to even from x's exact binary value (1/8 -> 0.12, 3/8 -> 0.38, 1/200 -> 0.01), printed as k / 100 with
 *     trailing zeros stripped and at least one decimal. For |gs|, |gn| < 2^31 that is Python's shortest repr.
 * Inputs: the outputs of s2d_annotation_layout as they sit on the device (vann, ann, members, member_off, chars,
 * clusters, pairs, and sizes, whose counts are read on the device), T / H / W of the descriptors, vidinfo[3]. nchars is
 * the capacity the layout was given for `chars`: strings are read only below it. When stage E's string capacity was
 * short the layout's sizes[2] exceeds it and the text is incomplete (the caller re-runs stage E, the layout and this
 * call). nvideos <= 65535.
 * Output: video v's text at out + video_off[v] .. out + video_off[v + 1] (int64 [nvideos + 1]); videos whose status is
 * not 1 get an empty range. *needed = video_off[nvideos], the bytes the batch needs; nothing is written at or past
 * `capacity` (the caller re-runs this call alone with a larger buffer: its inputs are intact). Two passes with a scan
 * between them, no host round trip: the call can be captured in a CUDA graph together with the layout.
 * work: int32 scratch of s2d_annotation_json_work_ints(total_rows, nvideos) elements, 8-byte aligned. */
int s2d_annotation_json_work_ints(int64_t total_rows, int nvideos, int64_t* out);
int s2d_annotation_json(const s2d_video_desc* descs, int nvideos, int64_t total_rows, const int32_t* vidinfo,
                        const int32_t* vann, const int32_t* ann, const int32_t* members, const int64_t* member_off,
                        const char* chars, int64_t nchars, const int32_t* clusters, const int32_t* pairs,
                        const int64_t* sizes,
                        int32_t* work, int64_t capacity, char* out, int64_t* video_off, int64_t* needed, void* stream);

/* K4a. Scores and selection per candidate query: iou = hits/uniq (double), match bit when
 * iou > matching_threshold (cotracker_matching.py:710), one-to-many flag when >= one2x_frames
 * frames hold more than one mask with iou > one2x_iou (cotracker_matching.py:1082-1111).
 * mbits is cleared inside. Maintains vidinfo[2] (max matched gid, matching.py:770-773).
 * With windowed track storage (desc.tstart / desc.Ttr) only the frames [tstart[q], tstart[q] + Ttr) of a
 * query carry votes; every other frame of its [v0, v1] is scored as intersection 0 / union 0 (iou 0.0), never
 * from whatever hits / uniq held before. */
int s2d_select(const s2d_video_desc* descs, int nvideos, int max_Nm, int64_t total_mbits_words,
               const int32_t* hits, const int32_t* uniq, const int32_t* gid_of,
               const int32_t* rowinfo, double matching_threshold, double one2x_iou,
               int one2x_frames, uint32_t* mbits, int32_t* one2x, int32_t* nmatch,
               int32_t* vidinfo, void* stream);

/* K4b. Temporal-correspondence grouping: per visibility cluster crop the match matrix to its
 * bounding box, Hamming DBSCAN #2 with the reference's eps/min_samples table, zero rows -> -1,
 * factor, coverage and one2x sums (cotracker_matching.py:764-840, 843-921).
 * work: int32 scratch of s2d_group_work_ints(total_rows, nvideos) elements, 8-byte aligned.
 * glabel[row] = group label or -1; grp_n / grp_one2x: int32 [16*total_rows], slot
 * 16*row0 + c*Nm + label = rows / one2x sum of that group; vidinfo[3] = final status. */
int s2d_group_work_ints(int64_t total_rows, int nvideos, int64_t* out);
int s2d_group(const s2d_video_desc* descs, int nvideos, int max_Nm, int max_NW, int64_t total_rows,
              const uint32_t* mbits, const int32_t* rowinfo, const int32_t* one2x, int32_t* work,
              int32_t* glabel, int32_t* grp_n, int32_t* grp_one2x, int32_t* vidinfo,
              int32_t* clusterinfo, void* stream);

/* The same with the pairwise distances of large problems taken from a Gram matrix computed on the tensor cores: for a
 * video v with gram_off[v] >= 0, gram + gram_off[v] is G = X X^T (int32 [Nm][Nm]) of the video's match rows as 0/1 vectors
 * (s2d_unpack_bits + s2d_overlap_i8 on mbits), and DBSCAN #2 uses dist(a, b) = G[a][a] + G[b][b] - 2 G[a][b] instead of
 * XOR + popc over the bit rows - O(Nm^2) reads instead of O(Nm^3 / 32) bit operations (a 300-frame video has Nm = 9 000
 * rows). gram_off: DEVICE int64 [nvideos], -1 = no Gram for that video; gram / gram_off NULL = s2d_group. Same results. */
int s2d_group_gram(const s2d_video_desc* descs, int nvideos, int max_Nm, int max_NW, int64_t total_rows,
                   const uint32_t* mbits, const int32_t* rowinfo, const int32_t* one2x, int32_t* work,
                   int32_t* glabel, int32_t* grp_n, int32_t* grp_one2x, int32_t* vidinfo,
                   int32_t* clusterinfo, const int32_t* gram, const int64_t* gram_off, void* stream);

/* Generic Hamming DBSCAN on one bit matrix (device), N rows of `stride` words, D columns
 * (padding bits must be zero). work: s2d_dbscan_work_ints(N, 1) int32, 8-byte aligned. */
int s2d_hamming_dbscan(const uint32_t* bits, int N, int stride, int D, double eps,
                       int min_samples, int32_t* work, int32_t* labels, void* stream);

/* K1. Dense mask-overlap contraction (cotracker_matching.py:653-657 for point-raster x mask;
 * model_training/mask2former_video/engine/train_loop.py:378-388 for mask x mask):
 *   I[a,b] = sum_px (A[a,px] != 0) * (B[b,px] != 0),  areaA[a], areaB[b]
 * _bits: operands bit-packed ([N][ceil(npix/32)] u32), AND + popc on CUDA cores.
 * _i8  : operands u8 0/1 ([N][npix]), tcgen05.mma kind::i8, int32 accumulators in TMEM. */
int s2d_pack_bits(const uint8_t* planes, int N, int64_t npix, uint32_t* bits, void* stream);
/* inverse: bit rows [N][stride_words] -> u8 0/1 planes [N][ncols] (ncols % 16 == 0; columns beyond the words are 0) */
int s2d_unpack_bits(const uint32_t* bits, int N, int stride_words, int64_t ncols, uint8_t* planes, void* stream);
int s2d_overlap_bits(const uint32_t* Abits, int Na, const uint32_t* Bbits, int Nb, int64_t nwords,
                     int32_t* I, int32_t* areaA, int32_t* areaB, void* stream);

/* Tensor-core variant: u8 planes (values 0/1) [N][npix], npix % 16 == 0, 16-byte aligned bases.
 * TMA (SWIZZLE_128B) -> 4-stage smem ring -> tcgen05.mma kind::i8 (M128 x N x K32, int32 in TMEM),
 * split-K over pixels with int32 atomics into I (cleared inside). */
int s2d_overlap_i8(const uint8_t* A, int Na, const uint8_t* B, int Nb, int64_t npix, int32_t* I,
                   void* stream);

/* One-hot Gram form straight from label maps: rows r = f * nlab + l for `nframes` frames and labels
 * 0..nlab-1 (nlab <= 254; tested down to 3 - with fewer labels per frame and many frames the label ring of
 * even the narrowest tiling does not fit in shared memory and the call returns an error);
 * G[r, r'] = |mask(f,l) AND mask(f',l')| (int32 [R][R]). `work`: int32 scratch
 * of s2d_overlap_gram_work_ints() elements (per-split partial tiles, summed by a second kernel). The u8 0/1
 * operand tiles are synthesised in shared memory from the 1 B/px label bytes, so HBM traffic is
 * nframes*npix bytes for 2*R^2*npix tensor-core ops (SURVEY.md section 8(d): the tensor-bound form). */
int s2d_overlap_gram_work_ints(int nframes, int nlab, int64_t npix, int64_t* out);
/* Which tiling s2d_overlap_gram_labels uses for this shape (host-only query): *out = 2: 256 x 256 blocks, two M128 x N256
 * MMA groups per k-block (gram_labels2_kernel); 1: 128 x 256 tiles; 0: 128 x 128 tiles (gram_labels_kernel). The wider
 * tilings need the label ring of 256 / nlab + 2 frames per operand to fit beside the operand stages. */
int s2d_overlap_gram_tiling(int nframes, int nlab, int* out);
/* Multiply-accumulate work the tensor cores actually EXECUTE for this shape (host-only query): 2 * M * N * K summed over the
 * launched tiles - only the tiles touching the upper triangle of the symmetric matrix run, and partial tiles run in full. The
 * algorithmic figure is 2 * R^2 * npix; tensor-pipe utilisation must be quoted from the executed figure. */
int s2d_overlap_gram_executed_ops(int nframes, int nlab, int64_t npix, double* out);
int s2d_overlap_gram_labels(const uint8_t* labels, int nframes, int nlab, int64_t npix, int32_t* work,
                            int32_t* G, void* stream);

/* Banded form of the Gram overlap ("all mask pairs within a frame window", BASELINE.json north_star kernel 1): only pairs
 * of rows whose frames are at most band_frames apart. Gband: int32 [R][(2 * band_frames + 1) * nlab],
 * Gband[f * nlab + l][(d + band_frames) * nlab + l2] = |mask(f, l) AND mask(f + d, l2)| for -band <= d <= band, 0 when frame
 * f + d does not exist. Only the 256 x 256 blocks of the symmetric matrix that touch the band are executed (long videos:
 * 300 frames x 30 labels, band 64 -> a third of the upper triangle), each block's pixel range split to fill whole waves.
 * Needs the 256 x 256 tiling (s2d_overlap_gram_tiling == 2). work: s2d_overlap_gram_band_work_ints() int32. */
int s2d_overlap_gram_band_work_ints(int nframes, int nlab, int64_t npix, int band_frames, int64_t* out);
int s2d_overlap_gram_labels_banded(const uint8_t* labels, int nframes, int nlab, int64_t npix, int band_frames,
                                   int32_t* work, int32_t* Gband, void* stream);

/* Rasterise tracks of one query into a u8 plane per frame (pred_tracks_to_binary_masks,
 * return_mask=False, cotracker_matching.py:453-503) - the dense A operand of K1. */
int s2d_rasterise_tracks(const float* tracks, int T, int P, int H, int W, uint8_t* planes,
                         void* stream);

/* f1 (first "next" row of the scope table). Colour-coded mask frames -> per-frame label ids:
 * label = 1 + rank of the pixel's (R,G,B) tuple among the frame's non-black colours in
 * lexicographic order, 0 for black. Replaces load_masks / convert_lblimg_to_maskid
 * (cotracker_occlusions.py:22-85, cotracker_matching.py:22-84, crw_utils.py:688-767).
 * rgb: u8 [F][npix][3] (R,G,B), labels: u8 [F][npix], ncolors: i32 [F] = number of non-black colours
 * (> 255: the frame does not fit u8 labels and its labels are undefined). work: u32 scratch of
 * s2d_color_to_labels_work_ints(F) elements. */
int s2d_color_to_labels_work_ints(int nframes, int64_t* out);
int s2d_color_to_labels(const uint8_t* rgb, int nframes, int64_t npix, uint32_t* work, uint8_t* labels,
                        int32_t* ncolors, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* S2D_B200_H */
