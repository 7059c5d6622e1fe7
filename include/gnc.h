/*
 * gnc.h - C ABI of libgnc.so, the B200 (sm_100a) implementation of the
 * GraphNet_Classifier hot path: image -> graph construction and the GraphNet
 * forward / backward operators.
 *
 * Conventions (every entry point):
 *   - extern "C", plain pointers and sizes, no framework types;
 *   - unless a parameter is documented as HOST, every pointer is a DEVICE pointer
 *     owned by the caller; nothing is allocated, freed or retained by the library;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *     all work is enqueued on it and the call returns without synchronising;
 *   - return value: GNC_OK (0) or a GNC_E* code; gnc_last_error() gives the text of
 *     the most recent failure on the calling thread;
 *   - fp32 data, row-major, leading dimensions (`ld*`) counted in elements;
 *     node / edge ids are int32 inside the library, int64 only at the
 *     edge_index boundary (the reference's torch.long tensors);
 *   - stateless and re-entrant (the launch counter below is the only global).
 *
 * The reference (alexisvannson/GraphNet_Classifier) is pure Python with no FFI of
 * its own; each entry point cites the reference lines whose work it replaces
 * (paths relative to the reference root).  INTEGRATION.md shows the ctypes
 * binding a maintainer of the reference would add.
 */
#ifndef GNC_H_
#define GNC_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GNC_OK 0
#define GNC_EINVAL 1   /* bad argument (shape, alignment, null pointer) */
#define GNC_ECUDA 2    /* a CUDA runtime call or kernel launch failed */
#define GNC_EWORKSPACE 3 /* caller-provided workspace too small */

typedef void* gnc_stream_t;

/* A gathered, column-concatenated matrix operand: logical row m is
 *   concat_s( base_s[(idx_s ? idx_s[m] : m) * ld_s + 0 .. width_s) ).
 * This is how cat([x[row], x[col], edge_attr]) (models/GNN.py:58-60, with the
 * gathers PyG's MetaLayer does at models/GNN.py:146/215) and cat([x, agg])
 * (models/GNN.py:100) are consumed without being materialised. */
typedef struct gnc_seg {
  const float* base;
  const int32_t* idx; /* NULL = identity */
  int64_t ld;
  int32_t width;
  int32_t _pad;
} gnc_seg_t;

/* ---- library state --------------------------------------------------------- */
int gnc_version(void);
const char* gnc_last_error(void);
/* number of kernels this library has launched since load / last reset */
uint64_t gnc_launch_count(void);
void gnc_reset_launch_count(void);

/* ---- graph construction ---------------------------------------------------- */

/* Edge count of the directed H x W grid (image_to_graph_optimized.py:22-37). */
int64_t gnc_grid_num_edges(int H, int W, int diagonals);

/* Batched pixel-graph builder: replaces image_to_graph_pixel_optimized lines
 * 71-87 + the casts at utils/dataloader.py:49-51 for B already-resized images.
 *   img        uint8  [B, H, W, 3]
 *   x          float  [B*H*W, 3]     pixel values 0..255 (un-normalised)
 *   pos        float  [B*H*W, 2]     (row, col); may be NULL (positions depend on the
 *                                    shape only, callers cache them)
 *   edge_index int64  [2, B*E]       contiguous rows (src; dst), graph b offset by
 *                                    b*H*W, edge order of create_grid_edges_optimized
 *                                    (image_to_graph_optimized.py:7-39); may be NULL
 * CSR outputs (all int32, any may be NULL as a group - pass all six or none):
 *   src32,dst32 [B*E]; dst_rowptr [B*N+1], dst_eid [B*E] (in-edges of each node,
 *   ascending edge id = the CPU summation order of models/GNN.py:99);
 *   src_rowptr, src_eid likewise for out-edges. */
int gnc_build_pixel_graph_u8(const uint8_t* img, int B, int H, int W, int diagonals,
                             float* x, float* pos, int64_t* edge_index,
                             int32_t* src32, int32_t* dst32,
                             int32_t* dst_rowptr, int32_t* dst_eid,
                             int32_t* src_rowptr, int32_t* src_eid,
                             gnc_stream_t stream);

/* Batched patch-graph builder (image_to_graph_patch.py:25-54): one node per
 * p x p tile, x = tile mean RGB (0..255), pos = tile centre, grid edges over the
 * (H/p) x (W/p) tiles.  Output shapes as above with N = (H/p)*(W/p). */
int gnc_build_patch_graph_u8(const uint8_t* img, int B, int H, int W, int patch,
                             float* x, float* pos, int64_t* edge_index,
                             int32_t* src32, int32_t* dst32,
                             int32_t* dst_rowptr, int32_t* dst_eid,
                             int32_t* src_rowptr, int32_t* src_eid,
                             gnc_stream_t stream);

/* Label map -> superpixel graph (image_to_graph_superpixel.py:34-71), one image
 * per call slot b; labels need not be contiguous, node id = rank among the
 * labels present.  `max_label` bounds label values (0 <= label <= max_label).
 *   img      uint8 [B, H, W, 3];  labels int32 [B, H, W]
 *   n_nodes  int32 [B]            S_b
 *   x        float [B, S_max, 3]  mean of img/255 per segment
 *   pos      float [B, S_max, 2]  centroid (row, col)
 *   adj      uint8 [B, S_max, S_max] 4-connected adjacency (symmetric, zero diag)
 *   n_edges  int32 [B]            2 * (#adjacent pairs)
 *   edges    int64 [B, 2, E_max]  (i,j),(j,i) for i<j lexicographic, local ids
 *   work     int32 [B * gnc_superpixel_workspace(S_max, max_label)] scratch
 * Entries beyond S_b / n_edges[b] are left zero. */
int64_t gnc_superpixel_workspace(int S_max, int max_label);
int gnc_build_superpixel_graph(const uint8_t* img, const int32_t* labels, int B, int H, int W,
                               int max_label, int S_max, int64_t E_max,
                               int32_t* n_nodes, float* x, float* pos, uint8_t* adj,
                               int32_t* n_edges, int64_t* edges, int32_t* work,
                               gnc_stream_t stream);
/* Block-diagonal batch of the per-image graphs above (graphs of DIFFERENT sizes, as superpixel graphs are):
 * offsets:  node_ptr int32 [B + 1], edge_ptr int64 [B + 1] = running sums of min(n_nodes, S_max) / min(n_edges, E_max);
 * compact:  xb float [node_ptr[B], 3], pb float [node_ptr[B], 2], eb int64 [2, e_total] (e_total = edge_ptr[B]) with
 *           the endpoints shifted by the image's node offset; graph b owns nodes node_ptr[b] .. node_ptr[b + 1]. */
int gnc_superpixel_batch_offsets(const int32_t* n_nodes, const int32_t* n_edges, int B, int S_max, int64_t E_max,
                                 int32_t* node_ptr, int64_t* edge_ptr, gnc_stream_t stream);
int gnc_superpixel_batch_compact(const float* x, const float* pos, const int64_t* edges, int B, int S_max, int64_t E_max,
                                 const int32_t* node_ptr, const int64_t* edge_ptr, float* xb, float* pb, int64_t* eb,
                                 int64_t e_total, gnc_stream_t stream);
/* The same batch at host-known sizes, for a build that reads nothing back (CUDA-graph capture).  x / pos / edges /
 * n_nodes / n_edges come from gnc_build_superpixel_graph called with S_max = S_cap and E_max = E_cap; node_ptr /
 * edge_ptr from gnc_superpixel_batch_offsets with the same capacities.
 *   xb float [B * S_cap + 1, 3], pb float [B * S_cap + 1, 2], eb int64 [2, B * E_cap]
 * Rows [0, node_ptr[B]) and edges [0, edge_ptr[B]) equal gnc_superpixel_batch_compact's output.  The other rows are
 * zero; the other edges are self-loops of those rows (edge edge_ptr[B] + k loops on row node_ptr[B] + k mod
 * (B * S_cap + 1 - node_ptr[B])), so no real node receives a padding edge.  `labels` (int32 [B, H, W], may be NULL) is
 * checked against [0, max_label].  *overflow (int32) is overwritten: 0 when everything fit, else bit 0 = a label out of
 * range, bit 1 = an image with more than S_cap nodes, bit 2 = more than E_cap edges.  Never writes outside the buffers. */
int gnc_superpixel_batch_padded(const float* x, const float* pos, const int64_t* edges, const int32_t* n_nodes,
                                const int32_t* n_edges, const int32_t* labels, int B, int H, int W, int max_label,
                                int S_cap, int64_t E_cap, const int32_t* node_ptr, const int64_t* edge_ptr, float* xb,
                                float* pb, int64_t* eb, int32_t* overflow, gnc_stream_t stream);

/* SLIC superpixel labels for B images (the stage the reference delegates to scikit-image,
 * image_to_graph_superpixel.py:31; parity unpinned - see csrc/slic.cu): RGB -> Lab, regular-grid
 * centres, `iters` assignment/update iterations, deterministic.
 *   img uint8 [B, H, W, 3]; labels int32 [B, H, W] in [0, gnc_slic_num_centers(H, W, n_segments));
 *   work: gnc_slic_workspace_bytes(...) bytes of scratch. */
int gnc_slic_num_centers(int H, int W, int n_segments);
int64_t gnc_slic_workspace_bytes(int B, int H, int W, int n_segments);
int gnc_slic_labels_u8(const uint8_t* img, int B, int H, int W, int n_segments, float compactness, int iters,
                       int32_t* labels, void* work, gnc_stream_t stream);
/* Debug aid: 1 = streaming form (one launch per iteration) with one set of centre atomics per pixel, -8 = streaming form
 * with one set per 8-pixel label run, anything else = default (one CTA per image runs the whole loop in one launch
 * when W % 8 == 0 and there are at most 1024 centres; the streaming form otherwise).  Same labels in every form. */
int gnc_debug_slic_run_length(int run);
/* Debug aid: 1 = gnc_slic_enforce_connectivity always uses the streaming (global-memory union-find) form, 0 = default
 * (one CTA per image with the forest in shared memory when H * W <= 65536).  Same result. */
int gnc_debug_slic_connect_streaming(int on);

/* Input staging, first half: the file decode behind  Image.open(path).convert('RGB')  (utils/dataloader.py:34 through
 * ImageFolder's loader, utils/image_to_graph/image_to_graph_optimized.py:65-68, utils/inference.py:47) for baseline
 * JPEG files, bit for bit what Pillow's libjpeg produces with its defaults (csrc/jpeg.cu).
 * gnc_jpeg_parse (HOST): markers of one file -> geometry, dequantisation and Huffman decode tables, position of the
 *   entropy-coded scan (relative to `data`; add the file's offset in the batch buffer before the device call).
 *   Returns GNC_OK, or GNC_JPEG_UNSUPPORTED for anything outside baseline / extended-sequential Huffman, 8 bit, one
 *   interleaved scan, greyscale or YCbCr 4:4:4 / 4:2:2 / 4:2:0 - decode those with Pillow on the host.
 * gnc_jpeg_decode_rgb_u8 (DEVICE): `stream` = the files' bytes back to back, `infos` = B parsed descriptors with
 *   scan_offset (into stream), block_offset (running sum of n_blocks), coef_offset (= 64 * block_offset), plane_offset
 *   (running sum of plane_bytes) and pixel_offset (running sum of width * height) filled in by the caller;
 *   coef: int16 [64 * total_blocks], planes: uint8 [sum plane_bytes], out: uint8 [3 * total_pixels] - image i's RGB
 *   pixels, row-major, at 3 * pixel_offset; `stream` itself must be 4-byte aligned.  Entropy decode: the 32 lanes of a
 *   warp decode 32 segments of an image's scan from guessed states and iterate until every segment starts where its
 *   predecessor stopped (Huffman streams are self-synchronising); scans with restart intervals or shorter than 4 KB,
 *   and all scans when `scratch` is NULL, are decoded by one thread. */
#define GNC_JPEG_UNSUPPORTED 4
typedef struct gnc_jpeg_huff {
  uint16_t look[512];     /* 9-bit lookahead: (code length << 8) | symbol, 0 = longer code */
  int32_t maxcode[18];    /* largest code of each length (-1: none), [17] = sentinel */
  int32_t valoff[17];     /* index of a length's first symbol minus its first code */
  uint8_t vals[256];
} gnc_jpeg_huff_t;
typedef struct gnc_jpeg_image {
  int32_t width, height, ncomp;
  int32_t hsamp[3], vsamp[3], qtab[3], dc_tab[3], ac_tab[3];
  int32_t restart_interval, mcu_x, mcu_y, _pad;
  int64_t scan_offset, scan_bytes, n_blocks, plane_bytes;
  int64_t block_offset, coef_offset, plane_offset, pixel_offset;
  uint16_t quant[4][64];  /* natural (row-major) order */
  gnc_jpeg_huff_t huff[8];/* [0..3] DC tables, [4..7] AC tables */
} gnc_jpeg_image_t;
int gnc_jpeg_parse(const uint8_t* data, int64_t size, gnc_jpeg_image_t* out);
/* HOST: a whole batch in one call - parses every file (on `threads` host threads), leaves out the unsupported ones
 * (index_out[j] = index of the j-th file that is in), copies the bytes of the others back to back into stream_out
 * (pinned memory, capacity >= sum of sizes) and fills infos_out[0 .. totals[0]) with all offsets set.
 * totals[5] = { files in, stream bytes, total blocks, plane bytes, pixels }. */
int gnc_jpeg_pack(const uint8_t* const* datas, const int64_t* sizes, int n, int threads, uint8_t* stream_out,
                  int64_t stream_capacity, gnc_jpeg_image_t* infos_out, int32_t* index_out, int64_t* totals);
int64_t gnc_jpeg_scratch_bytes(int64_t stream_bytes, int B);
int gnc_jpeg_decode_rgb_u8(const uint8_t* stream, const gnc_jpeg_image_t* infos, int B, int64_t total_blocks,
                           int64_t total_pixels, int16_t* coef, uint8_t* planes, uint8_t* out,
                           uint8_t* scratch /* gnc_jpeg_scratch_bytes(stream bytes, B), 4-byte aligned; NULL: sequential entropy decode */,
                           gnc_stream_t stream_);
/* Debug aid: 1 = the entropy stage always runs its sequential form (one thread per image); same coefficients. */
int gnc_debug_jpeg_sequential(int on);

/* Progressive JPEG files (SOF2, 8-bit Huffman, greyscale or YCbCr 4:4:4 / 4:2:2 / 4:2:0), bit for bit what Pillow's
 * libjpeg produces (csrc/jpeg.cu).  A progressive file codes its coefficients in several scans; every scan writes one
 * band Ss..Se of one component (AC) or coefficient 0 of one or more components (DC), at bit position Al, refining
 * (Ah != 0) or first (Ah == 0).  Two scans are linked when they write a common coefficient of a common component; a
 * CHAIN is a connected group of linked scans in file order.  Chains write disjoint coefficients and decode concurrently.
 * gnc_jpeg_pack_progressive (HOST): the batch form of gnc_jpeg_pack for progressive files.  Per file that is in:
 *   frames_out[j]  geometry, MCU counts, n_blocks, plane_bytes, block / coef / plane / pixel offsets and the
 *                  quantisation tables latched at each component's first scan (qtab[c] = c) - what jpeg_idct_kernel and
 *                  jpeg_color_kernel read; its huff[] and scan fields are unused;
 *   its scans      gnc_jpeg_scan_t, entropy segments as offsets into stream_out, tables as indices into tables_out;
 *   its chains     gnc_jpeg_chain_t, ordered longest first (entropy bytes) across the batch, each chain's scans
 *                  contiguous in scans_out in file order.
 *   Left out (index_out lists the files that are in): every file libjpeg would not decode by the plain path - other
 *   frame types and layouts, progressions jdphuff.c rejects or warns about, and files that end with a DC never coded or
 *   an AC coefficient 1..9 of some component not fully refined (libjpeg then smooths across blocks) - and files with a
 *   scan running past the file, no EOI, a DNL, or more than GNC_JPEG_MAX_SCANS scans / GNC_JPEG_MAX_TABLES tables.
 *   Capacities: scans n * GNC_JPEG_MAX_SCANS, chains the same, tables n * GNC_JPEG_MAX_TABLES always suffice.
 *   totals[8] = { files in, stream bytes, total blocks, plane bytes, pixels, scans, chains, tables }.
 * gnc_jpeg_decode_progressive_rgb_u8 (DEVICE): zeroes coef, decodes every chain (one lane per chain, one chain per warp
 *   by default; scans in file order, jdphuff.c's DC / AC first / refine procedures), then runs the
 *   baseline IDCT and colour stages on `frames`.  Sizes and buffers as gnc_jpeg_decode_rgb_u8. */
#define GNC_JPEG_MAX_SCANS 64
#define GNC_JPEG_MAX_TABLES 32
typedef struct gnc_jpeg_scan {
  int32_t image;          /* index into frames */
  int32_t ncomp;          /* components in the scan; > 1 only for DC scans, which are then interleaved */
  int32_t comp[3];        /* frame component indices, in frame order */
  int32_t dc_tab[3];      /* DC first scans: index into tables, per scan component */
  int32_t ac_tab;         /* AC scans: index into tables */
  int32_t Ss, Se, Ah, Al;
  int32_t restart_interval;
  int64_t offset, bytes;  /* entropy-coded segment in the stream */
} gnc_jpeg_scan_t;
typedef struct gnc_jpeg_chain {
  int32_t first_scan, n_scans;
  int64_t bytes;          /* entropy bytes of its scans */
} gnc_jpeg_chain_t;
int gnc_jpeg_pack_progressive(const uint8_t* const* datas, const int64_t* sizes, int n, int threads, uint8_t* stream_out,
                              int64_t stream_capacity, gnc_jpeg_image_t* frames_out, int32_t* index_out,
                              gnc_jpeg_scan_t* scans_out, int64_t scan_capacity, gnc_jpeg_chain_t* chains_out,
                              int64_t chain_capacity, gnc_jpeg_huff_t* tables_out, int64_t table_capacity, int64_t* totals);
int gnc_jpeg_decode_progressive_rgb_u8(const uint8_t* stream, const gnc_jpeg_image_t* frames, int B,
                                       const gnc_jpeg_scan_t* scans, const gnc_jpeg_chain_t* chains, int n_chains,
                                       const gnc_jpeg_huff_t* tables, int64_t total_blocks, int64_t total_pixels,
                                       int16_t* coef, uint8_t* planes, uint8_t* out, gnc_stream_t stream_);
/* Debug aid: chains per warp of the progressive entropy kernel (1..32; anything else = the default, 1).  Same result. */
int gnc_debug_jpeg_chains_per_warp(int n);

/* Input staging: the resize the reference applies to every image before building its graph,
 *   Image.open(path).convert('RGB').resize((r, r))     utils/image_to_graph/image_to_graph_optimized.py:65-70,
 *                                                      image_to_graph_patch.py / _superpixel.py likewise
 * = Pillow's two-pass BICUBIC ImagingResample (horizontal pass first, 8-bit intermediate, 22-bit fixed-point
 * coefficients).  Bit-identical to Pillow (csrc/resize.cu, oracle/resize.py).
 *   gnc_resize_bicubic_ksize   taps per output pixel along an axis resized in_size -> out_size (0 on bad sizes);
 *   gnc_resize_bicubic_coeffs  HOST: fills bounds int32 [out_size, 2] (first tap, tap count) and
 *                              kk int32 [out_size, ksize] with Pillow's tables for that axis;
 *   gnc_resize_bicubic_u8      src uint8 [B, H, W, 3] (src_pitch bytes between rows, src_image_stride bytes between
 *                              images) -> dst uint8 [B, OH, OW, 3] contiguous.  bounds_* / kk_* are DEVICE copies of
 *                              the tables of the x (W -> OW) and y (H -> OH) axes; an axis whose size does not change
 *                              is not filtered and takes NULL tables (Pillow does the same).  tmp: uint8
 *                              [B, H, OW, 3] scratch, needed only when both axes change. */
int gnc_resize_bicubic_ksize(int in_size, int out_size);
int gnc_resize_bicubic_coeffs(int in_size, int out_size, int32_t* bounds /*HOST*/, int32_t* kk /*HOST*/);
int gnc_resize_bicubic_u8(const uint8_t* src, int64_t B, int H, int W, int64_t src_pitch, int64_t src_image_stride,
                          int OH, int OW, const int32_t* bounds_x, const int32_t* kk_x, int ksize_x,
                          const int32_t* bounds_y, const int32_t* kk_y, int ksize_y, uint8_t* tmp, uint8_t* dst,
                          gnc_stream_t stream);
/* Ragged batches: n images, each of its own H x W, -> dst uint8 [n, OH, OW, 3] contiguous, in three launches whatever
 * the number of shapes; bit-identical to resizing each image on its own.
 *   images   DEVICE array of n descriptors.  The caller fills, from the shapes alone:
 *              ksize_x / ksize_y  gnc_resize_bicubic_ksize of the axis, 0 when its size already is OW / OH;
 *              tab_x / tab_y      int32 offsets into `tables` of the axis's bounds [out, 2] followed by its kk
 *                                 [out, ksize]; non-overlapping (out * (2 + ksize) int32 each, none for ksize 0);
 *              tmp_row            rows of tmp [h_rows, OW, 3] before this image: the running sum of height over the
 *                                 images before it whose width changes.
 *   h_rows   rows of tmp = the sum of height over the images whose width changes; max_w = their largest width.
 *   tables   int32 workspace, written here (gnc_resize_bicubic_coeffs's tables, computed on the device).
 * Sources may have any alignment and row pitch (pixels 3 bytes apart). */
typedef struct gnc_resize_image {
  const uint8_t* src;     /* [height, width, 3], rows `pitch` bytes apart */
  int64_t pitch;
  int64_t tmp_row;
  int64_t tab_x, tab_y;
  int32_t height, width;
  int32_t ksize_x, ksize_y;
} gnc_resize_image_t;
int gnc_resize_bicubic_ragged_u8(const gnc_resize_image_t* images, int64_t n, int OH, int OW, int64_t h_rows, int max_w,
                                 int32_t* tables, uint8_t* tmp, uint8_t* dst, gnc_stream_t stream);

/* Stable CSR of edge ids grouped by key (= edge_index row 0 or row 1): the order
 * index_add_ visits edges in (models/GNN.py:20).  key is read with an element
 * stride so that non-contiguous edge_index (SURVEY.md 8a row a1) is accepted.
 *   key int64 [E] (strided); rowptr int32 [N+1]; eid int32 [E];
 *   key32 int32 [E] or NULL (narrowed copy of key);
 *   work  int32 [gnc_csr_workspace(N)] scratch.
 * Returns GNC_EINVAL via the device flag if a key is outside [0, N) - checked
 * lazily: `bad` (int32 [1], device, may be NULL) is set non-zero. */
int64_t gnc_csr_workspace(int64_t N);
int gnc_csr_build(const int64_t* key, int64_t key_stride, int64_t E, int64_t N,
                  int32_t* rowptr, int32_t* eid, int32_t* key32, int32_t* work, int32_t* bad,
                  gnc_stream_t stream);

/* ---- aggregation / gathers -------------------------------------------------- */

/* out[v, :] (+)= sum over k in [rowptr[v], rowptr[v+1]) of src[eid[k], :], summed
 * sequentially in ascending k.  Replaces scatter_sum(edge_attr, col, dim=0)
 * (models/GNN.py:3-21, call site :99) and, with the source-side CSR, the
 * index_put_(accumulate) backward of the x[row] / x[col] gathers. */
int gnc_agg_csr_sum_f32(const int32_t* rowptr, const int32_t* eid,
                        const float* src, int64_t ld_src, int64_t N, int D,
                        float* out, int64_t ld_out, int accumulate, gnc_stream_t stream);

/* Two such sums over the same [E, D] tensor in ONE launch: out_a by CSR a, out_b by CSR b (N rows each, row pitch ld_out) -
 * the backward of the x[row] and x[col] gathers of EdgeProcessor.forward (models/GNN.py:57-58), i.e. the edge gradient
 * summed by source and by destination.  The two sums walk the node rows in step, so a row of `src` fetched for one is
 * still in L2 for the other on locality-preserving topologies.  Same bits as two gnc_agg_csr_sum_f32 calls. */
int gnc_agg_csr_sum_pair_f32(const int32_t* rowptr_a, const int32_t* eid_a, float* out_a,
                             const int32_t* rowptr_b, const int32_t* eid_b, float* out_b,
                             const float* src, int64_t ld_src, int64_t N, int D, int64_t ld_out, gnc_stream_t stream);

/* out[m, :] (+)= src[idx[m], :]   (x[row], x[col]; backward of the aggregation) */
int gnc_gather_rows_f32(const float* src, int64_t ld_src, const int32_t* idx, int64_t M, int D,
                        float* out, int64_t ld_out, int accumulate, gnc_stream_t stream);

/* out[m, :] = act( sum_s tables[s][idx[s][m], :] + bias ), 1 <= nsrc <= 4 (idx[s] NULL = identity).
 * tables / idx / ld are HOST arrays of device pointers / strides.  D % 4 == 0. */
int gnc_gather_add_rows_f32(const float* const* tables /*HOST*/, const int32_t* const* idx /*HOST*/,
                            const int64_t* ld /*HOST*/, int nsrc, const float* bias, int relu,
                            int64_t M, int D, float* out, int64_t ld_out, gnc_stream_t stream);

/* Edge family of a batched H x W grid graph (0 horizontal, 1 vertical, 2/3 diagonals): all edges of
 * a family share one geometry row (models/GNN.py:299-302 applied to grid positions).  cls int32 [B*E]. */
int gnc_grid_edge_class(int B, int H, int W, int diagonals, int32_t* cls, gnc_stream_t stream);
/* Paired destination slots of a batch of B grids H x W without diagonals (csrc/grid_topology.h): 2 B H W slots, slot 2v
 * for the horizontal in-edge of node v, 2v + 1 for the vertical one.  Writes each slot's source node (-1: no such edge,
 * a padding slot), destination node (s >> 1) and edge class (0 / 1), int32 [2 B H W] each. */
int gnc_grid_pair_slots(int B, int H, int W, int32_t* slot_src, int32_t* slot_dst, int32_t* slot_class, gnc_stream_t stream);

/* edge_attr[e] = [pos[dst[e]] - pos[src[e]], sum |.|]  (models/GNN.py:299-302).
 * pos float [N, P]; out float [E, P+1]; 1 <= P <= 8. */
int gnc_edge_geometry_f32(const float* pos, int P, const int32_t* src, const int32_t* dst, int64_t E,
                          float* out, gnc_stream_t stream);

/* ---- dense operators (nn.Linear / ReLU / LayerNorm of models/MLP.py:24-37) -- */

/* Y[M, N] = act( concat(segs)[M, K] * W[N, K]^T + bias ),  K = sum of widths.
 * relu != 0 applies max(.,0).  bias may be NULL. */
int gnc_linear_fwd_f32(const gnc_seg_t* segs /*HOST*/, int nseg, int64_t M,
                       const float* W, int64_t ldw, const float* bias, int N, int relu,
                       float* Y, int64_t ldy, gnc_stream_t stream);

/* The same with the reduction split over CTAs (few output tiles, long K: the classifier head's first layer,
 * models/GNN.py:315, K = number of nodes) and a deterministic slice-order reduction.
 * work: float [gnc_linear_fwd_splitk_workspace(M, N, K)] (0 = no split: work may be NULL). */
int64_t gnc_linear_fwd_splitk_workspace(int64_t M, int N, int64_t K);
int gnc_linear_fwd_splitk_f32(const gnc_seg_t* segs /*HOST*/, int nseg, int64_t M,
                              const float* W, int64_t ldw, const float* bias, int N, int relu,
                              float* Y, int64_t ldy, float* work, int64_t work_elems, gnc_stream_t stream);

/* Thin first layers (1 <= K <= 8 inputs: pixel channels / edge geometry, models/GNN.py:233-234):
 * Y[M, N] = act(X[M, K] * W[N, K]^T + bias), one streaming pass.  N % 4 == 0. */
int gnc_linear_narrowk_fwd_f32(const float* X, int64_t ldx, int64_t M, int K, const float* W, int64_t ldw,
                               const float* bias, int N, int relu, float* Y, int64_t ldy, gnc_stream_t stream);
/* Backward of the thin layer in one pass over (dY, Y, X): dZ = dY * (Y > 0) if Y != NULL,
 * dW[N, K] (+)= dZ^T X, db[N] (+)= column sums of dZ (dW / db may be NULL).  N <= 128.
 * work: float [gnc_linear_narrowk_wgrad_workspace(M, N, K)]. */
int64_t gnc_linear_narrowk_wgrad_workspace(int64_t M, int N, int K);
int gnc_linear_narrowk_wgrad_f32(const float* dY, int64_t lddy, const float* Y, int64_t ldy,
                                 const float* X, int64_t ldx, int64_t M, int N, int K,
                                 float* dW, int64_t lddw, float* db, int accumulate,
                                 float* work, int64_t work_elems, gnc_stream_t stream);

/* dX[M, K] (+)= dZ[M, N] * W[N, K]   (W may point at a column slice, ldw = full K) */
int gnc_linear_dgrad_f32(const float* dZ, int64_t lddz, int64_t M, int N,
                         const float* W, int64_t ldw, int K,
                         float* dX, int64_t lddx, int accumulate, gnc_stream_t stream);

/* dW[N, K] (+)= dZ[M, N]^T * concat(segs)[M, K]; deterministic split reduction.
 * work: float [gnc_linear_wgrad_workspace(M, N, K)]. */
int64_t gnc_linear_wgrad_workspace(int64_t M, int N, int K);
int gnc_linear_wgrad_f32(const float* dZ, int64_t lddz, int64_t M, int N,
                         const gnc_seg_t* segs /*HOST*/, int nseg,
                         float* dW, int64_t lddw, int accumulate,
                         float* work, int64_t work_elems, gnc_stream_t stream);

/* dZ = dY * (Y > 0) (if Y != NULL, else dZ = dY; dZ may be NULL to skip the
 * store), db[N] (+)= column sums of dZ.  Backward of bias + ReLU.
 * work: float [gnc_colsum_workspace(M, N)]. */
int64_t gnc_colsum_workspace(int64_t M, int N);
int gnc_relu_bwd_colsum_f32(const float* dY, int64_t lddy, const float* Y, int64_t ldy,
                            int64_t M, int N, float* dZ, int64_t lddz,
                            float* db, int accumulate, float* work, int64_t work_elems,
                            gnc_stream_t stream);

/* y = LayerNorm(z; gamma, beta, eps) (+ res).  mean / rstd float [M] are saved
 * for the backward (may be NULL).  models/MLP.py:34-35, residuals
 * models/GNN.py:62, 102. */
int gnc_layernorm_fwd_f32(const float* z, int64_t ldz, int64_t M, int D,
                          const float* gamma, const float* beta, float eps,
                          const float* res, int64_t ldres,
                          float* y, int64_t ldy, float* mean, float* rstd, gnc_stream_t stream);

/* dz = LN backward; dgamma/dbeta (+)= column reductions.
 * work: float [gnc_layernorm_bwd_workspace(M, D)]. */
int64_t gnc_layernorm_bwd_workspace(int64_t M, int D);
int gnc_layernorm_bwd_f32(const float* dy, int64_t lddy, const float* z, int64_t ldz,
                          const float* mean, const float* rstd, const float* gamma,
                          int64_t M, int D, float* dz, int64_t lddz,
                          float* dgamma, float* dbeta, int accumulate,
                          float* work, int64_t work_elems, gnc_stream_t stream);

/* ---- tensor-core engine (tcgen05, 3xTF32) for width-128 layers ----------------- */

/* Epilogue of gnc_tc_linear_f32.  With acc = A * B^T (fp32-accurate, see csrc/tc_linear.cu):
 *   dot_w != NULL : Y[m, 0] = relu(acc + bias) . dot_w + *dot_b         (decoder tail, models/GNN.py:289-295)
 *   gamma != NULL : Y = LayerNorm(acc + bias; gamma, beta, eps) + residual[m]   (models/MLP.py:34-35, GNN.py:62,102)
 *   otherwise     : Y = act(acc + bias + addend[m] + gather0[gather0_idx[m]] + gather1[gather1_idx[m]])
 *                       + residual[m],  act = relu if relu != 0
 * Every pointer may be NULL (term absent).  Rows of addend / gather / residual are 128 wide. */
typedef struct gnc_tc_epilogue {
  const float* bias;
  const float* addend;  int64_t ld_addend;
  const float* gather0; const int32_t* gather0_idx; int64_t ld_gather0;
  const float* gather1; const int32_t* gather1_idx; int64_t ld_gather1;
  int32_t relu; int32_t _pad0;
  const float* gamma; const float* beta; float eps; int32_t _pad1;
  const float* residual; int64_t ld_residual;
  const float* dot_w; const float* dot_b;
  const float* mask; int64_t ld_mask;   /* elementwise only: Y *= (mask[m] > 0) - ReLU backward fused into the data gradient */
  const int32_t* residual_idx;          /* LayerNorm epilogue only: residual row = residual[residual_idx[m]] (table lookup) */
  /* LayerNorm epilogue only, all optional (training): ln_z [M, 128] receives acc + bias (the LayerNorm input), ln_mean /
   * ln_rstd [M] the row statistics - what gnc_layernorm_bwd_f32 consumes, without a separate forward pass over z */
  float* ln_z; int64_t ld_ln_z; float* ln_mean; float* ln_rstd;
} gnc_tc_epilogue_t;

/* Y[M, N] = epilogue( A[M, K] * B^T ), B = W[N, K] (transpose_w = 0) or B = W^T with W[K, N]
 * (transpose_w = 1: the data gradient dX = dZ * W).  K = N = 128 only (GNC_EINVAL otherwise:
 * callers fall back to gnc_linear_*_f32).  epi is a HOST pointer. */
int gnc_tc_linear_f32(const float* A, int64_t lda, int64_t M, int K,
                      const float* W, int64_t ldw, int N, int transpose_w,
                      const gnc_tc_epilogue_t* epi /*HOST*/, float* Y, int64_t ldy, gnc_stream_t stream);

/* Y_s[M, 128] = A[M, 128] * W_s[128, 128]^T for nsets = 2 or 3 weight sets in one launch (A is read
 * from HBM once; the other sets hit L2).  W / ldw / Y are HOST arrays.  No epilogue terms. */
int gnc_tc_linear_multi_f32(const float* A, int64_t lda, int64_t M, int nsets,
                            const float* const* W /*HOST*/, const int64_t* ldw /*HOST*/,
                            float* const* Y /*HOST*/, int64_t ldy, gnc_stream_t stream);

/* Chained MLP on the tensor-core engine (csrc/tc_chain.cu): nlayers = 2 or 3 Linear(128,128) layers,
 * ReLU after every layer but the last, hidden activations never written to memory:
 *   z0 = W[0] a + bias[0] + gather0[gather0_idx[m]] + gather1[gather1_idx[m]]      (idx NULL: row m itself)
 *   z_l = W[l] relu(z_{l-1}) + bias[l]
 *   dot_w != NULL : Y[m, 0] = relu(z_last) . dot_w + *dot_b                        (decoder, models/GNN.py:289-295)
 *   otherwise     : Y = LayerNorm(z_last; gamma, beta, eps) (gamma NULL: identity) + residual[residual_idx[m]]
 * i.e. one EdgeProcessor / NodeProcessor MLP of models/GNN.py:57-64, 95-104 per launch.  Operands are
 * split into two fp16 pieces after an exact power-of-two scaling (three MMAs per product): 4.7e-7 rel-L2
 * per product, tighter than gnc_tc_linear_f32's 3xTF32.  DOMAIN: |A|, |hidden activations| < 4094 and
 * |W| < 255 (fp16 range after the scaling); outside it the outputs are inf / NaN, never silently wrong.
 * Models outside the domain use the per-layer engines (gnc_tc_linear_f32, gnc_linear_fwd_f32). */
typedef struct gnc_tc_chain {
  int32_t nlayers; int32_t _pad0;
  const float* W[3]; int64_t ldw[3]; const float* bias[3];
  const float* gather0; const int32_t* gather0_idx; int64_t ld_gather0;
  const float* gather1; const int32_t* gather1_idx; int64_t ld_gather1;
  const float* gamma; const float* beta; float eps; int32_t _pad1;
  const float* residual; const int32_t* residual_idx; int64_t ld_residual;
  const float* dot_w; const float* dot_b;
  /* pre-stage form (A == NULL, nlayers = 2): the first operand is
   *   relu(gather2[gather2_idx[m]] + gather0[gather0_idx[m]] + gather1[gather1_idx[m]] + pre_bias)
   * and W[0], W[1] are the two layers after it - the block-0 edge processor when the encoded edge latents
   * are a small table indexed by edge class. */
  const float* gather2; const int32_t* gather2_idx; int64_t ld_gather2; const float* pre_bias;
  /* two-operand first layer: z0 += operand2[m] W_operand2^T (3 layers, LayerNorm, residual by row, no gathers) -
   * cat([x, agg]) @ V0^T of NodeProcessor.forward (models/GNN.py:100) with V0 = [W_operand2 | W[0]]. */
  const float* operand2; int64_t ld_operand2; const float* W_operand2; int64_t ldw_operand2;
  /* narrow first layer folded into the launch (encoders, models/GNN.py:259-287: Linear(3, 128) on pixel channels /
   * edge geometry): A has narrow_k <= 8 columns and the chain's first operand is relu(A narrow_W^T + narrow_b),
   * followed by nlayers = 2 layers and LayerNorm.  narrow_W is [128, narrow_k] with row stride ld_narrow_W. */
  const float* narrow_W; int64_t ld_narrow_W; const float* narrow_b; int32_t narrow_k; int32_t _pad2;
  /* training forward (stash_a1 != NULL; 3 layers, gather0 [+ gather1], LayerNorm, residual by row - the edge / node
   * processor of a block, models/GNN.py:57-64, 95-104): the same launch also writes what the backward pass of the MLP
   * reads - the two hidden ReLU outputs a1, a2 and the LayerNorm input z (each [M, 128], row pitch ld_stash) and the
   * row statistics mean[M], rstd[M] = 1 / sqrt(var + eps) - instead of three per-layer launches that write and
   * re-read them. */
  float* stash_a1; float* stash_a2; float* stash_z; int64_t ld_stash; float* stash_mean; float* stash_rstd;
  /* aggregated first operand (agg_rowptr != NULL; the two-operand form above): A is the [E, 128] EDGE table and row m of the
   * first operand is sum_{k in [agg_rowptr[m], agg_rowptr[m + 1])} A[agg_eid[k]] in ascending k - scatter_sum(edge_attr, col)
   * of NodeProcessor.forward (models/GNN.py:99) formed by the kernel's loader instead of a launch of its own.  M is the number
   * of NODE rows; agg_rowptr is int32 [M + 1]; every row must have AT MOST TWO entries (the caller checks the topology once:
   * grid graphs without diagonals) - with those the sum is the reference's bit for bit. */
  const int32_t* agg_rowptr; const int32_t* agg_eid;
  /* paired destination slots (gnc_grid_pair_slots; grids without diagonals, at most two in-edges per node).
   * edge_slots = 1 (the three-layer edge form with two indexed gathers, or the pre-stage form): the M rows are slots, and a
   *   NEGATIVE gather0_idx marks a padding slot - its gathers read row 0 and its output row is exactly +0.0.
   * edge_slots = 2: as 1, and Y gets M / 2 node rows (M even) Y[v] = (0 + y[2v]) + y[2v + 1] instead of the M slot rows y -
   *   scatter_sum(edge_attr, col) of the next node processor, in the reference's order, with no [M, 128] edge output.
   * paired_operand = 1 (the two-operand node form, without agg_rowptr): A is the [2M, 128] slot table and row m of the
   *   first operand is (0 + A[2m]) + A[2m + 1]. */
  int32_t edge_slots; int32_t paired_operand;
} gnc_tc_chain_t;

int gnc_tc_mlp_chain_f32(const float* A, int64_t lda, int64_t M, const gnc_tc_chain_t* chain /*HOST*/,
                         float* Y, int64_t ldy, gnc_stream_t stream);

/* Y_l[M, 128] = A[M, 128] * W_l[128, 128]^T (+ bias_l, bias may be NULL) for nsets = 2 or 3 weight sets in one
 * launch of the chained kernel: A is read once and stays in tensor memory for all products (the P / Q / T
 * products of a GraphNet block).  W / ldw / bias / Y are HOST arrays. */
int gnc_tc_multi_chain_f32(const float* A, int64_t lda, int64_t M, int nsets,
                           const float* const* W /*HOST*/, const int64_t* ldw /*HOST*/,
                           const float* const* bias /*HOST, may be NULL*/, float* const* Y /*HOST*/,
                           int64_t ldy, gnc_stream_t stream);

/* Debug aid: timeline (clock64 << 8 | tag) of CTA 0's roles in later gnc_tc_mlp_chain_f32 launches,
 * buf = device uint64 [4 * cap] zeroed by the caller; NULL switches it off (scripts/chain_trace.py). */
int gnc_debug_chain_trace(unsigned long long* buf, int cap);

/* dW[N, K] (+)= dZ[M, N]^T * X[M, K] on the tensor-core engine (N = K = 128 only); both operands
 * stream once, partial products are flushed from TMEM into fp32 registers every 128 rows and the
 * per-CTA results are reduced deterministically.  db (may be NULL): db[N] (+)= column sums of dZ
 * (the bias gradient), computed on the same pass.  work: float [gnc_tc_wgrad_workspace(M)]. */
int64_t gnc_tc_wgrad_workspace(int64_t M);
int gnc_tc_wgrad_f32(const float* dZ, int64_t lddz, const float* X, int64_t ldx, int64_t M, int N, int K,
                     float* dW, int64_t lddw, int accumulate, float* db,
                     float* work, int64_t work_elems, gnc_stream_t stream);

/* Fused backward of one width-128 Linear layer (models/MLP.py:24-27 under autograd), both gradients from ONE read
 * of dZ and X:  dX[M,128] = dZ * W  (* (X > 0) when mask_by_x: ReLU backward of the layer that produced X;
 * + addend, e.g. the gradient arriving through a residual; addend may be NULL),  dW[128,128] (+)= dZ^T * X,
 * db[128] (+)= column sums of dZ (dW / db may be NULL).  W is [128 out, 128 in] with row pitch ldw, as torch stores it.
 * fp16 two-piece operands with a per-32-row-block power-of-two scale (csrc/tc_bwd.cu); deterministic.
 * work: float [gnc_tc_bwd_layer_workspace()]. */
int64_t gnc_tc_bwd_layer_workspace(void);
int gnc_tc_bwd_layer_f32(const float* dZ, int64_t lddz, const float* X, int64_t ldx, int64_t M,
                         const float* W, int64_t ldw, int mask_by_x, const float* addend, int64_t ld_addend,
                         float* dX, int64_t lddx, float* dW, int64_t lddw, float* db, int accumulate,
                         float* work, int64_t work_elems, gnc_stream_t stream);

/* Deferred form for a whole backward pass: with dW = db = NULL the launch above leaves its per-CTA partial sums in
 * `work` (gnc_tc_bwd_layer_parts(M) slices); every layer of the pass uses its own `work`, and ONE launch of the batch
 * reduction then finishes all of them in the same fixed order (same bits as the immediate form). */
typedef struct gnc_bwd_reduce_item {
  const float* work;   /* the layer's workspace */
  float* dW;           /* [128, 128], row pitch lddw; may be NULL */
  float* db;           /* [128]; may be NULL */
  int64_t lddw;
  int32_t parts;       /* gnc_tc_bwd_layer_parts(M) of that layer */
  int32_t accumulate;  /* add to dW / db instead of overwriting */
} gnc_bwd_reduce_item_t;
int32_t gnc_tc_bwd_layer_parts(int64_t M);
int gnc_tc_bwd_reduce_batch_f32(const gnc_bwd_reduce_item_t* items, int32_t n_items, gnc_stream_t stream);

/* Linear(D, 1) as a row dot product (the decoder's last layer, models/GNN.py:289-295):  y[m] = X[m, :] . w + b.
 * Backward in one pass over X:  dX[m, :] = dy[m] * w  (* (X[m, :] > 0) with relu_mask: X is a ReLU output and dX its
 * pre-activation gradient; dX may be NULL),  dw[D] (+)= sum_m dy[m] X[m, :],  db[1] (+)= sum_m dy[m].
 * D % 4 == 0, D <= 512.  work: float [gnc_dot_tail_bwd_workspace(M, D)]; fixed-order reductions (deterministic). */
int gnc_dot_tail_fwd_f32(const float* X, int64_t ldx, int64_t M, int D, const float* w, const float* b /*may be NULL*/,
                         float* y, gnc_stream_t stream);
int64_t gnc_dot_tail_bwd_workspace(int64_t M, int D);
int gnc_dot_tail_bwd_f32(const float* X, int64_t ldx, int64_t M, int D, const float* w, const float* dy, int relu_mask,
                         float* dX, int64_t lddx, float* dw, float* db, int accumulate,
                         float* work, int64_t work_elems, gnc_stream_t stream);

/* Loss and optimizer of the training step (reference utils/train_model.py:9-10, 38-42: nn.CrossEntropyLoss, Adam).
 * cross_entropy: loss[0] = scale * sum_b CE(logits[b, :], labels[b]), the same value added to total[0] (either pointer
 * may be NULL, not both) and, when dlogits is given,
 * dlogits[b, c] = scale * (softmax(logits[b])[c] - [c == labels[b]]); labels are int64; *bad_label_flag (device int, may
 * be NULL) is set to 1 when a label is outside [0, C).  One launch, fixed summation order.
 * adam_step: torch.optim.Adam's update (no weight decay, no amsgrad) over flat fp32 buffers of n elements, step >= 1 the
 * 1-based step count, gradients read as grad * grad_scale (the data-parallel average).  zero: cudaMemsetAsync. */
int gnc_cross_entropy_f32(const float* logits, int64_t ld, const int64_t* labels, int B, int C, float scale,
                          float* loss, float* total, float* dlogits, int64_t ldd, int* bad_label_flag,
                          gnc_stream_t stream);
int gnc_adam_step_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, double lr,
                      double beta1, double beta2, double eps, int64_t step, float grad_scale, gnc_stream_t stream);
int gnc_zero_f32(float* buf, int64_t n, gnc_stream_t stream);

/* Readout of a batch of graphs with different node counts (node_ptr int32 [B + 1], offsets into y [sum n_b]) into the
 * dense classifier input:  out[b, j] = j < n_b ? y[node_ptr[b] + j] : 0  for j < num_nodes  (pad / truncate to
 * num_nodes; equal to the reference's flatten, models/GNN.py:339, when n_b == num_nodes).  Backward: dy gets dout's
 * entries of the kept nodes and zero for truncated ones. */
int gnc_segment_readout_f32(const float* y, const int32_t* node_ptr, int B, int num_nodes, float* out, gnc_stream_t stream);
int gnc_segment_readout_bwd_f32(const float* dout, const int32_t* node_ptr, int B, int num_nodes, float* dy,
                                gnc_stream_t stream);

/* Connectivity enforcement of SLIC label maps (scikit-image's default post-pass; parity unpinned, the rule is stated in
 * csrc/slic_connect.cu): 4-connected components of equal labels, components smaller than min_size dissolved into the
 * component left of / above their first pixel, survivors numbered 0.. in scan order of their first pixel.
 * labels / out: int32 [B, H, W] (may alias); n_labels: int32 [B] (may be NULL); work: int32 [3 * B * H * W]. */
int64_t gnc_slic_connectivity_workspace(int B, int H, int W);
int gnc_slic_enforce_connectivity(const int32_t* labels, int B, int H, int W, int min_size, int32_t* out, int32_t* n_labels,
                                  int32_t* work, int64_t work_elems, gnc_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GNC_H_ */
