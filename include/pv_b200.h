/* pv_b200.h — C ABI of libpvb200.so: the B200-native (sm_100a) kernels behind the
 * pyannote.video face path (detect -> landmarks -> embed -> track -> cluster).
 *
 * The reference (pyannote-video 1.6.3) is pure Python that binds dlib 19.12 through dlib's
 * Python module; each entry point below names the dlib call site it replaces
 * (paths are relative to the reference checkout):
 *
 *   pyramid / srgemm / detect_decode  <- dlib.get_frontal_face_detector()(rgb, 1)
 *                                        pyannote/video/face/face.py:54,66
 *                                        (as dlib's CNN/MMOD detector, per BASELINE.json north_star)
 *   ert_forward                       <- dlib.shape_predictor.__call__   pyannote/video/face/face.py:58,70
 *   chip_extract / srgemm / embed_*   <- dlib.face_recognition_model_v1.compute_face_descriptor
 *                                        pyannote/video/face/face.py:62,74-75
 *   tracker_*                         <- dlib.correlation_tracker.start_track/update/get_position
 *                                        pyannote/video/tracking.py:203,231,250-251
 *   rect_overlap                      <- TrackingByDetection._match      pyannote/video/tracking.py:129-134
 *   pdist_* / hac_*                   <- scipy pdist + pyannote.algorithms HAC
 *                                        pyannote/video/face/clustering.py:92-119,138-148
 *
 * Conventions
 *   - every function returns int: 0 = ok, <0 = PV_ERR_*; pv_last_error() returns a message.
 *   - every data pointer is a DEVICE pointer owned by the caller (a torch.Tensor.data_ptr())
 *     unless the parameter name says host; outputs are pre-allocated by the caller.
 *   - the library owns only opaque handles from pv_*_create / pv_*_destroy.
 *   - the last argument of every launch is a cudaStream_t passed as void*; launches never
 *     synchronise the host.
 *   - no function has a CPU fallback: without a CUDA device they return PV_ERR_CUDA.
 */
#ifndef PV_B200_H
#define PV_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PV_OK 0
#define PV_ERR_INVALID (-1)
#define PV_ERR_CUDA (-2)
#define PV_ERR_UNSUPPORTED (-3)
#define PV_ERR_DEVICE_TIMEOUT (-4)

const char* pv_last_error(void);
int pv_version(void);
/* number of kernels this library has launched since load (bench.py: gpu_launches) */
int64_t pv_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * srgemm: "shifted-row GEMM", the one tensor-core kernel behind every convolution.
 *
 *   D[q, 0:N] = sum_t  X[q + off_t, col_t : col_t + w_t] * W_t[w_t, N]        q in [0, Q)
 *   Y[dst(q)] = act( scale * D[q] + shift (+ R[res(q)]) )                      if valid(q)
 *
 * X is a row-major bf16 matrix (an activation tensor in one of the row layouts of DESIGN.md);
 * a convolution is a list of taps (row offset, column segment).  128 consecutive rows q form
 * one tile = one 128xN fp32 accumulator in TMEM; operands are staged by TMA into 32/64/128-byte
 * swizzled shared memory and consumed by tcgen05.mma (cta_group::1, kind::f16, bf16 x bf16).
 * ------------------------------------------------------------------------------------------ */
#define PV_SR_MAX_TAPS 9
#define PV_SR_MAX_ENTRIES 192

/* one table entry = one A slab (128 + tail rows of one column segment) and the taps that read it.
 * Consecutive entries between a flag bit0 (opens a ring slot) and bit1 (closes it) share one
 * shared-memory slot and one mbarrier round trip. */
typedef struct PvSrEntry {
  int32_t a_row_off;     /* first row of the A slab, relative to the tile's first row q0          */
  int32_t b_row;         /* first row of this entry's weights in the packed matrix of class cls   */
  int32_t a_smem_off;    /* filled by the library: byte offsets inside the slot                   */
  int32_t b_smem_off;
  uint32_t slot_tx_bytes;/* filled by the library on the entry that opens a slot                  */
  int16_t a_col;         /* first column (element) of the segment inside X                        */
  int16_t cls;           /* segment-width class (0 or 1)                                          */
  int16_t n_taps;        /* taps sharing this slab (1..PV_SR_MAX_TAPS)                            */
  int16_t use_tail;      /* 1: slab = 128 + tail_rows rows, 0: 128 rows                           */
  int16_t flags;         /* bit0: first entry of a slot, bit1: last entry of a slot               */
  int16_t tap_rel[PV_SR_MAX_TAPS + 2]; /* row offset of each tap inside the slab                  */
} PvSrEntry;

/* maps an output grid position (n, y, x) to a row of a destination / residual matrix */
typedef struct PvRowMap {
  int32_t kind;        /* 2: faces side by side ("packed rows", embedder levels 4 / 3): image g = n / img holds img faces at
                             column pitch px, py rows per image:  row = (g*py + y)*w + (n - g*img)*px + x
                          0: padded NHWC  row = n*img + (y+py)*w + (x+px)
                          1: parity split row = plane*plane_rows + n*img + ((y+py)>>1)*w + ((x+px)>>1),
                             plane = ((y+py)&1)*2 + ((x+px)&1)                               */
  int32_t cols;        /* row length in elements                                              */
  int32_t w;           /* grid width of the destination                                       */
  int32_t py, px;
  int64_t img;         /* rows per image                                                      */
  int64_t plane_rows;  /* rows per parity plane (kind 1)                                      */
} PvRowMap;

typedef struct PvSrgemmDesc {
  /* operands (device pointers, bound for the lifetime of the plan) */
  const void* x;        /* bf16 [x_rows, x_cols]                                               */
  int64_t x_rows;
  int32_t x_cols;
  int32_t n_out;        /* N: multiple of 16, 16..256                                          */
  int32_t n_classes;    /* 1 or 2                                                              */
  int32_t class_width[2]; /* 16, 32 or 64 elements                                             */
  const void* w_packed[2]; /* bf16 [w_rows[c], class_width[c]]                                 */
  int64_t w_rows[2];
  int32_t tail_rows;    /* multiple of 8, 0..128                                               */
  int32_t n_entries;
  const PvSrEntry* entries; /* HOST pointer, copied                                            */
  int64_t x_row_stride_bytes; /* 0 = dense (x_cols*2); may be smaller than a row (overlapping rows) */
  int64_t weights_resident_max_bytes; /* keep all weights in smem for the launch if they fit in this many bytes (0 = stream) */
  const float* scale;   /* [N] */
  const float* shift;   /* [N] */
  /* output grid */
  int32_t hq, wq;       /* grid rows / cols per image; q = (n*hq + y)*wq + x                   */
  int32_t oh, ow;       /* valid output extent: y < oh && x < ow                               */
  int32_t relu;
  int32_t out_mode;     /* 0: bf16 rows via dst map; 2: fp32 channel 0 only; 3: fp32 rows (all N) */
  void* out;
  PvRowMap dst;
  const void* resid;    /* bf16 or NULL */
  PvRowMap res;
  int32_t max_ctas;     /* 0 = number of SMs                                                   */
  int32_t acc_split;    /* TMEM accumulators per tile that consecutive MMAs rotate over (0 = auto) */
  int32_t ctas_per_sm;  /* 1, 2 or 4 co-resident CTAs per SM (each gets 1/n of smem and TMEM); 0 = 1 */
  int32_t mma_warps;    /* 1, 2 or 4 MMA-issuing warps per CTA, each with its own accumulator; 0 = 1 */
} PvSrgemmDesc;

int pv_srgemm_create(const PvSrgemmDesc* desc, void** out_handle);
int pv_srgemm_run(void* handle, int64_t q_rows, void* stream);
int pv_srgemm_destroy(void* handle);
/* pipeline shape chosen for a plan (ring depth, slot bytes, weights resident?, TMEM accumulators) */
int pv_srgemm_info(void* handle, int* n_ring, int* slot_bytes, int* resident, int* n_acc, int* acc_split);
/* reads (and clears) the device-side error flag of a plan; 0 = none. Synchronises the stream. */
int pv_srgemm_check(void* handle, void* stream);

/* ------------------------------------------------------------------------------------------
 * detconv: the detector's conv layers 2..7 as 2-D tiled implicit GEMMs (csrc/detconv.cu) — the `con`
 * layers of dlib's MMOD CNN behind face_detector_(rgb, 1), pyannote/video/face/face.py:66.
 *
 *   out[b, oy, ox, n] = act( scale[n] * sum_{kh,kw,c} x[b, oy*s + kh - pad_y, ox*s + kw - pad_x, c] * w[n,c,kh,kw] + shift[n] )
 *
 * x is a plain NHWC bf16 tensor [B, H, pitch, c_in] (pitch >= W, even; columns W..pitch-1 must be zero),
 * zero padding comes from TMA out-of-bounds fill (stride 1: pad = k/2, stride 2: pad 0 — dlib's con_
 * defaults).  One tile = 8 x 16 output pixels = one 128 x N TMEM accumulator; the input patch is loaded
 * once per tile by a 4-D TMA box and every tap's A operand is a UMMA descriptor into that patch.
 * Compiled instances (c_in, n_out, kh, kw, stride, out_f32): (16,32,5,5,2,0) (32,32,5,5,2,0) (32,48,5,5,1,0)
 * (48,48,5,5,1,0) (48,16,9,1,1,1).
 * w_img: device image of the weights exactly as they sit in shared memory — for tap t = kh*KW+kw and
 * 16-channel chunk j an N x 16 tile at byte (t*(c_in/16)+j)*N*32, element (n,k) at
 * (k>>3)*(N*16) + (n>>3)*128 + (n&7)*16 + (k&7)*2   (un-swizzled K-major core matrices).
 * ------------------------------------------------------------------------------------------ */
typedef struct PvDetconvDesc {
  const void* x;         /* bf16 [B, H, pitch, c_in]                                            */
  int32_t B, H, W, pitch;
  int32_t c_in, n_out, kh, kw, stride, out_f32;
  const void* w_img;
  int64_t w_bytes;       /* kh*kw*(c_in/16)*n_out*32                                            */
  const float* scale;    /* [n_out] */
  const float* shift;    /* [n_out] */
  int32_t relu;
  void* out;             /* bf16 (or f32 when out_f32) [B, OH, out_pitch, out_cs]               */
  int32_t out_pitch, out_cs;
  /* rsconv only (embedder levels 4 / 3, faces side by side in one image row): */
  const void* resid;     /* optional bf16, same geometry as `out`: added before the ReLU (dlib add_prev)      */
  int32_t gap_period;    /* > 0: output columns x with x % gap_period == gap_pos are written as zeros         */
  int32_t gap_pos;       /*      (the zero column between two faces = the padding of both)                    */
} PvDetconvDesc;

int pv_detconv_create(const PvDetconvDesc* desc, void** out_handle);
int pv_detconv_run(void* handle, int B, void* stream);     /* first B images (B <= desc->B)      */
int pv_detconv_destroy(void* handle);
int pv_detconv_info(void* handle, int* n_stages, int* smem_bytes, int* tiles_x, int* tiles_y);
/* reads (and clears) the device-side error flag; 0 = none. Synchronises the stream. */
int pv_detconv_check(void* handle, void* stream);

/* ------------------------------------------------------------------------------------------
 * rsconv: the same layers as detconv, "row-streaming" decomposition (csrc/rsconv.cu) — default.
 * A work item is 128 output columns x seg_rows output rows; every input row is loaded once (one TMA box)
 * and multiplied, per filter column kw and 16-channel chunk, against ALL filter rows that use it side by
 * side ([W_kh(r_lo) | ... | W_kh(r_hi)], N up to 5*48 = 240), accumulating into a ring of TMEM row slots
 * (one 128 x n_out accumulator per output row).  Same PvDetconvDesc, same instances, different weight image:
 * for parity class q = kh mod stride (stride 1: only q = 0), filter column kw and chunk j one tile of
 * nq*n_out rows x 16 k (32 bytes per row), rows ordered by DECREASING kh (block b holds kh = q + stride*(nq-1-b));
 * K-major with the 32-byte swizzle: element (nn,k) at nn*32 + (((k>>3) ^ ((nn>>2)&1)) * 16) + (k&7)*2;
 * tiles ordered [q][kw][j].
 * ------------------------------------------------------------------------------------------ */
int pv_rsconv_create(const PvDetconvDesc* desc, void** out_handle);
int pv_rsconv_run(void* handle, int B, void* stream);
int pv_rsconv_destroy(void* handle);
int pv_rsconv_info(void* handle, int* n_stages, int* smem_bytes, int* strips, int* segs, int* seg_rows);
int pv_rsconv_check(void* handle, void* stream);
/* role timing of the last launch when the plan was created with PV_RS_DEBUG set: out8 (HOST) = cycles summed over
 * CTAs {MMA: wait slot, wait data, issue, input rows; epilogue: wait row, work, total; 0} */
int pv_rsconv_debug(void* handle, long long* out8);

/* ------------------------------------------------------------------------------------------
 * c12: detector conv1 (5x5 s2, RGB -> 16) + conv2 (5x5 s2, 16 -> 32), each with affine + ReLU, as ONE strip kernel
 * (csrc/c12.cu): the conv1 activations stay in shared memory / TMEM (232 MB per 1080p frame less HBM traffic each
 * way).  Replaces pv_conv1_fused + the first pv_rsconv launch behind face_detector_(rgb, 1),
 * pyannote/video/face/face.py:66.  plane: RGBA u8 [B,Hp,Wp,4] (A = 0: padding), Wp % 4 == 0.
 * w1_img (4096 B): eight blocks of 16 output channels x 16 k, 32-byte rows with the 32-byte swizzle (element (nn,k) of a
 * tile at nn*32 + (((k>>3) ^ ((nn>>2)&1))*16) + (k&7)*2, nn counted from the tile's first block):
 *   tile M0 = blocks [kh4, kh2, kh0], tile M1 = [kh3, kh1] with k = kw*4 + c (kw 0..3, c 0..2, c = 3 zero);
 *   tile P  = blocks [(kh4|0), (kh2|kh3), (kh0|kh1)] with k < 8: (kw 4, c = k) of the even plane row (k 3..7 zero),
 *             k >= 8: the same of the odd plane row.
 * w2_img (25600 B): the rsconv weight image of a (16 -> 32, 5x5, stride 2) layer.
 * out: bf16 [B, OH2, out_pitch, 32], OH1 = (Hp-5)/2+1, OH2 = (OH1-5)/2+1 (same for W).
 * ------------------------------------------------------------------------------------------ */
typedef struct PvC12Desc {
  const void* plane;
  int32_t B, Hp, Wp;
  const void* w1_img;
  int64_t w1_bytes;
  const void* w2_img;
  int64_t w2_bytes;
  const float* scale1;   /* [16] */
  const float* shift1;
  const float* scale2;   /* [32] */
  const float* shift2;
  void* out;
  int32_t out_pitch;
  const float* mean_host; /* 3 floats (HOST): pixel mean; input = (v - mean)/256 */
} PvC12Desc;
int pv_c12_create(const PvC12Desc* desc, void** out_handle);
int pv_c12_run(void* handle, int B, void* stream);
int pv_c12_destroy(void* handle);
int pv_c12_info(void* handle, int* smem_bytes, int* strips, int* segs, int* seg_rows, int* oh2, int* ow2);
int pv_c12_check(void* handle, void* stream);
/* role timing of the last launch when the plan was created with PV_C12_DEBUG set: out16 (HOST) = cycles summed over CTAs
 * {conv1 MMA: wait pixels, issue + slot waits (tile 1), issue + slot waits (tile 0), quads; conv2 MMA: wait A rows, wait slot, issue, rows; converter: wait raw,
 * wait slot, work; conv1 epilogue: wait row, wait A slot, work; conv2 epilogue: wait row, work} */
int pv_c12_debug(void* handle, long long* out16);

/* ------------------------------------------------------------------------------------------
 * host-side tracking control in C++ (csrc/control.cu, no device code; SURVEY.md §8(f) row f3): the per-frame
 * association and the per-shot link graph of TrackingByDetection — pyannote/video/tracking.py:129-182 (_match,
 * _associate: overlap matrix with the min-overlap rule, Munkres on max - overlap, pairs with overlap > 0),
 * :209-244,340-347 (link graph, connected components in node insertion order), :261-296 (_fix) and :298-329
 * (_fill_gaps).  Rectangles are drectangles (l,t,r,b doubles, area (r-l)(b-t)); status codes 0 forward, 1 detection,
 * 2 backward.
 * ------------------------------------------------------------------------------------------ */
/* match[d] = index of the tracker associated with detection d, or -1 */
int pv_ctl_associate(const double* positions, int n_trackers, const double* detections, int n_detections,
                     double min_overlap_ratio, int* match);
int pv_ctl_shot_create(void** out_handle);
int pv_ctl_shot_destroy(void* handle);
int pv_ctl_shot_add(void* handle, double t, const double* box, int status);
int pv_ctl_shot_link(void* handle, double ta, const double* box_a, int sa, double tb, const double* box_b, int sb);
/* components -> _fix -> _fill_gaps -> sorted by (first, last time): sizes first, then the rows */
int pv_ctl_shot_finish(void* handle, double min_overlap_ratio, double max_gap, int* n_tracks, int* n_rows);
/* track_len [n_tracks]; per row: time, integer box (l,t,r,b), counts {forward, detection, backward, error flag} */
int pv_ctl_shot_tracks(void* handle, int* track_len, double* row_t, long long* row_box, int* row_counts);

/* ------------------------------------------------------------------------------------------
 * HOG frontal face detector (csrc/hog.cu): dlib.get_frontal_face_detector()(rgb, 1), the detector the reference
 * really calls (pyannote/video/face/face.py:54,66).  Input = the tiled pyramid plane of pv_resize_bilinear /
 * pv_pyramid_tail; per usable level (both sides >= 80 px) a table entry.  pv_hog_features writes the 31-channel
 * Felzenszwalb features (cell 8) of every interior cell as bf16 x 32 channels into a feature plane
 * [B, FH, fpitch, 32] at (fy0 + y, fx0 + x) (tiles at least 10 zero cells apart; the plane is zeroed once by the
 * caller).  The sliding-window scores are ONE pv_rsconv launch over that plane (instance c_in 32, n_out 16, 10x10,
 * stride 1, fp32 out; filters = output channels).  pv_hog_decode thresholds, sorts (score desc, level, filter, row,
 * col) and applies greedy NMS (dlib test_box_overlap); boxes through fhog_to_image, pyramid_down<6>::rect_up and,
 * when `upsampled`, pyramid_down<2>::rect_down.  counts < 0 reports a candidate overflow.
 * ------------------------------------------------------------------------------------------ */
#define PV_HOG_MAX_LEVELS 24
typedef struct PvHogLevel {
  int32_t x0, y0, w, h;     /* level rectangle in the plane (pixels)                         */
  int32_t cx, cy;           /* cells: (int)(w / 8.f + 0.5f), same for h                       */
  int32_t fx0, fy0;         /* origin of the level's (cy-2) x (cx-2) feature tile             */
  int32_t px_off, cell_off, feat_off;   /* prefix sums of w*h, cx*cy, (cx-2)*(cy-2)           */
} PvHogLevel;
typedef struct PvHogGeo {
  int32_t n_levels, Hp, Wp;
  int32_t total_px, total_cells, total_feat;
  int32_t FH, FW, fpitch;
  PvHogLevel lv[PV_HOG_MAX_LEVELS];
} PvHogGeo;
/* uv18: device float[18] = cos(o*pi/9) (o < 9) then sin(o*pi/9); ori/mag: plane-sized scratch (u8 / f32 per pixel);
 * hist f32 [B, total_cells, 18]; nrm f32 [B, total_cells] */
int pv_hog_features(const void* plane_rgba, int B, const PvHogGeo* geo, const float* uv18, void* ori_u8, void* mag_f32,
                    float* hist, float* nrm, void* feat_bf16, void* stream);
/* scores: fp32 [B, OHs, opitch, 16] (the rsconv output; OHs = FH + 1); thr_dev: device float[D]; D <= 8 filters;
 * cand_*: [B, cap]; out_boxes int32 [B, max_det, 4] (l,t,r,b), out_scores f32, out_which int32 (filter index) */
int pv_hog_decode(const float* scores, int B, int OHs, int opitch, const PvHogGeo* geo, const float* thr_dev, int D,
                  int upsampled, double iou_thresh, double covered_thresh, int cap, int max_det, int* counts,
                  float* cand_score, int* cand_code, int* out_boxes, float* out_scores, int* out_which, int* out_counts,
                  void* stream);

/* ------------------------------------------------------------------------------------------
 * first-layer packing and the small layers of the embedder (csrc/layers.cu)
 * ------------------------------------------------------------------------------------------ */
/* RGBA u8 [B,H,W,4] (A==0: pyramid padding) -> "gathered" bf16 rows for a kw x kw stride-2 first conv:
 * out[ph*layout_plane_rows + (n*ceil(H/2)+i)*ceil(W/2)+j][k*3+c] = (img[n,2i+ph,2j+k,c]-mean[c])/256.
 * dlib input_rgb_image(_pyramid/_sized)::to_tensor. kw = 5 (16 cols) or 7 (32 cols). mean_host: 3 floats (HOST). */
int pv_pack_gathered(const void* rgba, void* out, int B, int H, int W, int kw, int64_t layout_plane_rows,
                     const float* mean_host, void* stream);
/* RGBA u8 plane -> normalised bf16 RGBX pixels split by row parity (the in-place first-layer input:
 * srgemm reads 8-pixel runs with x_row_stride_bytes = 16).  layout_plane_rows = rows of one parity plane
 * of the layout (pixel pairs), W even. */
int pv_plane_to_pixrows(const void* rgba, void* out, int B, int H, int W, int64_t layout_plane_rows,
                        const float* mean_host, void* stream);
/* first detector conv (5x5 stride 2, RGB -> 16) fused with input normalisation: reads the RGBA u8 plane
 * [B,Hp,Wp,4] in place (TMA, Wp % 4 == 0) and feeds tcgen05.mma from a normalised pixel-row buffer in
 * shared memory (csrc/conv1_fused.cu).  w_bf16 [16][3][5][5] (dlib order), scale/shift f32 [16],
 * oh = (Hp-5)/2+1, ow = (Wp-5)/2+1, out rows via `dst`, err_flag: device int. */
int pv_conv1_fused(const void* plane_rgba, int B, int Hp, int Wp, const void* w_bf16, const float* scale,
                   const float* shift, int relu, void* out, const PvRowMap* dst, int oh, int ow, const float* mean_host,
                   int* err_flag, void* stream);
/* role timing of the last pv_conv1_fused launch when the environment variable PV_C1_DEBUG is set: out8 (HOST) =
 * cycles summed over CTAs {MMA: wait accumulator, wait pixels, issue, tiles; converter: wait raw, wait slot, work;
 * epilogue: wait} */
int pv_conv1_debug(long long* out8);
/* packed-rows tensors [G][H][Wp][C] (F faces per image row at pitch W+1): dlib avg_pool<2,2,2,2> per face, channels
 * zero-extended Cin -> Cout (ares_down skip path), and the hand-over to a PvRowMap layout */
int pv_pr_avgpool(const void* in, int G, int F, int H, int W, int Wp, int Cin, void* out, int OWp, int Cout, void* stream);
int pv_pr_unpack(const void* in, int B, int F, int H, int W, int Wp, int C, void* out, const PvRowMap* dst, void* stream);
/* dlib max_pool<3,3,2,2> (pad 0) on bf16 NHWC [B,H,W,C] -> rows of `dst` */
int pv_maxpool3x3s2(const void* in, void* out, int B, int H, int W, int C, const PvRowMap* dst, void* stream);
/* dlib avg_pool<2,2,2,2> skip path of ares_down: parity-layout input -> skip (zero-extended to Cout)
 * and relu(skip) pre-written into the block output */
int pv_avgpool_skip(const void* in, int Cin, int64_t in_plane_rows, int in_hq, int in_wq, void* skip, void* out, int B,
                    int OH, int OW, int Cout, const PvRowMap* dst, void* stream);
/* avg_pool_everything + fc_no_bias<128>: bf16 [B,HW,C] -> float [B,D] */
int pv_embed_head(const void* in, int B, int HW, int C, const float* fc, float* out, int D, void* stream);

/* ------------------------------------------------------------------------------------------
 * detector input/output stages (csrc/detect.cu) — dlib pyramid_up / pyramid_down<6> /
 * loss_mmod::to_label around face_detector_(rgb, 1), pyannote/video/face/face.py:66
 * ------------------------------------------------------------------------------------------ */
/* bilinear resize (dlib resize_image + interpolate_bilinear) of a sub-rectangle of `src`
 * (3 or 4 u8 channels) into a sub-rectangle of the RGBA plane; copy_only=1 copies 1:1. */
int pv_resize_bilinear(const void* src, int src_channels, int64_t src_img_stride_bytes, int src_pitch_px, int sx0,
                       int sy0, int sw, int sh, void* dst_rgba, int64_t dst_img_stride_px, int dst_pitch_px, int dx0,
                       int dy0, int dw, int dh, float xs, float ys, int B, int copy_only, void* stream);
/* the small levels of the pyramid in ONE launch: one CTA per image builds levels k0..L-1 in order, each
 * from its predecessor inside the plane. rects_host i32 [(n_levels+1),4] (source level first), scales_host
 * f32 [n_levels,2]; both HOST arrays. */
int pv_pyramid_tail(void* plane_rgba, int64_t img_stride_px, int pitch_px, int B, int n_levels, const int* rects_host,
                    const float* scales_host, void* stream);
/* the 9x9 single-channel last conv runs as a 9x1 conv with the filter columns as channels;
 * score[n,y,x] = bias + sum_kw D[(n*Hq+y)*Wq + x+kw][kw] re-assembles it (D fp32 [rows, cols]) */
int pv_det_shift_sum(const float* D, int B, int Hq, int Wq, int cols, int OH, int OW, int KW, float bias, float* scores,
                     void* stream);
/* same re-assembly over the un-padded NHWC partials of detconv: P fp32 [B, H, pitch, cols] computed at the
 * un-padded positions; score[n,y,x] = bias + sum_kw P[n, y, x+kw-KW/2][kw], out-of-range columns contribute 0 */
int pv_det_shift_sum_nhwc(const float* P, int B, int H, int W, int pitch, int cols, int KW, float bias, float* scores,
                          void* stream);
/* cells of the score map above `thr` -> per-frame candidate lists (counts are zeroed first) */
int pv_det_candidates(const float* scores, int B, int cells, float thr, int* counts, float* cand_score, int* cand_cell,
                      int cap, void* stream);
/* candidates -> boxes in image space (integer, inclusive), sorted by score, greedy NMS with
 * dlib test_box_overlap(iou_thresh, covered_thresh); out_counts[n] < 0 reports candidate overflow */
int pv_det_nms(const int* counts, const float* cand_score, const int* cand_cell, int cap, int B, const int* level_rects,
               const float* level_fxy, int n_levels, int window, int ow, int cell_mul, int cell_add, double iou_thresh,
               double covered_thresh, int max_det, int* out_boxes, float* out_scores, int* out_counts, void* stream);

/* ------------------------------------------------------------------------------------------
 * landmarks and chips (csrc/landmarks.cu)
 * ------------------------------------------------------------------------------------------ */
/* dlib.shape_predictor (pyannote/video/face/face.py:58,70).  All model arrays are device pointers
 * that must outlive the handle: initial_shape f32[136], anchor_idx i32[S,P], deltas f32[S,P,2],
 * split_idx1/2 i32[S,T,15], split_thresh f32[S,T,15], leaf_values f32[S,T,16,136]. */
int pv_ert_create(const float* initial_shape, const int* anchor_idx, const float* deltas, const int* split_idx1,
                  const int* split_idx2, const float* split_thresh, const float* leaf_values, int stages, int trees,
                  int pool, void** out_handle);
int pv_ert_destroy(void* handle);
/* frames u8 [F,H,W,3]; rects i32 [M,4] (l,t,r,b); frame_idx i32 [M] -> out_parts i32 [M,68,2] */
int pv_ert_forward(void* handle, const void* frames, int H, int W, const int* rects, const int* frame_idx, int M,
                   int* out_parts, void* stream);
/* get_face_chip_details + extract_image_chip of compute_face_descriptor (face/face.py:74-75):
 * parts i32 [M,68,2] -> RGBA u8 chips [M,size,size,4]; from_pts f32 [68,2] chip-space targets,
 * pt_idx i32 [n_idx] the landmarks used for the similarity fit */
int pv_chip_extract(const void* frames, int H, int W, const int* parts, const int* frame_idx, int M,
                    const float* from_pts, const int* pt_idx, int n_idx, int size, void* out_rgba, void* stream);

/* ------------------------------------------------------------------------------------------
 * clustering (csrc/cluster.cu) — pyannote/video/face/clustering.py:92-119,138-148
 * ------------------------------------------------------------------------------------------ */
/* D[i][j] = ||x_i - x_j|| (metric 0, scipy pdist 'euclidean') or 1 - cos (metric 1); X f32 [n,128] */
int pv_pdist(const float* X, int64_t n, int dim, int metric, float* D, void* stream);
/* the same matrix from the tensor cores (csrc/gram.cu): <x_i, x_j> as a bf16 x 3 split GEMM with fp32 TMEM accumulation
 * (six products, error ~2^-24), distance epilogue fused.  Workspaces: xs_ws = 3 * npad * 128 bf16, norms_ws = npad floats,
 * npad = pv_gram_npad(n); err_flag: device int set by a pipeline timeout (may be NULL). */
int64_t pv_gram_npad(int64_t n);
int pv_gram_dist(const float* X, int64_t n, int dim, int metric, float* D, void* xs_ws, float* norms_ws, int* err_flag,
                 void* stream);
/* S' = P S P^T in two passes; CSR (offs i32 [tout+1], memb i32) lists the old clusters of each new one */
int pv_pool_rows(const float* S, int64_t tin, const int* offs, const int* memb, float* R, int64_t tout, void* stream);
int pv_pool_cols(const float* R, int64_t tin, const int* offs, const int* memb, float* Sout, int64_t tout, void* stream);
/* nearest cluster of every cluster under average linkage S[A][C]/(size_A*size_C) */
int pv_row_argmin(const float* S, int64_t t, const float* sizes, int* nn, float* nnd, void* stream);
/* one agglomeration round on the device (pyannote.algorithms' greedy loop behind clustering.py:138-148, as rounds of
 * reciprocal-nearest-neighbour merges): plan -> (caller: exclusive prefix sum of keep) -> members -> contract -> relabel */
int pv_hac_plan(const int* nn, const float* nnd, int64_t t, float threshold, int strict, int* keep, int* partner, void* stream);
int pv_hac_members(const int* keep, const int* partner, const int* newidx, const int* nn, const float* sizes, int64_t t,
                   int* m0, int* m1, float* sizes2, int* map, void* stream);
int pv_hac_contract(const float* S, int64_t t, const int* m0, const int* m1, float* S2, int64_t tout, void* stream);
int pv_hac_relabel(int* cl, int64_t n, const int* map, void* stream);
/* whole-stage form for one-embedding-per-track inputs (what a non-Python consumer binds instead of the Python loop in
 * clustering.py): X f32 [n][128] (device) -> labels i32 [n] (device), label = smallest row index of the row's cluster.
 * Allocates its work space (2 n^2 floats + the Gram operands) and synchronises the stream once per round.
 * rounds_out: HOST int or NULL. */
int pv_hac_threshold(const float* X, int64_t n, int dim, int metric, float threshold, int strict, int* labels, int* rounds_out,
                     void* stream);
/* TrackingByDetection._match (pyannote/video/tracking.py:129-134), HOST function on (l,t,r,b) doubles in dlib drectangle
 * arithmetic: intersection area, or 0 unless it covers at least `ratio` of both rectangles */
double pv_rect_overlap(const double* a_ltrb, const double* b_ltrb, double ratio);

/* ------------------------------------------------------------------------------------------
 * correlation-tracker bank (csrc/tracker.cu) — dlib.correlation_tracker start_track / update /
 * get_position, pyannote/video/tracking.py:203,231,250-251; one CTA per live track
 * ------------------------------------------------------------------------------------------ */
/* tables are HOST float arrays: cosine window [64], FHOG orientation cos/sin [9], FFT twiddles [32] */
int pv_tracker_create(int capacity, const float* hann64_host, const float* uu9_host, const float* vv9_host,
                      const float* tw_re32_host, const float* tw_im32_host, float padding, float lambda, float nu,
                      void** out_handle);
int pv_tracker_destroy(void* handle);
/* enable the 1-D scale filter of dlib's update(): 32 scales alpha^(k-16), 23x23 windows, FHOG cell 4.
 * Tables are HOST float[32]: Hann over scales, alpha^(k-16), DFT twiddles exp(-2 pi i m/32). */
int pv_tracker_enable_scale(void* handle, const float* hann32_host, const float* factor32_host, const float* tw_re32_host,
                            const float* tw_im32_host, double alpha, float lambda, float nu);
/* frame u8 [H,W,3]; ids i32 [n] bank slots; rects f32 [n,4] (l,t,r,b) */
int pv_tracker_start(void* handle, const void* frame, int H, int W, const int* ids, const float* rects, int n,
                     void* stream);
int pv_tracker_update(void* handle, const void* frame, int H, int W, const int* ids, int n, void* stream);
/* batched forms (tracks of many shots advance in one launch): frames u8 [F,H,W,3], frame_idx i32 [n] = frame of
 * track ids[i] (NULL: all tracks read frame 0) */
int pv_tracker_start_frames(void* handle, const void* frames, int H, int W, const int* frame_idx, const int* ids,
                            const float* rects, int n, void* stream);
int pv_tracker_update_frames(void* handle, const void* frames, int H, int W, const int* frame_idx, const int* ids, int n,
                             void* stream);
/* device pointers owned by the bank: positions f32 [capacity,4] and PSR f32 [capacity] */
int pv_tracker_state(void* handle, float** pos, float** psr);

/* ------------------------------------------------------------------------------------------
 * shot boundary detection (csrc/shot.cu) — pyannote/video/structure/shot.py: gray + resize, Farneback optical
 * flow (pyr_scale 0.5, 3 levels, winsize 15, 3 iterations, poly_n 5, poly_sigma 1.1, box-filter update) and the
 * displaced frame difference of every consecutive pair.  Geometry and tables are built by pyannote_video_b200/shot.py.
 * ------------------------------------------------------------------------------------------ */
#define PV_SHOT_MAX_LEVELS 4
#define PV_SHOT_MAX_TAPS 19
#define PV_SHOT_POLY_N 5
#define PV_SHOT_WINSIZE 15
#define PV_SHOT_ITERATIONS 3
typedef struct PvShotLevel {
  int32_t rows, cols;
  int32_t r_off;            /* float offset of the level's R [5, rows, cols] in a frame's R block            */
  int32_t radius;           /* pre-blur radius (taps = 2 * radius + 1), reflect-101 border                     */
  int32_t area2x;           /* 1: the level is an exact 2x downscale of level 0 (2x2 mean)                    */
  int32_t dn_off;           /* float offset in tab of the level-0 -> level resize table (-1: none)             */
  int32_t up_off;           /* float offset in tab of the coarser-level -> level flow resize table (-1: none)  */
  float taps[PV_SHOT_MAX_TAPS];
} PvShotLevel;
typedef struct PvShotGeo {
  int32_t h, w;             /* level-0 gray frame: rows, columns                                               */
  int32_t n_levels;         /* lv[0] is the coarsest level, lv[n_levels - 1] is level 0                        */
  int32_t r_stride;         /* floats of one frame's R block (all levels)                                      */
  PvShotLevel lv[PV_SHOT_MAX_LEVELS];
  float pg[2 * PV_SHOT_POLY_N + 1], pxg[2 * PV_SHOT_POLY_N + 1], pxxg[2 * PV_SHOT_POLY_N + 1];
  int32_t pad_;
  double ig11, ig03, ig33, ig55;
} PvShotGeo;
/* RGB u8 [B,H,W,3] -> gray u8 [B,h,w]; tab: device int32 x0 x1 cx0 cx1 [w] then y0 y1 cy0 cy1 [h] (11-bit weights) */
int pv_shot_gray_resize(const void* rgb, int B, int H, int W, const int* tab, int h, int w, void* out, void* stream);
/* global workspace floats per CTA when the shared-memory budget is exceeded (-1: bad geometry) */
int64_t pv_shot_polyexp_work_floats(const PvShotGeo* geo);
int64_t pv_shot_flow_work_floats(const PvShotGeo* geo);
/* gray u8 [B,h,w] -> R f32 [B, r_stride]; work: B * n_levels * polyexp_work_floats floats, or NULL if it fits on chip */
int pv_shot_polyexp(const void* gray, int B, const PvShotGeo* geo, const float* tab, float* work, float* R, void* stream);
/* pairs (p, p+1), p < P, of gray u8 [P+1,h,w] and R [P+1, r_stride] -> dfd f64 [P]; flow_out f32 [P,h,w,2] or NULL;
 * work: P * flow_work_floats floats, or NULL if it fits on chip */
int pv_shot_flow_dfd(const void* gray, const float* R, int P, const PvShotGeo* geo, const float* tab, float* work,
                     double* dfd, float* flow_out, void* stream);

/* ------------------------------------------------------------------------------------------
 * shot threading (csrc/orb.cu) — pyannote/video/structure/thread.py: RGB resize then gray, cv2.ORB_create() features
 * (500 features, scale 1.2, 8 levels, edge 31, FAST 20, Harris, patch 31, WTA_K 2) and the exact Hamming 2-NN
 * ratio count (best < 0.7 * second, float64) of shot pairs.  Geometry and tables are built by
 * pyannote_video_b200/thread.py.
 * ------------------------------------------------------------------------------------------ */
#define PV_ORB_LEVELS 8
typedef struct PvOrbGeo {
  int32_t n_levels;
  int32_t rows[PV_ORB_LEVELS], cols[PV_ORB_LEVELS];
  int32_t off[PV_ORB_LEVELS];      /* byte offset of level k in a frame's pyramid plane                             */
  int32_t tab_off[PV_ORB_LEVELS];  /* int offset in tab of level k's INTER_LINEAR_EXACT taps from level k - 1:
                                      x offset [cols], x weight [cols], y offset [rows], y weight [rows] (k >= 1)  */
  int32_t quota[PV_ORB_LEVELS];    /* features kept per level (ties at the cut are all kept)                       */
  float scale[PV_ORB_LEVELS];      /* keypoint coordinate scale of level k (float32 1.2^k)                         */
  float gauss[7];                  /* the 7-tap sigma-2 float32 Gaussian of the descriptor smoothing               */
  int32_t plane;                   /* bytes of one frame's pyramid plane (sum of rows * cols)                      */
  int32_t cand_cap;                /* keypoint slots per frame: bounds the non-max-suppression survivors           */
} PvOrbGeo;
/* RGB u8 [B,H,W,3] -> per channel INTER_LINEAR resize, then RGB2GRAY -> u8 [B,h,w]; tab as pv_shot_gray_resize */
int pv_orb_resize_gray(const void* rgb, int B, int H, int W, const int* tab, int h, int w, void* gray, void* stream);
/* workspace bytes per frame of pv_orb_detect (-1: bad geometry) */
int64_t pv_orb_work_bytes(const PvOrbGeo* geo);
/* gray u8 [B,h,w] -> per frame f: count[f] keypoints (-1: candidate overflow) in kp f32 [B, cand_cap, 5]
 * (x, y, octave, response, angle; sorted by octave, y, x) and desc u8 [B, cand_cap, 32]; work: B * work_bytes */
int pv_orb_detect(const void* gray, int B, const PvOrbGeo* geo, const int* tab, void* work, float* kp, void* desc,
                  int* count, void* stream);
/* desc u8 [N,32] packed by frame (offsets i32 [F+1]); pairs i32 [P,2] (query frame, train frame) -> counts i32 [P]:
 * queries whose best Hamming distance < 0.7 * the second best; 0 when either side has < 2 descriptors */
int pv_thread_match(const void* desc, const int* offsets, const int* pairs, int P, int* counts, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PV_B200_H */
