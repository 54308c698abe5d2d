// h264_common.cuh — device-side data layout and the per-4x4-block transform/quantise/reconstruct
// routines shared by the intra and inter macroblock kernels.  One warp encodes one macroblock; inside
// the warp, lane b (0..15) owns luma block blkIdx b and lanes 16..23 own the chroma blocks
// (16..19 Cb, 20..23 Cr).  Encoder decisions follow DESIGN.md §5 (restated on the CPU by oracle/h264_ref.c).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "h264_tables.cuh"
#include "h264_cavlc.cuh"

namespace b2v {

constexpr int MB_I16 = 0, MB_P16 = 1, MB_PCM = 2, MB_I4 = 3;
constexpr int COEF_BLOCKS = 27;            // 0 luma DC | 1..16 luma | 17,18 chroma DC | 19..26 chroma AC
constexpr int MB_BITS_LIMIT = 3200;         // A.3.1: bits of macroblock_layer() per macroblock
constexpr int MB_WORDS = 128;              // per-macroblock bit scratch: 128 x u32 = 4096 bits
constexpr unsigned FULL = 0xffffffffu;

struct __align__(8) MbInfo {
  int16_t mvx, mvy;        // quarter-sample units
  uint8_t type;            // MB_*
  uint8_t i16_mode, chroma_mode;
  uint8_t cbp;             // luma bits 0..3 | chroma << 4
};

// Feedback record of the rate controller / paint-over scheduler.  fb[k & 1] is written after picture k (rc_step, last block of
// its slice scan); picture k is CODED from fb[k & 1] as it stood before that — the state after picture k-2 — because the entropy
// coding of picture k-1, where its size becomes known, overlaps the analysis of picture k on another stream.  The two records
// alternate, so nothing a running kernel reads is ever written concurrently.  Mirrors oracle/h264_ref.c struct rcfb / rc_step.
struct RcFb {
  int32_t qp;              // CBR: QP decided for the picture two ahead (-1 = not initialised)
  int32_t static_run;      // consecutive pictures in which every macroblock was skipped
  int32_t remaining;       // paint-over pictures still to schedule
  int32_t paint;           // the picture that reads this record is coded at the paint-over QP
  long long fullness;      // leaky bucket: bits spent above the target
  long long X;             // complexity of the picture just coded: bits x quantiser step (0 = key frame / unknown)
};
struct RcState {
  RcFb fb[2];
  int32_t last_qp;         // QP of the picture whose slice scan ran last (read by its pack kernel)
  int32_t frames;
  int32_t pic_coded;       // set by the slice scan when a slice holds a non-skipped macroblock; consumed and cleared by rc_step (last slice-scan block)
  int32_t scan_done;       // slice-scan blocks that have finished this picture (the last one runs the rate-control step)
  long long pic_bits;      // RBSP bits of the picture just scanned (rate-control step -> AuHeader.total_bits)
};
constexpr int RC_QP_MIN = 10, RC_QP_MAX = 51, RC_STATIC_PARK = 1 << 20, RC_DEBT_PICTURES = 32;
// quantiser step in Q6 (64 * 2^(qp/6)); complexity X = bits * rc_qs[qp]
__device__ const int32_t rc_qs[52] = {
  64, 72, 81, 91, 102, 114, 128, 144, 161, 181, 203, 228, 256, 287, 323, 362, 406, 456, 512, 575, 645, 724, 813, 912, 1024, 1149,
  1290, 1448, 1625, 1825, 2048, 2299, 2580, 2896, 3251, 3649, 4096, 4598, 5161, 5793, 6502, 7298, 8192, 9195, 10321, 11585, 13004,
  14596, 16384, 18390, 20643, 23170};

struct ChunkAgg; struct ChunkInc;
struct FrameCtx {          // everything a kernel needs about the picture being coded
  int cw, ch, mbw, mbh, slice_rows, n_slices;   // n_slices: of THIS picture
  int seg_cols;            // > 0 (IDR pictures): slices of seg_cols macroblocks inside a row, whatever slice_rows is — the macroblocks
                           // of an intra slice are a serial chain, so shorter slices shorten the chain (DESIGN.md §5.2); 0 = whole rows
  int idr, rc_mode, qp_fixed;
  int paint_trigger, paint_qp, paint_burst;   // paint-over: `paint_burst` refinement pictures after `paint_trigger` all-skipped pictures (0 = off)
  int pic;                 // picture counter of this encoder (parity selects the feedback record and the double-buffered side data)
  long long target_bits;
  int frame_num, idr_pic_id;
  const uint8_t* cur;      // NV12 coded size
  const uint8_t* ref;      // previous reconstruction (NV12)
  uint8_t* recon;          // reconstruction being written
  MbInfo* mbinfo;          // this picture's records (double-buffered: the entropy kernels of picture k read them while picture k+1 is analysed)
  const MbInfo* mbinfo_prev;   // the previous picture's records (temporal motion predictor)
  unsigned long long* me_pub;  // [mbs] anchor macroblocks publish (pic+1) << 32 | new-content flag << 16 | (mvx & 0xff) << 8 | mvy & 0xff as soon as motion estimation is done
  int n_anchor;                // anchors of a P picture (one per 4x4 group of macroblocks, groups counted inside each band)
  uint8_t* i4modes;        // [mbs][16] Intra4x4PredMode per block (raster), valid for MB_I4
  int16_t* coef;           // [mbs][27][16]
  uint8_t* nnz;            // [mbs][32]: 0..15 luma raster, 16..19 Cb, 20..23 Cr
  uint32_t* mb_words;      // [mbs][MB_WORDS]
  uint32_t* mb_nbits;      // [mbs]: bit count | I_PCM flag in bit 30 | skip flag in bit 31
  uint32_t* slice_buf;     // [n_slices][slice_words]
  int slice_words;
  uint32_t* slice_size;    // [n_slices] final NAL bytes (start code + header + EP'd payload)
  uint32_t* slice_rbsp;    // [n_slices] RBSP bytes before emulation prevention
  long long* slice_bits;   // [n_slices]
  int* progress;           // [mbh] intra wavefront progress counters
  int chunks_per_slice;    // k_slice_build: blocks per slice (chunks of up to 256 macroblocks), set at launch
  struct ChunkAgg* chunk_agg; struct ChunkInc* chunk_inc;   // [chunks] look-back records of k_slice_build
  int* slice_done;         // [n_slices] chunks of the slice that have finished copying (reset by the last one)
  RcState* rc;
  const uint8_t* param_sets; int param_len;   // SPS+PPS NAL bytes (IDR pictures)
  // bands ("stripes", pixelflux h264_fullframe = False): groups of band_rows macroblock rows, each an independent H.264
  // stream.  Full-frame coding is the one-band case (band_rows = mbh, striped = 0).
  int band_rows, n_bands, striped;
  int param_len_last;      // SPS+PPS of the last band (may be shorter / cropped), stored behind the regular set
  int* band_fn;            // [n_bands] frame_num of each band's next picture (advances only when the band is coded)
  int* band_coded;         // [n_bands] set by the slice scan when a band holds a non-skipped macroblock; cleared by the pack kernel
  int au_data_off;         // bytes from the AuHeader to the first NAL (AuHeader + band table)
  const unsigned long long* csc_ts;            // device stamps of this picture's CSC launch (or null)
  uint8_t* au;             // AuHeader + access unit
  int* overflow;
};

__device__ __forceinline__ int clip3i(int lo, int hi, int v) { return min(hi, max(lo, v)); }
__device__ __forceinline__ int clip255(int v) { return min(255, max(0, v)); }

__device__ __forceinline__ int rc_initial_qp(long long target_bits, int mbs) {
  long long per_mb = target_bits / (mbs > 0 ? mbs : 1);
  return per_mb >= 400 ? 22 : per_mb >= 200 ? 26 : per_mb >= 100 ? 30 : per_mb >= 50 ? 34 : per_mb >= 25 ? 38 : 42;
}
// QP of this picture, from the feedback record it may see (the state after picture pic-2).  oracle/h264_ref.c rc_frame_qp.
__device__ __forceinline__ int frame_qp(const FrameCtx& f) {
  const RcFb& fb = f.rc->fb[f.pic & 1];
  // paint-over: the scene has been static for `paint_trigger` pictures -> `paint_burst` pictures at the (finer) paint-over QP
  const bool paint = f.paint_trigger > 0 && !f.idr && fb.paint;
  if (f.rc_mode == 1) return clip3i(0, 51, paint ? f.paint_qp : f.qp_fixed);
  int q = fb.qp;
  if (q < 0) q = rc_initial_qp(f.target_bits, f.mbw * f.mbh);
  // an IDR in mid-stream is not coded finer than a fresh start with 4x the picture budget would be (bounds the key-frame burst)
  if (f.idr) q = max(q, rc_initial_qp(4 * f.target_bits, f.mbw * f.mbh));
  if (paint && f.paint_qp < q) q = clip3i(0, 51, f.paint_qp);
  return q;
}
// slice geometry (mirrors oracle/h264_ref.c avail_top / avail_left / code_slice)
__device__ __forceinline__ bool top_in_slice(const FrameCtx& f, int mby) { return f.seg_cols ? false : (mby % f.slice_rows) != 0; }
__device__ __forceinline__ bool left_in_slice(const FrameCtx& f, int mbx) { return f.seg_cols ? (mbx % f.seg_cols) != 0 : mbx > 0; }
__device__ __forceinline__ int segs_per_row(const FrameCtx& f) { return f.seg_cols ? (f.mbw + f.seg_cols - 1) / f.seg_cols : 1; }
__device__ __forceinline__ int slice_of(const FrameCtx& f, int mbx, int mby) { return f.seg_cols ? mby * segs_per_row(f) + mbx / f.seg_cols : mby / f.slice_rows; }
struct SliceGeo { int row0, row1, x0, x1, mb0, n_mb; };      // macroblock rows [row0,row1) x columns [x0,x1); mb0 = first macroblock
__device__ __forceinline__ SliceGeo slice_geo(const FrameCtx& f, int s) {
  SliceGeo g;
  if (f.seg_cols) {
    const int segs = segs_per_row(f);
    g.row0 = s / segs; g.row1 = g.row0 + 1; g.x0 = (s - g.row0 * segs) * f.seg_cols; g.x1 = min(f.mbw, g.x0 + f.seg_cols);
  } else { g.row0 = s * f.slice_rows; g.row1 = min(f.mbh, g.row0 + f.slice_rows); g.x0 = 0; g.x1 = f.mbw; }
  g.mb0 = g.row0 * f.mbw + g.x0; g.n_mb = (g.row1 - g.row0) * (g.x1 - g.x0);
  return g;
}

__device__ __forceinline__ int pos_class(int r) { int x = r & 3, y = r >> 2; return ((x | y) & 1) == 0 ? 0 : ((x & y) & 1) ? 1 : 2; }

// forward core transform, rows then columns (exact integer)
__device__ __forceinline__ void fwd4x4(const int in[16], int out[16]) {
  int t[16];
#pragma unroll
  for (int i = 0; i < 4; i++) {
    int a = in[4 * i], b = in[4 * i + 1], c = in[4 * i + 2], d = in[4 * i + 3];
    int s03 = a + d, d03 = a - d, s12 = b + c, d12 = b - c;
    t[4 * i] = s03 + s12; t[4 * i + 1] = 2 * d03 + d12; t[4 * i + 2] = s03 - s12; t[4 * i + 3] = d03 - 2 * d12;
  }
#pragma unroll
  for (int j = 0; j < 4; j++) {
    int s03 = t[j] + t[12 + j], d03 = t[j] - t[12 + j], s12 = t[4 + j] + t[8 + j], d12 = t[4 + j] - t[8 + j];
    out[j] = s03 + s12; out[4 + j] = 2 * d03 + d12; out[8 + j] = s03 - s12; out[12 + j] = d03 - 2 * d12;
  }
}
// 8.5.12.2 inverse transform: rows, columns, (x + 32) >> 6
__device__ __forceinline__ void inv4x4(const int d[16], int r[16]) {
  int t[16];
#pragma unroll
  for (int i = 0; i < 4; i++) {
    int p0 = d[4 * i], p1 = d[4 * i + 1], p2 = d[4 * i + 2], p3 = d[4 * i + 3];
    int e0 = p0 + p2, e1 = p0 - p2, e2 = (p1 >> 1) - p3, e3 = p1 + (p3 >> 1);
    t[4 * i] = e0 + e3; t[4 * i + 1] = e1 + e2; t[4 * i + 2] = e1 - e2; t[4 * i + 3] = e0 - e3;
  }
#pragma unroll
  for (int j = 0; j < 4; j++) {
    int e0 = t[j] + t[8 + j], e1 = t[j] - t[8 + j], e2 = (t[4 + j] >> 1) - t[12 + j], e3 = t[4 + j] + (t[12 + j] >> 1);
    r[j] = (e0 + e3 + 32) >> 6; r[4 + j] = (e1 + e2 + 32) >> 6; r[8 + j] = (e1 - e2 + 32) >> 6; r[12 + j] = (e0 - e3 + 32) >> 6;
  }
}
__device__ __forceinline__ int quant1(int w, int mf, int f, int qbits) {
  int a = (abs(w) * mf + f) >> qbits;
  a = min(a, 2047);
  return w < 0 ? -a : a;
}

struct QuantParams { int mf[3]; int dq[3]; int qbits, f, qshift; };
__device__ __forceinline__ QuantParams make_quant(int qp, bool intra) {
  QuantParams q;
  int m = qp % 6;
#pragma unroll
  for (int c = 0; c < 3; c++) { q.mf[c] = quant_mf[m][c]; q.dq[c] = dequant_v[m][c]; }
  q.qbits = 15 + qp / 6; q.f = (1 << q.qbits) / (intra ? 3 : 6); q.qshift = qp / 6;
  return q;
}

// scan-order position k -> raster index; evaluated at compile time inside unrolled loops
__device__ __forceinline__ constexpr int zz(int k) {
  return k == 0 ? 0 : k == 1 ? 1 : k == 2 ? 4 : k == 3 ? 8 : k == 4 ? 5 : k == 5 ? 2 : k == 6 ? 3 : k == 7 ? 6 :
         k == 8 ? 9 : k == 9 ? 12 : k == 10 ? 13 : k == 11 ? 10 : k == 12 ? 7 : k == 13 ? 11 : k == 14 ? 14 : 15;
}
__device__ __forceinline__ constexpr int pcls(int r) { return (((r & 3) | (r >> 2)) & 1) == 0 ? 0 : (((r & 3) & (r >> 2)) & 1) ? 1 : 2; }

// True when every (AC, if DC_SEPARATE) coefficient of the transformed block w quantises to level 0: quant1() gives 0 exactly when
// |w|*MF + f < 2^qbits, and MF only depends on the position class, so three maxima decide it — a third of the cost of quantising
// the sixteen coefficients one by one.  Exact, not a heuristic: the levels it predicts to be zero ARE zero.
template <bool DC_SEPARATE>
__device__ __forceinline__ bool block_quantises_to_zero(const int w[16], const QuantParams& q) {
  int m[3] = {0, 0, 0};
#pragma unroll
  for (int r = 0; r < 16; r++) {
    if (DC_SEPARATE && r == 0) continue;
    m[pcls(r)] = max(m[pcls(r)], abs(w[r]));
  }
  const int lim = (1 << q.qbits) - q.f;
  return m[0] * q.mf[0] < lim && m[1] * q.mf[1] < lim && m[2] * q.mf[2] < lim;
}

// Quantise one transformed 4x4 block.  lv[k]: scan-order levels.  When dc_separate the
// DC coefficient is returned un-quantised in w_dc and lv[0] = 0.  Returns the number of non-zero levels.
template <bool DC_SEPARATE>
__device__ __forceinline__ int quant_block(const int w[16], const QuantParams& q, int lv[16], int& w_dc) {
  int n = 0;
#pragma unroll
  for (int k = 0; k < 16; k++) {
    if (DC_SEPARATE && k == 0) { w_dc = w[0]; lv[0] = 0; continue; }
    lv[k] = quant1(w[zz(k)], q.mf[pcls(zz(k))], q.f, q.qbits);
    n += lv[k] != 0;
  }
  return n;
}
template <bool DC_SEPARATE>
__device__ __forceinline__ int tq_block(const int res[16], const QuantParams& q, int lv[16], int& w_dc) {
  int w[16];
  fwd4x4(res, w);
  return quant_block<DC_SEPARATE>(w, q, lv, w_dc);
}
// dequantise + inverse transform; when USE_DC the (already dequantised) dc replaces d[0]
template <bool USE_DC>
__device__ __forceinline__ void recon_block(const int lv[16], const QuantParams& q, int dc, int resid[16]) {
  int d[16];
#pragma unroll
  for (int k = 0; k < 16; k++) d[zz(k)] = (lv[k] * q.dq[pcls(zz(k))]) << q.qshift;
  if (USE_DC) d[0] = dc;
  inv4x4(d, resid);
}

// store 16 scan-order levels as int16 (two 16-byte stores)
__device__ __forceinline__ void store_levels(int16_t* dst, const int lv[16]) {
  uint32_t p[8];
#pragma unroll
  for (int i = 0; i < 8; i++) p[i] = ((uint32_t)lv[2 * i] & 0xffffu) | ((uint32_t)lv[2 * i + 1] << 16);
  uint4* d4 = reinterpret_cast<uint4*>(dst);
  d4[0] = make_uint4(p[0], p[1], p[2], p[3]);
  d4[1] = make_uint4(p[4], p[5], p[6], p[7]);
}

// ---------------------------------------------------------------------------------------------
// Per-warp shared memory tile of one macroblock
struct MbTile {
  uint8_t cur_y[16][16];
  uint8_t cur_uv[8][16];     // interleaved Cb,Cr
  uint8_t pred_y[16][16];
  uint8_t pred_uv[8][16];
  uint8_t rec_y[16][16];
  uint8_t rec_uv[8][16];
  int dc[16];                // luma DC exchange (raster block position)
  int dcl[16];
  int16_t lvs[COEF_BLOCKS][16];   // scan-order levels of every block, for the I_PCM size check
};

// Lanes 0..15: luma block `lane` (blkIdx), lanes 16..23: chroma.  Reads cur/pred from the tile, writes levels,
// nnz and the reconstruction into the tile (rec_y / rec_uv), returns cbp (all lanes).
//   INTRA16: luma DC separated + Hadamard (8.5.2 / 8.5.10), cbp luma is 0 or 15.
template <bool INTRA16>
__device__ __forceinline__ int transform_mb(MbTile& t, int lane, int qp, int16_t* coef_mb, uint8_t* nnz_mb, int& luma_bits, int& chroma_bits) {
  const bool is_luma = lane < 16, is_chroma = lane >= 16 && lane < 24;
  const int qpc = chroma_qp_tab[qp];
  const QuantParams q = make_quant(is_chroma ? qpc : qp, INTRA16);
  int lv[16], w[16], res[16], w_dc = 0, n = 0, bx = 0, by = 0, comp = 0;
  // residual of this lane's block.  The two shapes (luma: 4 consecutive bytes per row; chroma: every other byte of 8) differ only in
  // how the 16 samples are picked out; everything from the transform on runs ONCE for the whole warp (lanes 24..31 carry zeros)
  if (is_luma) {
    bx = blk_x[lane] * 4; by = blk_y[lane] * 4;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      uint32_t c = *reinterpret_cast<const uint32_t*>(&t.cur_y[by + i][bx]);
      uint32_t p = *reinterpret_cast<const uint32_t*>(&t.pred_y[by + i][bx]);
#pragma unroll
      for (int j = 0; j < 4; j++) res[4 * i + j] = (int)((c >> (8 * j)) & 255) - (int)((p >> (8 * j)) & 255);
    }
  } else if (is_chroma) {
    comp = (lane - 16) >> 2;
    int b = (lane - 16) & 3;
    bx = (b & 1) * 4; by = (b >> 1) * 4;
    const int sh = 8 * comp;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const uint2 c = *reinterpret_cast<const uint2*>(&t.cur_uv[by + i][bx * 2]), p = *reinterpret_cast<const uint2*>(&t.pred_uv[by + i][bx * 2]);
      res[4 * i + 0] = (int)((c.x >> sh) & 255) - (int)((p.x >> sh) & 255);
      res[4 * i + 1] = (int)((c.x >> (sh + 16)) & 255) - (int)((p.x >> (sh + 16)) & 255);
      res[4 * i + 2] = (int)((c.y >> sh) & 255) - (int)((p.y >> sh) & 255);
      res[4 * i + 3] = (int)((c.y >> (sh + 16)) & 255) - (int)((p.y >> (sh + 16)) & 255);
    }
  } else {
#pragma unroll
    for (int k = 0; k < 16; k++) { lv[k] = 0; res[k] = 0; }
  }
  fwd4x4(res, w);
  // ---- inter macroblock in which NOTHING survives quantisation (the common case on a desktop: static regions, and scrolled
  // regions whose prediction repeats last picture's residual): decided from the transformed coefficients with three maxima per
  // block + the chroma DC Hadamard — no level is computed.  The result is exactly what the full path below would produce
  // (every level 0 -> reconstruction = prediction, nothing stored, cbp 0), so the oracle needs no counterpart. ----
  if (!INTRA16) {
    // AC positions for everybody; the DC position counts for luma only (chroma DC goes through the 2x2 Hadamard below)
    bool z = block_quantises_to_zero<true>(w, q);
    if (is_luma) z = z && abs(w[0]) * q.mf[0] < (1 << q.qbits) - q.f;
    {
      const int b = (lane - 16) & 3, d = is_chroma ? w[0] : 0;
      const int o1 = __shfl_xor_sync(FULL, d, 1), o2 = __shfl_xor_sync(FULL, d, 2), o3 = __shfl_xor_sync(FULL, d, 3);
      // 2x2 Hadamard output b of this component's four DC coefficients (lane b holds d_b; d_(b^x) arrives by xor-shuffle)
      const int s1 = (b & 1) ? -1 : 1, s2 = (b & 2) ? -1 : 1;
      const int tk = d + s1 * o1 + s2 * o2 + s1 * s2 * o3;      // == the tk the full path computes (sign of the whole row is irrelevant for |tk|)
      if (is_chroma) z = z && (abs(tk) * q.mf[0] + 2 * q.f < (1 << (q.qbits + 1)));
    }
    if (__all_sync(FULL, z)) {
      if (is_luma) {
#pragma unroll
        for (int i = 0; i < 4; i++) *reinterpret_cast<uint32_t*>(&t.rec_y[by + i][bx]) = *reinterpret_cast<const uint32_t*>(&t.pred_y[by + i][bx]);
      }
      reinterpret_cast<uint32_t*>(&t.rec_uv[0][0])[lane] = reinterpret_cast<const uint32_t*>(&t.pred_uv[0][0])[lane];
      if (lane < 24) nnz_mb[lane] = 0;
      luma_bits = 0; chroma_bits = 0;
      return 0;
    }
  }
  if (is_luma) n = INTRA16 ? quant_block<true>(w, q, lv, w_dc) : quant_block<false>(w, q, lv, w_dc);
  else if (is_chroma) n = quant_block<true>(w, q, lv, w_dc);
  // ---- coefficient decimation of inter luma (DESIGN.md §5.4; oracle/h264_ref.c encode_inter_mb): block score = 9 if any
  // |level| > 1, else sum over its +-1 levels of {3,2,2,1,1,1,0..}[zeros just below]; an 8x8 quadrant (lanes 4k..4k+3) scoring
  // < 4 is zeroed, the whole luma when the macroblock scores < 6 ------------------------------------------------------
  if (!INTRA16) {
    int sc = 0;
    if (is_luma) {
      int zeros = 0; bool big = false;
#pragma unroll
      for (int k = 0; k < 16; k++) {
        const int v = lv[k];
        if (v == 0) { zeros++; }
        else { big |= abs(v) > 1; sc += zeros == 0 ? 3 : zeros <= 2 ? 2 : zeros <= 5 ? 1 : 0; zeros = 0; }
      }
      if (big) sc = 9;
    }
    int s8 = sc + __shfl_xor_sync(FULL, sc, 1);
    s8 += __shfl_xor_sync(FULL, s8, 2);
    int smb = s8 + __shfl_xor_sync(FULL, s8, 4);
    smb += __shfl_xor_sync(FULL, smb, 8);
    if (is_luma && (s8 < 4 || smb < 6)) {
#pragma unroll
      for (int k = 0; k < 16; k++) lv[k] = 0;
      n = 0;
    }
  }
  // ---- DC paths -------------------------------------------------------------------------------
  int dc_deq = 0;
  if (INTRA16) {
    if (is_luma) t.dc[(by >> 2) * 4 + (bx >> 2)] = w_dc;
    __syncwarp();
    int dl = 0;
    if (is_luma) {   // lane r computes Hadamard output element r = (i,j): sum_ab H[i][a] d[a][b] H[b][j]
      const int r = lane, i = r >> 2, j = r & 3;
      int acc = 0;
#pragma unroll
      for (int a = 0; a < 4; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) {
          // H = [[1,1,1,1],[1,1,-1,-1],[1,-1,-1,1],[1,-1,1,-1]]
          int ha = (i == 0) ? 1 : (i == 1) ? (a < 2 ? 1 : -1) : (i == 2) ? ((a == 0 || a == 3) ? 1 : -1) : ((a & 1) ? -1 : 1);
          int hb = (j == 0) ? 1 : (j == 1) ? (b < 2 ? 1 : -1) : (j == 2) ? ((b == 0 || b == 3) ? 1 : -1) : ((b & 1) ? -1 : 1);
          acc += ha * hb * t.dc[a * 4 + b];
        }
      int v = (acc + 1) >> 1;
      dl = quant1(v, q.mf[0], 2 * q.f, q.qbits + 1);
      t.dcl[r] = dl;
    }
    __syncwarp();
    if (is_luma) {
      // scan-order store of the DC levels: lane k writes level at raster zigzag4x4[k]
      coef_mb[lane] = (int16_t)t.dcl[zigzag4x4[lane]];
      t.lvs[0][lane] = (int16_t)t.dcl[zigzag4x4[lane]];
      const int r = (by >> 2) * 4 + (bx >> 2), i = r >> 2, j = r & 3;
      int acc = 0;
#pragma unroll
      for (int a = 0; a < 4; a++)
#pragma unroll
        for (int b = 0; b < 4; b++) {
          int ha = (i == 0) ? 1 : (i == 1) ? (a < 2 ? 1 : -1) : (i == 2) ? ((a == 0 || a == 3) ? 1 : -1) : ((a & 1) ? -1 : 1);
          int hb = (j == 0) ? 1 : (j == 1) ? (b < 2 ? 1 : -1) : (j == 2) ? ((b == 0 || b == 3) ? 1 : -1) : ((b & 1) ? -1 : 1);
          acc += ha * hb * t.dcl[a * 4 + b];
        }
      const int ls = 16 * q.dq[0];
      dc_deq = qp >= 36 ? (acc * ls) << (q.qshift - 6) : (acc * ls + (1 << (5 - q.qshift))) >> (6 - q.qshift);
    }
  }
  // chroma DC: 2x2 Hadamard across the 4 lanes of a component (xor-shuffles stay inside the group)
  int cdc_level = 0;
  {
    int b = (lane - 16) & 3;
    int o1 = __shfl_xor_sync(FULL, w_dc, 1), o2 = __shfl_xor_sync(FULL, w_dc, 2), o3 = __shfl_xor_sync(FULL, w_dc, 3);
    // value of block index k seen from lane b: k = b ^ x
    int d0, d1, d2, d3;
    d0 = (b == 0) ? w_dc : (b == 1) ? o1 : (b == 2) ? o2 : o3;
    d1 = (b == 1) ? w_dc : (b == 0) ? o1 : (b == 3) ? o2 : o3;
    d2 = (b == 2) ? w_dc : (b == 3) ? o1 : (b == 0) ? o2 : o3;
    d3 = (b == 3) ? w_dc : (b == 2) ? o1 : (b == 1) ? o2 : o3;
    int tk = (b == 0) ? d0 + d1 + d2 + d3 : (b == 1) ? d0 - d1 + d2 - d3 : (b == 2) ? d0 + d1 - d2 - d3 : d0 - d1 - d2 + d3;
    if (is_chroma) cdc_level = quant1(tk, q.mf[0], 2 * q.f, q.qbits + 1);
    int l1 = __shfl_xor_sync(FULL, cdc_level, 1), l2 = __shfl_xor_sync(FULL, cdc_level, 2), l3 = __shfl_xor_sync(FULL, cdc_level, 3);
    int c0 = (b == 0) ? cdc_level : (b == 1) ? l1 : (b == 2) ? l2 : l3;
    int c1 = (b == 1) ? cdc_level : (b == 0) ? l1 : (b == 3) ? l2 : l3;
    int c2 = (b == 2) ? cdc_level : (b == 3) ? l1 : (b == 0) ? l2 : l3;
    int c3 = (b == 3) ? cdc_level : (b == 2) ? l1 : (b == 1) ? l2 : l3;
    int fq = (b == 0) ? c0 + c1 + c2 + c3 : (b == 1) ? c0 - c1 + c2 - c3 : (b == 2) ? c0 + c1 - c2 - c3 : c0 - c1 - c2 + c3;
    if (is_chroma) {
      dc_deq = ((fq * (16 * q.dq[0])) << q.qshift) >> 5;
      // chroma DC levels: coef block 17 + comp, entries 0..3 (rest zero)
      coef_mb[(17 + comp) * 16 + b] = (int16_t)cdc_level;
      t.lvs[17 + comp][b] = (int16_t)cdc_level;
    }
  }
  // ---- inter macroblock whose every level quantised to zero (most of a desktop picture): the reconstruction is the
  // prediction, nothing is coded; skip the inverse transform, the level stores and the size estimate ----
  if (!INTRA16) {
    const unsigned any_ac = __ballot_sync(FULL, n > 0), any_dc = __ballot_sync(FULL, is_chroma && cdc_level != 0);
    if ((any_ac | any_dc) == 0u) {
      if (is_luma) {
#pragma unroll
        for (int i = 0; i < 4; i++) *reinterpret_cast<uint32_t*>(&t.rec_y[by + i][bx]) = *reinterpret_cast<const uint32_t*>(&t.pred_y[by + i][bx]);
      }
      reinterpret_cast<uint32_t*>(&t.rec_uv[0][0])[lane] = reinterpret_cast<const uint32_t*>(&t.pred_uv[0][0])[lane];
      if (lane < 24) nnz_mb[lane] = 0;
      luma_bits = 0; chroma_bits = 0;
      return 0;
    }
  }
  // ---- reconstruction into the tile -------------------------------------------------------------
  int resid[16];
  if (is_luma) {
    if (INTRA16) recon_block<true>(lv, q, dc_deq, resid); else recon_block<false>(lv, q, 0, resid);
#pragma unroll
    for (int i = 0; i < 4; i++) {
      uint32_t p = *reinterpret_cast<const uint32_t*>(&t.pred_y[by + i][bx]);
      uint32_t o = 0;
#pragma unroll
      for (int j = 0; j < 4; j++) o |= (uint32_t)clip255((int)((p >> (8 * j)) & 255) + resid[4 * i + j]) << (8 * j);
      *reinterpret_cast<uint32_t*>(&t.rec_y[by + i][bx]) = o;
    }
    store_levels(coef_mb + (1 + lane) * 16, lv);
    store_levels(&t.lvs[1 + lane][0], lv);
    nnz_mb[(by >> 2) * 4 + (bx >> 2)] = (uint8_t)n;
  } else if (is_chroma) {
    recon_block<true>(lv, q, dc_deq, resid);
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
      for (int j = 0; j < 4; j++) t.rec_uv[by + i][(bx + j) * 2 + comp] = (uint8_t)clip255((int)t.pred_uv[by + i][(bx + j) * 2 + comp] + resid[4 * i + j]);
    store_levels(coef_mb + (19 + (lane - 16)) * 16, lv);
    store_levels(&t.lvs[19 + (lane - 16)][0], lv);
    nnz_mb[16 + (lane - 16)] = (uint8_t)n;
  }
  // ---- coded block pattern -----------------------------------------------------------------------
  unsigned nzmask = __ballot_sync(FULL, n > 0);
  unsigned dcmask = __ballot_sync(FULL, is_chroma && cdc_level != 0);
  int cbp_l;
  if (INTRA16) cbp_l = (nzmask & 0xffffu) ? 15 : 0;
  else cbp_l = ((nzmask & 0x000fu) ? 1 : 0) | ((nzmask & 0x00f0u) ? 2 : 0) | ((nzmask & 0x0f00u) ? 4 : 0) | ((nzmask & 0xf000u) ? 8 : 0);
  int cbp_c = (nzmask & 0xff0000u) ? 2 : (dcmask ? 1 : 0);
  // ---- size estimate for the I_PCM decision and the intra mode decision (DESIGN.md §5.7): exact CAVLC size of every
  // coded block with the longest coeff_token of the four nC tables ----------------------------------------------
  __syncwarp();
  {
    bool coded = false; int start = 0, maxc = 16, nC = NC_WORST;
    if (lane == 0) coded = INTRA16;
    else if (lane <= 16) { coded = (cbp_l >> ((lane - 1) >> 2)) & 1; if (INTRA16) { start = 1; maxc = 15; } }
    else if (lane <= 18) { coded = cbp_c != 0; maxc = 4; nC = NC_CHROMA_DC; }
    else if (lane <= 26) { coded = cbp_c == 2; start = 1; maxc = 15; }
    CountSink cs;
    if (coded) cavlc_block(cs, &t.lvs[lane][start], maxc, nC);
    luma_bits = __reduce_add_sync(FULL, lane <= 16 ? cs.n : 0);
    chroma_bits = __reduce_add_sync(FULL, lane > 16 ? cs.n : 0);
  }
  return cbp_l | (cbp_c << 4);
}

// I_PCM: the reconstruction becomes the source samples, every block counts 16 coefficients for its neighbours' nC.
__device__ __forceinline__ void apply_pcm(MbTile& t, int lane, uint8_t* nnz_mb) {
  const int r8 = lane >> 1, c8 = (lane & 1) * 8;
  *reinterpret_cast<uint2*>(&t.rec_y[r8][c8]) = *reinterpret_cast<const uint2*>(&t.cur_y[r8][c8]);
  if (lane < 16) *reinterpret_cast<uint2*>(&t.rec_uv[r8][c8]) = *reinterpret_cast<const uint2*>(&t.cur_uv[r8][c8]);
  if (lane < 24) nnz_mb[lane] = 16;
}

}  // namespace b2v
