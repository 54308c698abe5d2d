// h264_encoder.cu — host side of the H.264 Constrained-Baseline encoder: parameter sets (7.3.2.1/2),
// HBM buffers, per-picture sequencing (frame_num, idr_pic_id, reference swap) and the kernel pipeline
//   [k_intra_rows | k_inter_mb] -> k_cavlc_mb -> k_slice_build -> k_pack_au
// The output format is what the reference's consumers require (SURVEY.md §8 a13): Annex-B, CAVLC,
// no B-frames, 4:2:0, in-band SPS/PPS on every IDR (src/selkies/rtc.py:394-401,
// src/selkies/webrtc/codecs/h264.py:281-321).
#include <cstdio>
#include <cstring>
#include <vector>

#include "h264_common.cuh"
#include <algorithm>
#include "b2v_internal.h"
#include "h264_encoder.h"
#include "h264_kernels.h"

namespace b2v {

static thread_local char g_enc_err[256] = "";
const char* encoder_last_error() { return g_enc_err; }

struct Encoder {
  EncoderConfig cfg{};
  int mbw = 0, mbh = 0, n_slices = 0;
  int seg_cols = 0, n_seg_slices = 0, seg_slice_words = 0;   // IDR pictures: sub-row slices (0 = whole rows)
  uint8_t* recon[2] = {nullptr, nullptr};
  int cur = 0;
  // side data the analysis kernels write and the entropy kernels read: double-buffered by picture parity, so the entropy coding
  // of picture k (packing stream) overlaps the analysis of picture k+1 (main stream)
  MbInfo* mbinfo[2] = {nullptr, nullptr};
  uint8_t* i4modes[2] = {nullptr, nullptr};
  int16_t* coef[2] = {nullptr, nullptr};
  uint8_t* nnz[2] = {nullptr, nullptr};
  void *chunk_agg = nullptr, *chunk_inc = nullptr; int* slice_done = nullptr;   // k_slice_build look-back records (h264_entropy.cu)
  unsigned long long* me_pub = nullptr;   // anchor macroblocks' vectors of the picture being analysed (h264_inter.cu)
  uint32_t *mb_words = nullptr, *mb_nbits = nullptr, *slice_buf = nullptr, *slice_size = nullptr, *slice_rbsp = nullptr;
  long long* slice_bits = nullptr;
  int slice_words = 0;
  int* progress = nullptr;
  int* overflow = nullptr;
  RcState* rc = nullptr;
  uint8_t* param_sets = nullptr; int param_len = 0, param_len_last = 0;
  int band_rows = 0, n_bands = 1, striped = 0, au_data_off = (int)sizeof(AuHeader);
  int *band_fn = nullptr, *band_coded = nullptr;
  cudaEvent_t ev_analysed[2] = {nullptr, nullptr}, ev_packed[2] = {nullptr, nullptr};   // two-stream schedule, by picture parity
  long long pic = 0;       // pictures encoded so far
  size_t au_cap = 0;
  int frame_num = 0, idr_count = 0;
  bool have_ref = false;
};

namespace {

struct HostBits {
  std::vector<uint8_t> buf; uint64_t acc = 0; int n = 0;
  void put(int len, uint32_t v) {
    if (!len) return;
    if (len < 32) v &= (1u << len) - 1;
    acc = (acc << len) | v; n += len;
    while (n >= 8) { buf.push_back((uint8_t)(acc >> (n - 8))); n -= 8; }
  }
  void ue(uint32_t v) { uint32_t x = v + 1; int len = 0; while ((x >> len) > 1) len++; put(len, 0); put(len + 1, x); }
  void se(int v) { ue(v > 0 ? (uint32_t)(2 * v - 1) : (uint32_t)(-2 * v)); }
  void trailing() { put(1, 1); if (n) put(8 - n, 0); }
};

void append_nal(std::vector<uint8_t>& out, int ref_idc, int type, const std::vector<uint8_t>& rbsp) {
  out.insert(out.end(), {0, 0, 0, 1});
  out.push_back((uint8_t)((ref_idc << 5) | type));
  int zeros = 0;
  for (uint8_t b : rbsp) {
    if (zeros == 2 && b <= 3) { out.push_back(3); zeros = 0; }
    out.push_back(b);
    zeros = b == 0 ? zeros + 1 : 0;
  }
}

int level_idc_for(int mbs) { return mbs <= 3600 ? 31 : mbs <= 8704 ? 42 : mbs <= 22080 ? 51 : mbs <= 36864 ? 52 : 62; }

std::vector<uint8_t> make_param_sets(const EncoderConfig& c, int mbw, int mbh, int crop_b) {
  std::vector<uint8_t> out;
  HostBits b;
  b.put(8, 66); b.put(8, 0xC0); b.put(8, (uint32_t)level_idc_for(mbw * mbh));
  b.ue(0);                 // seq_parameter_set_id
  b.ue(4);                 // log2_max_frame_num_minus4
  b.ue(2);                 // pic_order_cnt_type
  b.ue(1);                 // max_num_ref_frames
  b.put(1, 0);             // gaps_in_frame_num_value_allowed_flag
  b.ue(mbw - 1); b.ue(mbh - 1);
  b.put(1, 1);             // frame_mbs_only_flag
  b.put(1, 1);             // direct_8x8_inference_flag
  const int crop_r = (c.coded_w - c.width) / 2;
  if (crop_r || crop_b) { b.put(1, 1); b.ue(0); b.ue(crop_r); b.ue(0); b.ue(crop_b); } else b.put(1, 0);
  // E.1.1 VUI: BT.709 limited-range colour description, centre-sited chroma, no picture reordering
  b.put(1, 1);             // vui_parameters_present_flag
  b.put(1, 0); b.put(1, 0);        // aspect_ratio_info_present_flag, overscan_info_present_flag
  b.put(1, 1); b.put(3, 5); b.put(1, 0); b.put(1, 1);   // video_signal_type: format 5, limited range, colour description
  b.put(8, 1); b.put(8, 1); b.put(8, 1);               // primaries / transfer / matrix = BT.709
  b.put(1, 1); b.ue(1); b.ue(1);   // chroma_loc_info: type 1 (centre) for both fields
  b.put(1, 0); b.put(1, 0); b.put(1, 0); b.put(1, 0);   // timing_info, nal_hrd, vcl_hrd, pic_struct
  b.put(1, 1);             // bitstream_restriction_flag
  b.put(1, 1);             // motion_vectors_over_pic_boundaries_flag
  b.ue(0); b.ue(0);        // max_bytes_per_pic_denom, max_bits_per_mb_denom
  b.ue(10); b.ue(10);      // log2_max_mv_length_horizontal / vertical
  b.ue(0);                 // max_num_reorder_frames
  b.ue(1);                 // max_dec_frame_buffering
  b.trailing();
  append_nal(out, 3, 7, b.buf);
  HostBits p;
  p.ue(0); p.ue(0);
  p.put(1, 0);             // entropy_coding_mode_flag (CAVLC)
  p.put(1, 0);             // bottom_field_pic_order_in_frame_present_flag
  p.ue(0);                 // num_slice_groups_minus1
  p.ue(0); p.ue(0);        // num_ref_idx_l0/l1_default_active_minus1
  p.put(1, 0); p.put(2, 0);
  p.se(0); p.se(0); p.se(0);
  p.put(1, 1);             // deblocking_filter_control_present_flag
  p.put(1, 0);             // constrained_intra_pred_flag
  p.put(1, 0);             // redundant_pic_cnt_present_flag
  p.trailing();
  append_nal(out, 3, 8, p.buf);
  return out;
}

}  // namespace

#define ECK(call)                                                                                        \
  do { cudaError_t e_ = (call);                                                                          \
       if (e_ != cudaSuccess) { snprintf(g_enc_err, sizeof g_enc_err, "%s -> %s", #call, cudaGetErrorString(e_)); encoder_destroy(e); return -2; } \
  } while (0)

int encoder_create(const EncoderConfig* cfg_in, Encoder** out) {
  if (!cfg_in || !out || (cfg_in->coded_w & 15) || (cfg_in->coded_h & 15)) {
    snprintf(g_enc_err, sizeof g_enc_err, "bad encoder config");
    return -1;
  }
  Encoder* e = new Encoder();
  e->cfg = *cfg_in;
  e->mbw = cfg_in->coded_w / 16; e->mbh = cfg_in->coded_h / 16;
  // slice_rows <= 0: the default rule (oracle/h264_ref.c b2v_ref_enc_create): P pictures in slices of 8 macroblock rows, one slice per
  // band in striped mode — inside a slice the row above predicts the motion vector and P_Skip infers a moving one, which halves the
  // bytes of a scrolling picture against one row per slice.  IDR pictures are sliced on their own (seg_cols below).
  if (e->cfg.slice_rows <= 0) {
    const bool striped = e->cfg.stripe_rows > 0 && e->cfg.stripe_rows < e->mbh;
    e->cfg.slice_rows = striped ? e->cfg.stripe_rows : (e->mbh < 8 ? e->mbh : 8);
  }
  const EncoderConfig* cfg = &e->cfg;
  e->n_slices = (e->mbh + cfg->slice_rows - 1) / cfg->slice_rows;
  const size_t mbs = (size_t)e->mbw * e->mbh, fb = (size_t)cfg->coded_w * cfg->coded_h * 3 / 2;
  ECK(cudaMalloc((void**)&e->recon[0], fb));
  ECK(cudaMalloc((void**)&e->recon[1], fb));
  ECK(cudaMemset(e->recon[0], 0, fb));
  ECK(cudaMemset(e->recon[1], 0, fb));
  for (int b = 0; b < 2; b++) {
    ECK(cudaMalloc((void**)&e->mbinfo[b], mbs * sizeof(MbInfo)));
    ECK(cudaMemset(e->mbinfo[b], 0, mbs * sizeof(MbInfo)));
    ECK(cudaMalloc((void**)&e->i4modes[b], mbs * 16));
    ECK(cudaMemset(e->i4modes[b], 2, mbs * 16));
    ECK(cudaMalloc((void**)&e->coef[b], mbs * COEF_BLOCKS * 16 * sizeof(int16_t)));
    ECK(cudaMemset(e->coef[b], 0, mbs * COEF_BLOCKS * 16 * sizeof(int16_t)));
    ECK(cudaMalloc((void**)&e->nnz[b], mbs * 32));
    ECK(cudaMemset(e->nnz[b], 0, mbs * 32));
  }
  ECK(cudaMalloc((void**)&e->me_pub, mbs * sizeof(unsigned long long)));
  ECK(cudaMemset(e->me_pub, 0, mbs * sizeof(unsigned long long)));
  ECK(cudaMalloc((void**)&e->mb_words, mbs * MB_WORDS * sizeof(uint32_t)));
  ECK(cudaMalloc((void**)&e->mb_nbits, mbs * sizeof(uint32_t)));
  e->slice_words = cfg->slice_rows * e->mbw * MB_WORDS + 64;
  // IDR pictures: slices shorter than a row (same rule as oracle/h264_ref.c auto_seg_cols: about 540 slices, none under 30 macroblocks)
  // (idr_slice_mbs < 0: IDR pictures in slices of slice_rows whole rows, like P pictures — rows of a slice then wait on the row above)
  if (cfg->idr_slice_mbs >= 0) {
    int cols = cfg->idr_slice_mbs;
    if (cols == 0) { int segs = 540 / e->mbh; const int cap = e->mbw / 30; if (segs > cap) segs = cap; cols = segs <= 1 ? e->mbw : (e->mbw + segs - 1) / segs; }
    if (cols >= e->mbw) cols = e->mbw;          // one slice per macroblock row
    e->seg_cols = cols;
  }
  if (e->seg_cols) { e->n_seg_slices = e->mbh * ((e->mbw + e->seg_cols - 1) / e->seg_cols); e->seg_slice_words = e->seg_cols * MB_WORDS + 64; }
  const size_t nsl_max = (size_t)(e->n_seg_slices > e->n_slices ? e->n_seg_slices : e->n_slices);
  size_t sb_words = (size_t)e->n_slices * e->slice_words;
  if ((size_t)e->n_seg_slices * e->seg_slice_words > sb_words) sb_words = (size_t)e->n_seg_slices * e->seg_slice_words;
  ECK(cudaMalloc((void**)&e->slice_buf, sb_words * sizeof(uint32_t)));
  ECK(cudaMemset(e->slice_buf, 0, sb_words * sizeof(uint32_t)));
  ECK(cudaMalloc((void**)&e->slice_size, nsl_max * sizeof(uint32_t)));
  ECK(cudaMalloc((void**)&e->slice_rbsp, nsl_max * sizeof(uint32_t)));
  ECK(cudaMalloc((void**)&e->slice_bits, nsl_max * sizeof(long long)));
  {   // k_slice_build's look-back records: one per chunk of up to 256 macroblocks (32 bytes cover either record type)
    const size_t cps_row = ((size_t)cfg->slice_rows * e->mbw + 255) / 256, cps_seg = e->seg_cols ? ((size_t)e->seg_cols + 255) / 256 : 0;
    const size_t chunks = std::max((size_t)e->n_slices * cps_row, (size_t)e->n_seg_slices * cps_seg) + 1;
    ECK(cudaMalloc((void**)&e->chunk_agg, chunks * 32)); ECK(cudaMemset(e->chunk_agg, 0, chunks * 32));
    ECK(cudaMalloc((void**)&e->chunk_inc, chunks * 32)); ECK(cudaMemset(e->chunk_inc, 0, chunks * 32));
    ECK(cudaMalloc((void**)&e->slice_done, nsl_max * sizeof(int))); ECK(cudaMemset(e->slice_done, 0, nsl_max * sizeof(int)));
  }
  ECK(cudaMalloc((void**)&e->progress, e->mbh * sizeof(int)));
  ECK(cudaMalloc((void**)&e->overflow, sizeof(int)));
  ECK(cudaMemset(e->overflow, 0, sizeof(int)));
  ECK(cudaMalloc((void**)&e->rc, sizeof(RcState)));
  RcState rc0{}; rc0.fb[0].qp = rc0.fb[1].qp = -1;
  ECK(cudaMemcpy(e->rc, &rc0, sizeof rc0, cudaMemcpyHostToDevice));
  // bands: full-frame coding is one band of mbh rows; striped mode gives every band its own SPS (height = the band's)
  const int crop_b = (cfg->coded_h - cfg->height) / 2;
  e->striped = cfg->stripe_rows > 0 && cfg->stripe_rows < e->mbh;
  if (e->striped && cfg->stripe_rows % cfg->slice_rows) { snprintf(g_enc_err, sizeof g_enc_err, "stripe_rows must be a multiple of slice_rows"); encoder_destroy(e); return -1; }
  e->band_rows = e->striped ? cfg->stripe_rows : e->mbh;
  e->n_bands = (e->mbh + e->band_rows - 1) / e->band_rows;
  std::vector<uint8_t> ps = make_param_sets(*cfg, e->mbw, e->band_rows, e->striped ? 0 : crop_b);
  e->param_len = (int)ps.size();
  if (e->striped) {
    std::vector<uint8_t> last = make_param_sets(*cfg, e->mbw, e->mbh - (e->n_bands - 1) * e->band_rows, crop_b);
    e->param_len_last = (int)last.size();
    ps.insert(ps.end(), last.begin(), last.end());
    e->au_data_off = au_data_offset(e->n_bands);
  }
  ECK(cudaMalloc((void**)&e->param_sets, ps.size()));
  ECK(cudaMemcpy(e->param_sets, ps.data(), ps.size(), cudaMemcpyHostToDevice));
  ECK(cudaMalloc((void**)&e->band_fn, e->n_bands * sizeof(int)));
  ECK(cudaMemset(e->band_fn, 0, e->n_bands * sizeof(int)));
  ECK(cudaMalloc((void**)&e->band_coded, e->n_bands * sizeof(int)));
  ECK(cudaMemset(e->band_coded, 0, e->n_bands * sizeof(int)));
  for (int b = 0; b < 2; b++) {
    ECK(cudaEventCreateWithFlags(&e->ev_analysed[b], cudaEventDisableTiming));
    ECK(cudaEventCreateWithFlags(&e->ev_packed[b], cudaEventDisableTiming));
  }
  e->au_cap = (size_t)e->au_data_off + (size_t)e->n_bands * (e->param_len + e->param_len_last) + nsl_max * 16 + mbs * (MB_WORDS * 4 + 8) + 1024;
  *out = e;
  return 0;
}

void encoder_destroy(Encoder* e) {
  if (!e) return;
  void* ptrs[] = {e->recon[0], e->recon[1], e->mbinfo[0], e->mbinfo[1], e->coef[0], e->coef[1], e->nnz[0], e->nnz[1], e->mb_words, e->mb_nbits, e->slice_buf,
                  e->slice_size, e->slice_rbsp, e->slice_bits, e->progress, e->overflow, e->rc, e->param_sets, e->i4modes[0],
                  e->i4modes[1], e->band_fn, e->band_coded, e->me_pub, e->chunk_agg, e->chunk_inc, e->slice_done};
  for (void* p : ptrs) if (p) cudaFree(p);
  for (int b = 0; b < 2; b++) {
    if (e->ev_analysed[b]) cudaEventDestroy(e->ev_analysed[b]);
    if (e->ev_packed[b]) cudaEventDestroy(e->ev_packed[b]);
  }
  delete e;
}

size_t encoder_au_capacity(const Encoder* e) { return e->au_cap; }
int encoder_au_data_offset(const Encoder* e) { return e->au_data_off; }
int encoder_band_count(const Encoder* e) { return e->striped ? e->n_bands : 0; }
const uint8_t* encoder_recon(const Encoder* e) { return e->recon[e->cur]; }

int encoder_encode(Encoder* e, const EncodeFrameParams* p, cudaStream_t st) {
  const bool idr = p->idr || !e->have_ref;
  e->cur ^= 1;
  const int par = (int)(e->pic & 1);          // parity of this picture: feedback record, side-data buffers, events
  if (idr) e->frame_num = 0;
  FrameCtx f{};
  f.cw = e->cfg.coded_w; f.ch = e->cfg.coded_h; f.mbw = e->mbw; f.mbh = e->mbh;
  const bool seg = idr && e->seg_cols > 0;
  f.slice_rows = e->cfg.slice_rows; f.n_slices = seg ? e->n_seg_slices : e->n_slices; f.seg_cols = seg ? e->seg_cols : 0;
  f.idr = idr; f.rc_mode = p->rc_mode; f.qp_fixed = p->qp_fixed; f.target_bits = p->target_bits;
  f.frame_num = e->frame_num; f.idr_pic_id = e->idr_count; f.pic = (int)(e->pic & 0x7fffffff);
  f.cur = p->cur; f.ref = e->recon[e->cur ^ 1]; f.recon = e->recon[e->cur];
  f.mbinfo = e->mbinfo[par]; f.mbinfo_prev = e->mbinfo[par ^ 1]; f.i4modes = e->i4modes[par]; f.coef = e->coef[par]; f.nnz = e->nnz[par];
  f.me_pub = e->me_pub;
  f.chunk_agg = (ChunkAgg*)e->chunk_agg; f.chunk_inc = (ChunkInc*)e->chunk_inc; f.slice_done = e->slice_done; f.chunks_per_slice = 1;
  {   // anchors: ceil(mbw/4) columns x (groups of 4 rows inside every band)
    const int rows_last = e->mbh - (e->n_bands - 1) * e->band_rows;
    f.n_anchor = ((e->mbw + 3) / 4) * ((e->n_bands - 1) * ((e->band_rows + 3) / 4) + (rows_last + 3) / 4);
  }
  f.mb_words = e->mb_words; f.mb_nbits = e->mb_nbits;
  f.slice_buf = e->slice_buf; f.slice_words = seg ? e->seg_slice_words : e->slice_words; f.slice_size = e->slice_size; f.slice_rbsp = e->slice_rbsp;
  f.slice_bits = e->slice_bits; f.paint_trigger = p->paint_trigger; f.paint_qp = p->paint_qp; f.paint_burst = p->paint_burst; f.progress = e->progress; f.rc = e->rc;
  f.band_rows = e->band_rows; f.n_bands = e->n_bands; f.striped = e->striped; f.param_len_last = e->param_len_last;
  f.band_fn = e->band_fn; f.band_coded = e->band_coded; f.au_data_off = e->au_data_off;
  f.param_sets = e->param_sets; f.param_len = e->param_len; f.csc_ts = p->csc_ts; f.au = p->au; f.overflow = e->overflow;
  int n = 0;
  // Two-stream schedule (no per-stage events requested): ANALYSIS of picture k on `st` (CSC before it, by the caller), ENTROPY
  // coding of picture k (CAVLC, slice scan + rate-control step, copy, emulation-prevention count, pack) on `st_pack`, overlapping
  // the analysis of picture k+1.  What makes that legal:
  //  * the side data the two halves share (MbInfo, levels, nnz, Intra4x4 modes) is double-buffered by picture parity;
  //  * the rate controller feeds back two pictures late: picture k reads the record left by picture k-2 (RcFb), which the scan
  //    of picture k-1 — possibly still running — never touches;
  //  * the analysis of picture k waits for the pack of picture k-2: that releases this parity's side data, the reconstruction
  //    buffer it is about to overwrite (the pack's copy kernel reads I_PCM samples from it) and the record of k-2.
  const bool overlap = p->st_pack != nullptr && p->ev == nullptr;
  if (overlap) cudaStreamWaitEvent(st, e->ev_packed[par], 0);           // pack of picture k-2 (no-op before the first two)
  n += idr ? launch_intra(f, st) : launch_inter(f, st);
  if (p->ev) cudaEventRecord(p->ev[2], st);
  cudaStream_t sp = st;
  if (overlap) {
    sp = p->st_pack;
    cudaEventRecord(e->ev_analysed[par], st);
    cudaStreamWaitEvent(sp, e->ev_analysed[par], 0);
  }
  n += launch_cavlc(f, sp);
  if (p->ev) cudaEventRecord(p->ev[3], st);
  n += launch_slice_build(f, sp);
  if (p->ev) cudaEventRecord(p->ev[4], st);
  n += launch_pack_cap(f, (long long)e->au_cap, sp);
  if (p->ev) cudaEventRecord(p->ev[5], st);
  if (overlap) cudaEventRecord(e->ev_packed[par], sp);
  if (idr) e->idr_count++;
  e->frame_num = (e->frame_num + 1) & 255;
  e->have_ref = true;
  e->pic++;
  return n;
}

}  // namespace b2v
