// h264_encoder.h — interface between the session layer (b2v_api.cu) and the H.264 Baseline
// encoder kernels (h264_*.cu).  B200 carries no NVENC block, so stage (c) of the hot path is a
// software encoder made of CUDA kernels: one warp per macroblock.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace b2v {

struct Encoder;

struct EncoderConfig {
  int width, height;       // visible size (SPS cropping)
  int coded_w, coded_h;    // multiples of 16
  int slice_rows;          // macroblock rows per slice
  int stripe_rows;         // macroblock rows per band (multiple of slice_rows); 0 = full-frame
  int idr_slice_mbs;       // IDR pictures: macroblocks per slice inside a row (needs slice_rows == 1); 0 = default rule, < 0 = whole rows
};

struct EncodeFrameParams {
  const uint8_t* cur;      // NV12, coded size, device
  uint8_t* au;             // device buffer, encoder_au_capacity() bytes; AuHeader first
  int idr;
  int rc_mode;             // B2V_RC_CBR | B2V_RC_CQP
  int qp_fixed;
  int paint_trigger, paint_qp, paint_burst;   // paint-over: `paint_burst` pictures at paint_qp after `paint_trigger` all-skipped pictures (0 = off)
  int64_t target_bits;     // per frame, CBR
  cudaEvent_t* ev;         // null, or 6 timing events: encoder records ev[2..5] after each stage (forces the serial schedule)
  cudaStream_t st_pack;    // null = everything on `st`; else the entropy coding of this picture (k_cavlc_mb ... k_pack_au) runs here,
                           // overlapping the analysis of the next picture on `st`.  The access unit is complete on st_pack.
  const unsigned long long* csc_ts;   // null, or the CSC launch's device stamps to forward in the AuHeader
};

int  encoder_create(const EncoderConfig* cfg, Encoder** out);
void encoder_destroy(Encoder* e);
size_t encoder_au_capacity(const Encoder* e);
int  encoder_au_data_offset(const Encoder* e);   // AuHeader + band table (+ slack for an in-place stripe header)
int  encoder_band_count(const Encoder* e);       // 0 when full-frame
// enqueue one frame on `st` (and `p->st_pack`); returns the number of kernel launches issued
int  encoder_encode(Encoder* e, const EncodeFrameParams* p, cudaStream_t st);
const uint8_t* encoder_recon(const Encoder* e);   // NV12 reconstruction of the last encoded frame
const char* encoder_last_error();

}  // namespace b2v
