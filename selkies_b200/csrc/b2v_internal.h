// b2v_internal.h — shared declarations between the C-ABI (b2v_api.cu) and the kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace b2v {

// ---- colour conversion spec (DESIGN.md §3; BT.709 limited range, 14-bit coefficients) ----
constexpr int KYR = 2991, KYG = 10064, KYB = 1016;
constexpr int KUR = -1649, KUG = -5547, KUB = 7196;
constexpr int KVR = 7196, KVG = -6536, KVB = -660;

// per-destination-index bilinear tap: i0 | (i1-i0)<<15 in .x low 16 / bit 15.., weight in .y
struct Tap { int32_t i0; int32_t i1; int32_t f; int32_t pad; };

struct CscParams {
  const uint8_t* src;   // BGRA, device
  int src_w, src_h, src_stride;
  int dst_w, dst_h;     // visible (scaled) size
  int coded_w, coded_h; // output plane size (multiples of 16 for the encoder; == dst for csc-only)
  uint8_t* out_y;       // coded_h rows, pitch coded_w
  uint8_t* out_uv;      // coded_h/2 rows, pitch coded_w
  const Tap* tx;        // dst_w taps (null when 1:1)
  const Tap* ty;        // dst_h taps
  unsigned long long* ts; // null, or {min block-start, max block-end} %globaltimer stamps of this launch (B2V_FLAG_TIMING)
  int matrix;             // 0 = BT.709 limited range (H.264 path), 1 = JFIF full-range BT.601 (JPEG stripe path)
};

// ---- access-unit container: what the H.264 and JPEG pack kernels write into the output buffer, and the host reads ----
// 64-byte record the pack kernel writes in front of the access unit in HBM; travels to the host
// with the first D2H chunk.
struct AuHeader {
  int32_t size;            // bytes of data following this header (Annex-B NALs, or JFIF stripes back to back)
  int32_t qp;              // slice QP used
  int32_t is_idr;
  int32_t n_slices;
  int64_t total_bits;      // before emulation prevention
  int32_t next_qp;         // rate controller output for the next frame
  int32_t overflow;        // non-zero if a macroblock exceeded its scratch budget (must never happen)
  uint64_t csc_t0, csc_t1;  // %globaltimer stamps of the CSC launch of this picture (0 when timing is off)
  int32_t pad[4];
};
static_assert(sizeof(AuHeader) == 64, "AuHeader must be 64 bytes");

// striped H.264 and JPEG: one record per band (stripe) right after the AuHeader (offsets relative to the first data byte)
struct BandEntry { int32_t off, size, coded, frame_num; };

// bytes from the AuHeader to the first data byte when a table of n_bands records follows it (+ slack for an in-place stripe header)
constexpr int au_data_offset(int n_bands) { return (int)sizeof(AuHeader) + ((n_bands * (int)sizeof(BandEntry) + 16 + 63) & ~63); }

// returns number of kernel launches issued (1)
int launch_csc(const CscParams& p, cudaStream_t st);
void make_taps_host(Tap* t, int dn, int sn);

}  // namespace b2v
