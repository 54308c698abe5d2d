// jpeg.cu — JPEG stripe encoder (CaptureSettings.output_mode = 0, the reference's "jpeg" encoder: selkies.py:3209-3212).
//
// The picture is cut into horizontal stripes of `stripe_rows` MCU rows (16 luma rows each); every stripe that changed since the
// previous picture is delivered as one complete baseline JFIF file (4:2:0, Annex K tables, IJG quality scaling), which is what the
// reference's client hands to ImageDecoder per stripe (addons/selkies-web-core/selkies-ws-core.js:3166-3182, 2374-2393).  A stripe
// that stayed unchanged for `paint_trigger` pictures is sent once more at the paint-over quality (CaptureSettings.
// paint_over_jpeg_quality / use_paint_over_quality / paint_over_trigger_frames).
//
// JPEG's entropy coding is serial in the bitstream, but — as with CAVLC — nothing a block writes depends on its neighbours'
// BITS, only on the previous block's DC level.  So:
//   k_jpeg_diff   one block per stripe: did any byte of the stripe change? -> quality of the stripe and whether it is delivered
//   k_jpeg_dct    one THREAD per 8x8 block: level shift, accurate integer LL&M forward DCT, quantisation, levels in scan order
//   k_jpeg_size   one thread per block: DC difference against the previous block of its component, exact Huffman size
//   k_jpeg_scan   one block per stripe: prefix sum -> bit offset of every block, stripe size
//   k_jpeg_write  one thread per block: Huffman codes shifted into the stripe's bit string (atomicOr)
//   k_jpeg_ff     one block per stripe: pad the last byte with 1-bits, count the FF bytes -> size of the stripe's file
//   k_jpeg_pack   one block per stripe: JFIF header, FF byte stuffing, EOI, stripe table
// The bit sinks, the stuffing rule (JpegEscape) and its count and copy are shared with the H.264 back end (bitstream.cuh).
// CPU restatement (byte-identical to libjpeg-turbo in its single-component mode): oracle/jpeg_ref.c.
#include <cstdio>
#include <cstring>
#include <vector>

#include "b2v_internal.h"     // AuHeader, BandEntry: the JPEG mode uses the access-unit container of the striped H.264 mode
#include "bitstream.cuh"
#include "jpeg.h"

namespace b2v {

namespace {

// scan position -> natural index; constexpr so that the unrolled quantiser indexes its register array with literals
__host__ __device__ constexpr int jzz(int k) {
  constexpr int t[64] = {0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
                         35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
  return t[k];
}
// Huffman tables, built on the host from Annex K (code | size << 16), index = [dc luma, dc chroma][category] / [ac luma, ac chroma][run << 4 | size]
__constant__ uint32_t c_dc[2][12];
__constant__ uint32_t c_ac[2][256];

const uint8_t h_std_luma_q[64] = {
  16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56, 14, 17, 22, 29, 51, 87, 80, 62,
  18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92, 49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};
const uint8_t h_std_chroma_q[64] = {
  17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99, 99, 99, 99, 99,
  99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99};
const uint8_t h_zigzag[64] = {
  0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21, 28,
  35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
const uint8_t h_dc_luma_bits[16] = {0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0};
const uint8_t h_dc_chroma_bits[16] = {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0};
const uint8_t h_dc_vals[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
const uint8_t h_ac_luma_bits[16] = {0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d};
const uint8_t h_ac_luma_vals[162] = {
  0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71, 0x14, 0x32, 0x81, 0x91, 0xa1, 0x08,
  0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72, 0x82, 0x09, 0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26, 0x27, 0x28,
  0x29, 0x2a, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59,
  0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89,
  0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6,
  0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2,
  0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};
const uint8_t h_ac_chroma_bits[16] = {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77};
const uint8_t h_ac_chroma_vals[162] = {
  0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22, 0x32, 0x81, 0x08, 0x14, 0x42, 0x91,
  0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1, 0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26,
  0x27, 0x28, 0x29, 0x2a, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58,
  0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x82, 0x83, 0x84, 0x85, 0x86, 0x87,
  0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4,
  0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda,
  0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};

void build_huff(uint32_t* out, int n_out, const uint8_t bits[16], const uint8_t* vals) {   // T.81 Annex C
  for (int i = 0; i < n_out; i++) out[i] = 0;
  int code = 0, k = 0;
  for (int len = 1; len <= 16; len++) {
    for (int i = 0; i < bits[len - 1]; i++, k++) out[vals[k]] = (uint32_t)code++ | ((uint32_t)len << 16);
    code <<= 1;
  }
}
void qtable(int quality, bool chroma, uint8_t out[64]) {          // IJG quality rule, natural order
  quality = quality < 1 ? 1 : quality > 100 ? 100 : quality;
  const int scale = quality < 50 ? 5000 / quality : 200 - 2 * quality;
  const uint8_t* base = chroma ? h_std_chroma_q : h_std_luma_q;
  for (int i = 0; i < 64; i++) { int v = (base[i] * scale + 50) / 100; out[i] = (uint8_t)(v < 1 ? 1 : v > 255 ? 255 : v); }
}
size_t put_marker(uint8_t* o, int m, int len) { o[0] = 0xFF; o[1] = (uint8_t)m; o[2] = (uint8_t)(len >> 8); o[3] = (uint8_t)len; return 4; }
size_t put_dht(uint8_t* o, int tc_th, const uint8_t bits[16], const uint8_t* vals, int nvals) {
  size_t n = put_marker(o, 0xC4, 2 + 1 + 16 + nvals);
  o[n++] = (uint8_t)tc_th; memcpy(o + n, bits, 16); n += 16; memcpy(o + n, vals, nvals); n += nvals;
  return n;
}
// JFIF header of a w x h 4:2:0 image; *h_off = offset of the 16-bit height inside it (patched per stripe on the device)
size_t make_header(uint8_t* o, int w, int h, int quality, int* h_off) {
  size_t n = 0;
  uint8_t q[64];
  o[n++] = 0xFF; o[n++] = 0xD8;
  n += put_marker(o + n, 0xE0, 16); memcpy(o + n, "JFIF\0\1\1\0\0\1\0\1\0\0", 14); n += 14;
  for (int t = 0; t < 2; t++) {
    qtable(quality, t == 1, q);
    n += put_marker(o + n, 0xDB, 67); o[n++] = (uint8_t)t;
    for (int k = 0; k < 64; k++) o[n++] = q[h_zigzag[k]];
  }
  n += put_marker(o + n, 0xC0, 8 + 9);
  o[n++] = 8; *h_off = (int)n; o[n++] = (uint8_t)(h >> 8); o[n++] = (uint8_t)h; o[n++] = (uint8_t)(w >> 8); o[n++] = (uint8_t)w; o[n++] = 3;
  for (int c = 0; c < 3; c++) { o[n++] = (uint8_t)(c + 1); o[n++] = (uint8_t)(c == 0 ? 0x22 : 0x11); o[n++] = (uint8_t)(c ? 1 : 0); }
  n += put_dht(o + n, 0x00, h_dc_luma_bits, h_dc_vals, 12);
  n += put_dht(o + n, 0x10, h_ac_luma_bits, h_ac_luma_vals, 162);
  n += put_dht(o + n, 0x01, h_dc_chroma_bits, h_dc_vals, 12);
  n += put_dht(o + n, 0x11, h_ac_chroma_bits, h_ac_chroma_vals, 162);
  n += put_marker(o + n, 0xDA, 12);
  o[n++] = 3; o[n++] = 1; o[n++] = 0x00; o[n++] = 2; o[n++] = 0x11; o[n++] = 3; o[n++] = 0x11;
  o[n++] = 0; o[n++] = 63; o[n++] = 0;
  return n;
}

constexpr int JPEG_BLOCK_WORDS = 80;           // per-8x8-block share of the stripe bit string: 2560 bits (worst case 63 x 26 + 20 < 1700)
constexpr int JT = STUFF_THREADS;

struct JpegCtx {
  int cw, ch, w, h;                 // coded (multiple of 16) and visible size
  int mcu_w, mcu_h, stripe_rows, n_stripes;
  const uint8_t* cur;               // NV12, JFIF matrix, coded size
  uint8_t* prev;                    // previous picture (change detection); updated by k_jpeg_diff
  int16_t* lev;                     // [blocks][64] scan order
  uint32_t* bits;                   // [blocks] Huffman size of the block
  long long* off;                   // [blocks] bit offset inside the stripe's scan
  uint32_t* sbuf;                   // [n_stripes][stripe_words]
  long long stripe_words;
  long long* sbits;                 // [n_stripes]
  int* s_static;                    // [n_stripes] consecutive unchanged pictures
  int* s_flags;                     // [n_stripes] bit 0: deliver, bit 1: paint-over quality
  uint32_t* ssize;                  // [n_stripes] bytes of the stripe's file (0 = not delivered)
  const uint16_t* qt;               // [2 qualities][2 tables][64] quantiser << 3, natural order
  const uint8_t* hdr;               // [2 qualities][hdr_len]
  int hdr_len, hdr_h_off;
  int first, paint_trigger;
  uint8_t* au; long long au_cap; int au_data_off;
};

__device__ __forceinline__ int stripe_of_mcu_row(const JpegCtx& c, int my) { return my / c.stripe_rows; }

// ---- change detection: block per stripe ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(JT) k_jpeg_diff(JpegCtx c) {
  const int s = blockIdx.x, tid = threadIdx.x;
  const int r0 = s * c.stripe_rows * 16, r1 = min(c.ch, r0 + c.stripe_rows * 16);
  const size_t ysz = (size_t)c.cw * c.ch;
  int changed = 0;
  // luma rows r0..r1, chroma rows r0/2..r1/2: compare and refresh the copy, 16 bytes per step
  const uint4* cy = reinterpret_cast<const uint4*>(c.cur + (size_t)r0 * c.cw); uint4* py = reinterpret_cast<uint4*>(c.prev + (size_t)r0 * c.cw);
  const size_t ny = (size_t)(r1 - r0) * c.cw / 16;
  for (size_t i = tid; i < ny; i += JT) { const uint4 a = cy[i], b = py[i]; if (a.x != b.x || a.y != b.y || a.z != b.z || a.w != b.w) { changed = 1; py[i] = a; } }
  const uint4* cu = reinterpret_cast<const uint4*>(c.cur + ysz + (size_t)(r0 / 2) * c.cw); uint4* pu = reinterpret_cast<uint4*>(c.prev + ysz + (size_t)(r0 / 2) * c.cw);
  const size_t nu = (size_t)((r1 - r0) / 2) * c.cw / 16;
  for (size_t i = tid; i < nu; i += JT) { const uint4 a = cu[i], b = pu[i]; if (a.x != b.x || a.y != b.y || a.z != b.z || a.w != b.w) { changed = 1; pu[i] = a; } }
  changed = __syncthreads_or(changed);
  if (tid == 0) {
    int st = c.s_static[s], fl;
    if (c.first || changed) { st = 0; fl = 1; }
    else { st = min(st + 1, 1 << 20); fl = (c.paint_trigger > 0 && st == c.paint_trigger) ? 3 : 0; }     // static long enough: once more, finer
    c.s_static[s] = st; c.s_flags[s] = fl;
  }
}

#define JDS(x, n) (((x) + (1 << ((n) - 1))) >> (n))
// accurate integer LL&M forward DCT, one 1-D pass over 8 values with stride st (oracle/jpeg_ref.c b2v_ref_jpeg_fdct)
template <int PASS>
__device__ __forceinline__ void fdct8(int* p, int st) {
  int t0 = p[0] + p[7 * st], t7 = p[0] - p[7 * st], t1 = p[st] + p[6 * st], t6 = p[st] - p[6 * st];
  int t2 = p[2 * st] + p[5 * st], t5 = p[2 * st] - p[5 * st], t3 = p[3 * st] + p[4 * st], t4 = p[3 * st] - p[4 * st];
  const int t10 = t0 + t3, t13 = t0 - t3, t11 = t1 + t2, t12 = t1 - t2;
  if (PASS == 0) { p[0] = (t10 + t11) << 2; p[4 * st] = (t10 - t11) << 2; }
  else { p[0] = JDS(t10 + t11, 2); p[4 * st] = JDS(t10 - t11, 2); }
  constexpr int sh = PASS == 0 ? 11 : 15;
  int z1 = (t12 + t13) * 4433;
  p[2 * st] = JDS(z1 + t13 * 6270, sh);
  p[6 * st] = JDS(z1 - t12 * 15137, sh);
  z1 = t4 + t7; int z2 = t5 + t6, z3 = t4 + t6, z4 = t5 + t7; const int z5 = (z3 + z4) * 9633;
  t4 *= 2446; t5 *= 16819; t6 *= 25172; t7 *= 12299;
  z1 *= -7373; z2 *= -20995; z3 *= -16069; z4 *= -3196;
  z3 += z5; z4 += z5;
  p[7 * st] = JDS(t4 + z1 + z3, sh); p[5 * st] = JDS(t5 + z2 + z4, sh);
  p[3 * st] = JDS(t6 + z2 + z3, sh); p[st] = JDS(t7 + z1 + z4, sh);
}

// block index -> (mcu x, mcu y, k): blocks are numbered in scan order, 6 per MCU (4 Y, Cb, Cr), MCUs in raster order
__device__ __forceinline__ void block_pos(const JpegCtx& c, int b, int& mx, int& my, int& k) { const int m = b / 6; k = b - 6 * m; my = m / c.mcu_w; mx = m - my * c.mcu_w; }

__global__ void __launch_bounds__(128) k_jpeg_dct(JpegCtx c) {
  const int b = blockIdx.x * 128 + threadIdx.x;
  if (b >= c.mcu_w * c.mcu_h * 6) return;
  int mx, my, k;
  block_pos(c, b, mx, my, k);
  const int fl = c.s_flags[stripe_of_mcu_row(c, my)];
  if (!(fl & 1)) return;                                       // stripe not delivered: nothing to do
  int d[64];
  if (k < 4) {
    const uint8_t* p = c.cur + (size_t)(my * 16 + (k >> 1) * 8) * c.cw + mx * 16 + (k & 1) * 8;
#pragma unroll
    for (int y = 0; y < 8; y++) {
      const uint2 v = *reinterpret_cast<const uint2*>(p + (size_t)y * c.cw);
#pragma unroll
      for (int x = 0; x < 4; x++) { d[8 * y + x] = (int)((v.x >> (8 * x)) & 255u) - 128; d[8 * y + 4 + x] = (int)((v.y >> (8 * x)) & 255u) - 128; }
    }
  } else {
    const uint8_t* p = c.cur + (size_t)c.cw * c.ch + (size_t)(my * 8) * c.cw + mx * 16;
    const int sh = (k - 4) * 8;
#pragma unroll
    for (int y = 0; y < 8; y++) {
      const uint4 v = *reinterpret_cast<const uint4*>(p + (size_t)y * c.cw);      // 8 interleaved (Cb,Cr) pairs
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int x = 0; x < 8; x++) d[8 * y + x] = (int)((w[x >> 1] >> (sh + 16 * (x & 1))) & 255u) - 128;
    }
  }
#pragma unroll
  for (int i = 0; i < 8; i++) fdct8<0>(d + 8 * i, 1);
#pragma unroll
  for (int i = 0; i < 8; i++) fdct8<1>(d + i, 8);
  const uint16_t* q = c.qt + ((fl >> 1) & 1) * 128 + (k >= 4 ? 64 : 0);
  int16_t* out = c.lev + (size_t)b * 64;
  // quantise (round half away from zero) into scan order; written as 8 x 16-byte stores
#pragma unroll
  for (int g = 0; g < 8; g++) {
    uint32_t pk[4];
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const int n = jzz(g * 8 + j), qv = q[n];
      int t = d[n];
      const int a = (abs(t) + (qv >> 1)) / qv;
      t = t < 0 ? -a : a;
      if (j & 1) pk[j >> 1] |= (uint32_t)t << 16; else pk[j >> 1] = (uint32_t)t & 0xffffu;
    }
    reinterpret_cast<uint4*>(out)[g] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
  }
}

// previous block of the same component inside the stripe (-1: none, predictor 0)
__device__ __forceinline__ int prev_block(const JpegCtx& c, int b, int mx, int my, int k) {
  if (k >= 1 && k <= 3) return b - 1;
  const bool first_mcu = mx == 0 && (my % c.stripe_rows) == 0;
  if (first_mcu) return -1;
  return b - 6 + (k == 0 ? 3 : 0);
}
__device__ __forceinline__ int bitlen_dev(int v) { return 32 - __clz(v); }

// the magnitude bits of a coefficient: the low nb bits of t (negative t: of t - 1); the Huffman codes fit their lengths already
template <class S>
__device__ __forceinline__ void code_block(S& s, const int16_t* lv, int pred_dc, int chroma) {
  int t = (int)lv[0] - pred_dc, t2 = t;
  if (t < 0) { t = -t; t2--; }
  int nb = bitlen_dev(t);
  uint32_t e = c_dc[chroma][nb];
  s.put((int)(e >> 16), e & 0xffffu);
  s.put(nb, (uint32_t)t2 & ((1u << nb) - 1u));
  int r = 0;
  for (int k = 1; k < 64; k++) {
    t = lv[k];
    if (t == 0) { r++; continue; }
    while (r > 15) { e = c_ac[chroma][0xF0]; s.put((int)(e >> 16), e & 0xffffu); r -= 16; }
    t2 = t;
    if (t < 0) { t = -t; t2--; }
    nb = bitlen_dev(t);
    e = c_ac[chroma][(r << 4) + nb];
    s.put((int)(e >> 16), e & 0xffffu);
    s.put(nb, (uint32_t)t2 & ((1u << nb) - 1u));
    r = 0;
  }
  if (r > 0) { e = c_ac[chroma][0]; s.put((int)(e >> 16), e & 0xffffu); }
}

template <bool WRITE>
__global__ void __launch_bounds__(128) k_jpeg_code(JpegCtx c) {
  const int b = blockIdx.x * 128 + threadIdx.x;
  if (b >= c.mcu_w * c.mcu_h * 6) return;
  int mx, my, k;
  block_pos(c, b, mx, my, k);
  const int s = stripe_of_mcu_row(c, my);
  if (!(c.s_flags[s] & 1)) { if (!WRITE) c.bits[b] = 0; return; }
  const int16_t* lv = c.lev + (size_t)b * 64;
  const int pb = prev_block(c, b, mx, my, k);
  const int pred = pb < 0 ? 0 : (int)c.lev[(size_t)pb * 64];
  if (WRITE) { GlobalSink w{c.sbuf + (size_t)s * c.stripe_words, c.off[b]}; code_block(w, lv, pred, k >= 4); }
  else { CountSink n; code_block(n, lv, pred, k >= 4); c.bits[b] = (uint32_t)n.n; }
}

// ---- scan: block per stripe, prefix sum of the block sizes ---------------------------------------------------------------------
__global__ void __launch_bounds__(JT) k_jpeg_scan(JpegCtx c) {
  __shared__ long long s_w[JT / 32];
  __shared__ long long s_carry;
  const int s = blockIdx.x, tid = threadIdx.x;
  const int my0 = s * c.stripe_rows, my1 = min(c.mcu_h, my0 + c.stripe_rows);
  const int b0 = my0 * c.mcu_w * 6, nb = (my1 - my0) * c.mcu_w * 6;
  if (tid == 0) s_carry = 0;
  __syncthreads();
  for (int base = 0; base < nb; base += JT) {
    const int i = base + tid;
    const long long off = block_scan<JT>(i < nb ? (long long)c.bits[b0 + i] : 0LL, s_w, s_carry);
    if (i < nb) c.off[b0 + i] = off;
  }
  if (tid == 0) c.sbits[s] = s_carry;
}

// ---- ff count: block per stripe.  Pads the last byte with 1-bits, counts the FF bytes (each gets a 00 stuffed behind it) and
// publishes the size of the stripe's file ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(JT) k_jpeg_ff(JpegCtx c) {
  __shared__ int s_w[JT / 32];
  const int s = blockIdx.x, tid = threadIdx.x;
  if (!(c.s_flags[s] & 1)) { if (tid == 0) c.ssize[s] = 0; return; }
  uint32_t* w = c.sbuf + (size_t)s * c.stripe_words;
  const long long bits = c.sbits[s], nbytes = (bits + 7) >> 3;
  if (tid == 0 && (bits & 7)) { const int padn = 8 - (int)(bits & 7); atomicOr(&w[bits >> 5], ((1u << padn) - 1u) << (32 - (int)(bits & 31) - padn)); __threadfence(); }
  __syncthreads();
  const int ff = count_escapes<JpegEscape>(w, nbytes, s_w);
  if (tid == 0) c.ssize[s] = (uint32_t)(c.hdr_len + nbytes + ff + 2);
}

// ---- pack: block per stripe.  header | stuffed scan bytes | EOI, stripes back to back; stripe table entry; AuHeader ------------------
__global__ void __launch_bounds__(JT) k_jpeg_pack(JpegCtx c) {
  __shared__ int s_w[JT / 32];
  __shared__ int s_carry;
  __shared__ long long s_part[JT / 32];
  __shared__ long long s_base;
  const int s = blockIdx.x, tid = threadIdx.x;
  const int fl = c.s_flags[s];
  uint8_t* au = c.au + c.au_data_off;
  const long long cap = c.au_cap - c.au_data_off;
  long long part = 0;                                      // byte offset of this stripe's file: the sizes of the stripes before it
  for (int j = tid; j < s; j += JT) part += c.ssize[j];
  part = block_sum<JT>(part, s_part);
  if (tid == 0) s_base = part;
  __syncthreads();
  const long long slot = s_base;
  BandEntry* be = reinterpret_cast<BandEntry*>(c.au + sizeof(AuHeader)) + s;
  uint32_t* w = c.sbuf + (size_t)s * c.stripe_words;
  if (s == c.n_stripes - 1 && tid == 0) {
    AuHeader* h = reinterpret_cast<AuHeader*>(c.au);
    const long long total = slot + c.ssize[s];
    h->size = (int32_t)(total < cap ? total : cap); h->qp = 0; h->is_idr = 1; h->n_slices = c.n_stripes; h->total_bits = total * 8; h->next_qp = 0;
    h->overflow = total > cap ? 2 : 0; h->csc_t0 = 0; h->csc_t1 = 0;
  }
  if (!(fl & 1)) {
    if (tid == 0) { be->off = (int32_t)slot; be->size = 0; be->coded = 0; be->frame_num = 0; }
    return;
  }
  const long long nbytes = (c.sbits[s] + 7) >> 3;
  const uint8_t* hdr = c.hdr + ((fl >> 1) & 1) * c.hdr_len;
  for (int i = tid; i < c.hdr_len; i += JT) if (slot + i < cap) au[slot + i] = hdr[i];
  __syncthreads();
  if (tid == 0 && slot + c.hdr_h_off + 1 < cap) {        // this stripe's visible height
    const int y0 = s * c.stripe_rows * 16, hh = min(c.h, y0 + c.stripe_rows * 16) - y0;
    au[slot + c.hdr_h_off] = (uint8_t)(hh >> 8); au[slot + c.hdr_h_off + 1] = (uint8_t)hh;
  }
  const long long out0 = slot + c.hdr_len;
  const int ff = stuff_copy<JpegEscape>(w, nbytes, au + out0, cap - out0, s_w, s_carry);
  clear_bits<JT>(w, nbytes, c.stripe_words);
  if (tid == 0) {
    const long long end = out0 + nbytes + ff;
    if (end + 2 <= cap) { au[end] = 0xFF; au[end + 1] = 0xD9; }
    be->off = (int32_t)slot; be->size = (int32_t)(end + 2 - slot); be->coded = 1; be->frame_num = (fl >> 1) & 1;
  }
}

}  // namespace

struct JpegEncoder {
  JpegConfig cfg{};
  int mcu_w = 0, mcu_h = 0, n_stripes = 0, stripe_rows = 0, hdr_len = 0, hdr_h_off = 0;
  long long stripe_words = 0;
  uint8_t *prev = nullptr, *hdr = nullptr;
  int16_t* lev = nullptr; uint32_t *bits = nullptr, *sbuf = nullptr; long long *off = nullptr, *sbits = nullptr;
  int *s_static = nullptr, *s_flags = nullptr;
  uint32_t* ssize = nullptr;
  uint16_t* qt = nullptr;
  size_t au_cap = 0; int au_data_off = 0;
  bool first = true;
};

static thread_local char g_jerr[256] = "";
const char* jpeg_last_error() { return g_jerr; }

#define JCK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { snprintf(g_jerr, sizeof g_jerr, "%s -> %s", #call, cudaGetErrorString(e_)); jpeg_destroy(e); return -2; } } while (0)

int jpeg_create(const JpegConfig* cfg, JpegEncoder** out) {
  if (!cfg || !out || (cfg->coded_w & 15) || (cfg->coded_h & 15)) { snprintf(g_jerr, sizeof g_jerr, "bad JPEG config"); return -1; }
  JpegEncoder* e = new JpegEncoder();
  e->cfg = *cfg;
  e->mcu_w = cfg->coded_w / 16; e->mcu_h = cfg->coded_h / 16;
  e->stripe_rows = cfg->stripe_rows > 0 && cfg->stripe_rows < e->mcu_h ? cfg->stripe_rows : e->mcu_h;
  e->n_stripes = (e->mcu_h + e->stripe_rows - 1) / e->stripe_rows;
  const size_t blocks = (size_t)e->mcu_w * e->mcu_h * 6, fb = (size_t)cfg->coded_w * cfg->coded_h * 3 / 2;
  e->stripe_words = (long long)e->stripe_rows * e->mcu_w * 6 * JPEG_BLOCK_WORDS + 64;
  // Huffman + quantiser tables, headers (two qualities: normal, paint-over)
  uint32_t dc[2][12], ac[2][256];
  build_huff(dc[0], 12, h_dc_luma_bits, h_dc_vals); build_huff(dc[1], 12, h_dc_chroma_bits, h_dc_vals);
  build_huff(ac[0], 256, h_ac_luma_bits, h_ac_luma_vals); build_huff(ac[1], 256, h_ac_chroma_bits, h_ac_chroma_vals);
  JCK(cudaMemcpyToSymbol(c_dc, dc, sizeof dc)); JCK(cudaMemcpyToSymbol(c_ac, ac, sizeof ac));
  uint16_t qt[2][2][64]; uint8_t q8[64];
  std::vector<uint8_t> hdr[2];
  for (int v = 0; v < 2; v++) {
    const int quality = v ? cfg->paint_quality : cfg->quality;
    for (int t = 0; t < 2; t++) { qtable(quality, t == 1, q8); for (int i = 0; i < 64; i++) qt[v][t][i] = (uint16_t)(q8[i] << 3); }
    hdr[v].resize(1024);
    hdr[v].resize(make_header(hdr[v].data(), cfg->width, e->stripe_rows * 16, quality, &e->hdr_h_off));
  }
  e->hdr_len = (int)hdr[0].size();
  JCK(cudaMalloc((void**)&e->qt, sizeof qt)); JCK(cudaMemcpy(e->qt, qt, sizeof qt, cudaMemcpyHostToDevice));
  JCK(cudaMalloc((void**)&e->hdr, 2 * e->hdr_len));
  JCK(cudaMemcpy(e->hdr, hdr[0].data(), e->hdr_len, cudaMemcpyHostToDevice)); JCK(cudaMemcpy(e->hdr + e->hdr_len, hdr[1].data(), e->hdr_len, cudaMemcpyHostToDevice));
  JCK(cudaMalloc((void**)&e->prev, fb)); JCK(cudaMemset(e->prev, 0, fb));
  JCK(cudaMalloc((void**)&e->lev, blocks * 64 * sizeof(int16_t)));
  JCK(cudaMalloc((void**)&e->bits, blocks * sizeof(uint32_t)));
  JCK(cudaMalloc((void**)&e->off, blocks * sizeof(long long)));
  JCK(cudaMalloc((void**)&e->sbuf, (size_t)e->n_stripes * e->stripe_words * 4)); JCK(cudaMemset(e->sbuf, 0, (size_t)e->n_stripes * e->stripe_words * 4));
  JCK(cudaMalloc((void**)&e->sbits, e->n_stripes * sizeof(long long)));
  JCK(cudaMalloc((void**)&e->s_static, e->n_stripes * sizeof(int))); JCK(cudaMemset(e->s_static, 0, e->n_stripes * sizeof(int)));
  JCK(cudaMalloc((void**)&e->s_flags, e->n_stripes * sizeof(int)));
  JCK(cudaMalloc((void**)&e->ssize, e->n_stripes * sizeof(uint32_t)));
  e->au_data_off = au_data_offset(e->n_stripes);
  // output capacity: 16 bits per pixel-equivalent (128 bytes per 8x8 block) — above anything quality <= 100 produces on real content;
  // a picture that would not fit is reported (AuHeader.overflow) and fails the session loudly instead of being truncated silently
  e->au_cap = (size_t)e->au_data_off + (size_t)e->n_stripes * (e->hdr_len + 2) + blocks * 128 + 4096;
  *out = e;
  return 0;
}

void jpeg_destroy(JpegEncoder* e) {
  if (!e) return;
  void* ptrs[] = {e->prev, e->hdr, e->lev, e->bits, e->off, e->sbuf, e->sbits, e->s_static, e->s_flags, e->qt, e->ssize};
  for (void* p : ptrs) if (p) cudaFree(p);
  delete e;
}
size_t jpeg_au_capacity(const JpegEncoder* e) { return e->au_cap; }
int jpeg_au_data_offset(const JpegEncoder* e) { return e->au_data_off; }
int jpeg_stripe_count(const JpegEncoder* e) { return e->n_stripes; }
int jpeg_stripe_rows(const JpegEncoder* e) { return e->stripe_rows; }

int jpeg_encode(JpegEncoder* e, const uint8_t* cur_nv12, uint8_t* au, int force_all, cudaStream_t st) {
  JpegCtx c{};
  c.cw = e->cfg.coded_w; c.ch = e->cfg.coded_h; c.w = e->cfg.width; c.h = e->cfg.height;
  c.mcu_w = e->mcu_w; c.mcu_h = e->mcu_h; c.stripe_rows = e->stripe_rows; c.n_stripes = e->n_stripes;
  c.cur = cur_nv12; c.prev = e->prev; c.lev = e->lev; c.bits = e->bits; c.off = e->off; c.sbuf = e->sbuf; c.stripe_words = e->stripe_words;
  c.sbits = e->sbits; c.s_static = e->s_static; c.s_flags = e->s_flags; c.ssize = e->ssize; c.qt = e->qt; c.hdr = e->hdr; c.hdr_len = e->hdr_len; c.hdr_h_off = e->hdr_h_off;
  c.first = (e->first || force_all) ? 1 : 0; c.paint_trigger = e->cfg.paint_trigger;
  c.au = au; c.au_cap = (long long)e->au_cap; c.au_data_off = e->au_data_off;
  const int blocks = e->mcu_w * e->mcu_h * 6;
  k_jpeg_diff<<<e->n_stripes, JT, 0, st>>>(c);
  k_jpeg_dct<<<(blocks + 127) / 128, 128, 0, st>>>(c);
  k_jpeg_code<false><<<(blocks + 127) / 128, 128, 0, st>>>(c);
  k_jpeg_scan<<<e->n_stripes, JT, 0, st>>>(c);
  k_jpeg_code<true><<<(blocks + 127) / 128, 128, 0, st>>>(c);
  k_jpeg_ff<<<e->n_stripes, JT, 0, st>>>(c);
  k_jpeg_pack<<<e->n_stripes, JT, 0, st>>>(c);
  e->first = false;
  return 7;
}

}  // namespace b2v
