// csc.cu — fused BGRA -> BT.709 limited-range NV12 colour conversion (+ bilinear scale), sm_100a.
//
// Replaces the colour-conversion stage of the reference's native capture module
// (pixelflux, call site src/selkies/media_pipeline.py:299-300; legacy GStreamer
// `videoconvert`, docs/component.md:338-344).  Integer spec: DESIGN.md §3; the CPU
// restatement it must match bit-for-bit is oracle/csc_ref.c.
//
// Roofline: HBM-bound streaming kernel, 4 B/px read + 1.5 B/px written (5.5 B/px algorithmic).
//   fast path  (1:1, width % 4 == 0): one thread = 4 px x 2 rows per unit: two 16-byte loads
//              (ld.global.nc.L1::no_allocate.v4), two 4-byte Y stores and one 4-byte CbCr store, all
//              warp-contiguous (512 B / 128 B / 128 B per warp instruction).  Two units per thread are
//              issued back to back so four 16-byte loads are in flight per thread.
//   arithmetic: dp2a (two 16-bit coefficient x 8-bit pixel MACs per instruction); rounding
//              constant and the +16 / +128 offsets are folded into the accumulator seed.
//   scaled path (bilinear scale, 16-byte aligned source): one CTA per 64 x 8 output tile, its source footprint staged in
//              shared memory.
//   general path (ragged widths, unaligned scaled sources, footprints over 96 KB): one thread per 2x2 output block, taps
//              from tables.
// A TMA / mbarrier variant of the 1:1 kernel was built, measured slower at 4K and equal at 8K, and removed (profiles/README.md).
#include "b2v_internal.h"

namespace b2v {

// tools/lab/csc_lab.cu compiles this file with -DCSC_TRACE to get a per-CTA timeline; the library build has none of it
#ifdef CSC_TRACE
__device__ __forceinline__ unsigned long long trace_now() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define TRACE_START(cta) do { if (threadIdx.x == 0) { unsigned sm; asm volatile("mov.u32 %0, %%smid;" : "=r"(sm)); g_trace[4 * (cta)] = trace_now(); g_trace[4 * (cta) + 2] = sm; } } while (0)
#define TRACE_END(cta) do { __syncthreads(); if (threadIdx.x == 0) g_trace[4 * (cta) + 1] = trace_now(); } while (0)
#else
#define TRACE_START(cta)
#define TRACE_END(cta)
#endif

__device__ __forceinline__ int dp2a_lo(int coef, unsigned px, int acc) {
  int d; asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(coef), "r"(px), "r"(acc)); return d;
}
__device__ __forceinline__ int dp2a_hi(int coef, unsigned px, int acc) {
  int d; asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(coef), "r"(px), "r"(acc)); return d;
}
__device__ __forceinline__ uint4 ld_stream(const uint8_t* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ void st_stream(uint8_t* p, unsigned v) {
  asm volatile("st.global.cs.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// pixel word: byte0 = B, byte1 = G, byte2 = R, byte3 = A (ignored: coefficient 0)
__host__ __device__ constexpr int pack16(int lo, int hi) { return (int)(((unsigned)lo & 0xffffu) | ((unsigned)hi << 16)); }
// Colour matrices (14-bit coefficients).  0: BT.709 limited range, the H.264 path (DESIGN.md §3).  1: JFIF full-range BT.601, the
// JPEG stripe path (0.5 is coded as 8191 so that a saturated red / blue stays at 255; greys still give exactly 128) — the same
// numbers as oracle/csc_ref.c MATRIX[].
template <int M> struct Mx;
template <> struct Mx<0> { static constexpr int YR = KYR, YG = KYG, YB = KYB, UR = KUR, UG = KUG, UB = KUB, VR = KVR, VG = KVG, VB = KVB, YOFF = 16; };
template <> struct Mx<1> { static constexpr int YR = 4899, YG = 9617, YB = 1868, UR = -2765, UG = -5427, UB = 8191, VR = 8191, VG = -6860, VB = -1332, YOFF = 0; };
__device__ const int c_mx[2][10] = {{KYR, KYG, KYB, KUR, KUG, KUB, KVR, KVG, KVB, 16}, {4899, 9617, 1868, -2765, -5427, 8191, 8191, -6860, -1332, 0}};
constexpr int Y_SEED = (16 << 14) + (1 << 13);      // matrix 0
constexpr int C_SEED = (128 << 16) + (1 << 15);

__device__ __forceinline__ unsigned dp2a_lo_u(unsigned coef, unsigned px, unsigned acc) {
  unsigned d; asm("dp2a.lo.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(coef), "r"(px), "r"(acc)); return d;
}
__device__ __forceinline__ unsigned dp2a_hi_u(unsigned coef, unsigned px, unsigned acc) {
  unsigned d; asm("dp2a.hi.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(coef), "r"(px), "r"(acc)); return d;
}
// Luma with the coefficients scaled by 4 (all three are positive and 4*KYG still fits an UNSIGNED 16-bit dp2a lane):
// 4*(k.px) + 4*seed puts (k.px + seed) >> 14 into byte 2 of the accumulator, exactly (the factor 4 is exact), so the result is
// picked up by the same byte permute that packs four pixels — no shift instruction per pixel.  Chroma (>> 16) sits in byte 2 already.
template <int M>
__device__ __forceinline__ unsigned luma_b2(unsigned px) {      // Y in byte 2
  using X = Mx<M>;
  static_assert(4 * X::YG < 65536 && 4 * (X::YR + X::YG + X::YB) * 255 + 4 * ((X::YOFF << 14) + (1 << 13)) < (1 << 24), "luma accumulator must stay below byte 3");
  constexpr unsigned lo = (unsigned)pack16(4 * X::YB, 4 * X::YG), hi = (unsigned)pack16(4 * X::YR, 0), seed = 4u * (unsigned)((X::YOFF << 14) + (1 << 13));
  return dp2a_hi_u(hi, px, dp2a_lo_u(lo, px, seed));
}
__device__ __forceinline__ int chroma_acc(int clo, int chi, unsigned px, int acc) {
  return dp2a_hi(chi, px, dp2a_lo(clo, px, acc));
}
// byte 2 of each of four accumulators -> one word
__device__ __forceinline__ unsigned pack4_b2(unsigned a, unsigned b, unsigned c, unsigned d) {
  return __byte_perm(__byte_perm(a, b, 0x0062), __byte_perm(c, d, 0x0062), 0x5410);
}

// 4 px x 2 rows -> Y (two u32) + CbCr (one u32 = Cb0 Cr0 Cb1 Cr1)
template <int M = 0>
__device__ __forceinline__ void convert_quad(const uint4& a, const uint4& b, unsigned& y0, unsigned& y1, unsigned& uv) {
  using X = Mx<M>;
  constexpr int CU_LO = pack16(X::UB, X::UG), CU_HI = pack16(X::UR, 0), CV_LO = pack16(X::VB, X::VG), CV_HI = pack16(X::VR, 0);
  y0 = pack4_b2(luma_b2<M>(a.x), luma_b2<M>(a.y), luma_b2<M>(a.z), luma_b2<M>(a.w));
  y1 = pack4_b2(luma_b2<M>(b.x), luma_b2<M>(b.y), luma_b2<M>(b.z), luma_b2<M>(b.w));
  int u0 = chroma_acc(CU_LO, CU_HI, b.y, chroma_acc(CU_LO, CU_HI, b.x, chroma_acc(CU_LO, CU_HI, a.y, chroma_acc(CU_LO, CU_HI, a.x, C_SEED))));
  int v0 = chroma_acc(CV_LO, CV_HI, b.y, chroma_acc(CV_LO, CV_HI, b.x, chroma_acc(CV_LO, CV_HI, a.y, chroma_acc(CV_LO, CV_HI, a.x, C_SEED))));
  int u1 = chroma_acc(CU_LO, CU_HI, b.w, chroma_acc(CU_LO, CU_HI, b.z, chroma_acc(CU_LO, CU_HI, a.w, chroma_acc(CU_LO, CU_HI, a.z, C_SEED))));
  int v1 = chroma_acc(CV_LO, CV_HI, b.w, chroma_acc(CV_LO, CV_HI, b.z, chroma_acc(CV_LO, CV_HI, a.w, chroma_acc(CV_LO, CV_HI, a.z, C_SEED))));
  uv = pack4_b2((unsigned)u0, (unsigned)v0, (unsigned)u1, (unsigned)v1);
}

// ---- fast path ---------------------------------------------------------------------------
// grid.x covers 4-px quads of a row, grid.y strides over groups of U row pairs.
constexpr int CSC_U = 2;         // units (row pairs) per thread
constexpr int CSC_BLOCK = 160;   // threads per block (launch_csc steps down to 128 / 96 / 64 when one of those divides the row)
template <int M>
__global__ void __launch_bounds__(256) csc_bgra_nv12_fast(CscParams p, int quads, int pairs) {
  constexpr int U = CSC_U;
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  TRACE_START(blockIdx.y * gridDim.x + blockIdx.x);
  if (p.ts && threadIdx.x == 0) {   // device-side stopwatch of this launch: first block start .. last block end
    unsigned long long t0; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0)); atomicMin(p.ts, t0);
  }
  const uint8_t* __restrict__ src = p.src + (size_t)(q < quads ? q : 0) * 16;
  if (q < quads)
  for (int pr0 = blockIdx.y * U; pr0 < pairs; pr0 += gridDim.y * U) {
    uint4 a[U], b[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      int pr = pr0 + u;
      if (pr < pairs) {
        int r0 = min(2 * pr, p.src_h - 1), r1 = min(2 * pr + 1, p.src_h - 1);   // bottom padding rows replicate
        a[u] = ld_stream(src + (size_t)r0 * p.src_stride);
        b[u] = ld_stream(src + (size_t)r1 * p.src_stride);
      }
    }
#pragma unroll
    for (int u = 0; u < U; u++) {
      int pr = pr0 + u;
      if (pr < pairs) {
        unsigned y0, y1, uv;
        convert_quad<M>(a[u], b[u], y0, y1, uv);
        st_stream(p.out_y + (size_t)(2 * pr) * p.coded_w + q * 4, y0);
        st_stream(p.out_y + (size_t)(2 * pr + 1) * p.coded_w + q * 4, y1);
        st_stream(p.out_uv + (size_t)pr * p.coded_w + q * 4, uv);
      }
    }
  }
  if (p.ts) {
    __syncthreads();
    if (threadIdx.x == 0) { unsigned long long t1; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1)); atomicMax(p.ts + 1, t1); }
  }
  TRACE_END(blockIdx.y * gridDim.x + blockIdx.x);
}

// ---- general path: bilinear scale and/or ragged width, one thread per 2x2 output block -----
__device__ __forceinline__ void fetch_bgr(const CscParams& p, int x, int y, int& B, int& G, int& R) {
  int x0, x1, fx, y0, y1, fy;
  if (p.tx) { Tap t = p.tx[x]; x0 = t.i0; x1 = t.i1; fx = t.f; } else { x0 = x1 = x; fx = 0; }
  if (p.ty) { Tap t = p.ty[y]; y0 = t.i0; y1 = t.i1; fy = t.f; } else { y0 = y1 = y; fy = 0; }
  const uint8_t* r0 = p.src + (size_t)y0 * p.src_stride;
  const uint8_t* r1 = p.src + (size_t)y1 * p.src_stride;
  unsigned p00 = *(const unsigned*)(r0 + x0 * 4);
  if (fx == 0 && fy == 0) { B = p00 & 255; G = (p00 >> 8) & 255; R = (p00 >> 16) & 255; return; }
  unsigned p01 = *(const unsigned*)(r0 + x1 * 4), p10 = *(const unsigned*)(r1 + x0 * 4), p11 = *(const unsigned*)(r1 + x1 * 4);
  int out[3];
#pragma unroll
  for (int c = 0; c < 3; c++) {
    int s = 8 * c;
    int top = (int)((p00 >> s) & 255) * (256 - fx) + (int)((p01 >> s) & 255) * fx;
    int bot = (int)((p10 >> s) & 255) * (256 - fx) + (int)((p11 >> s) & 255) * fx;
    out[c] = (top * (256 - fy) + bot * fy + (1 << 15)) >> 16;
  }
  B = out[0]; G = out[1]; R = out[2];
}

__global__ void __launch_bounds__(256) csc_bgra_nv12_general(CscParams p) {
  int bx = blockIdx.x * blockDim.x + threadIdx.x;   // 2x2 block column
  int by = blockIdx.y * blockDim.y + threadIdx.y;
  if (bx * 2 >= p.coded_w || by * 2 >= p.coded_h) return;
  const int* mx = c_mx[p.matrix];
  int sb = 0, sg = 0, sr = 0;
  unsigned yy[4];
#pragma unroll
  for (int k = 0; k < 4; k++) {
    int x = min(bx * 2 + (k & 1), p.dst_w - 1), y = min(by * 2 + (k >> 1), p.dst_h - 1);
    int B, G, R;
    fetch_bgr(p, x, y, B, G, R);
    yy[k] = (unsigned)(mx[0] * R + mx[1] * G + mx[2] * B + (mx[9] << 14) + (1 << 13)) >> 14;
    sb += B; sg += G; sr += R;
  }
  unsigned cb = (unsigned)(mx[3] * sr + mx[4] * sg + mx[5] * sb + C_SEED) >> 16;
  unsigned cr = (unsigned)(mx[6] * sr + mx[7] * sg + mx[8] * sb + C_SEED) >> 16;
  *(uint16_t*)(p.out_y + (size_t)(by * 2) * p.coded_w + bx * 2) = (uint16_t)(yy[0] | (yy[1] << 8));
  *(uint16_t*)(p.out_y + (size_t)(by * 2 + 1) * p.coded_w + bx * 2) = (uint16_t)(yy[2] | (yy[3] << 8));
  *(uint16_t*)(p.out_uv + (size_t)by * p.coded_w + bx * 2) = (uint16_t)(cb | (cr << 8));
}

// ---- scaled path: fused bilinear scale + CSC through a shared-memory tile -----------------------------------------------------
// One CTA produces SC_TW x SC_TH output pixels (one thread per 2x2 block: the chroma sample needs all four).  The source
// footprint of the tile — tx[first].i0 .. tx[last].i1 by ty[first].i0 .. ty[last].i1, a few KB whatever the scale factor — is
// staged in shared memory with 16-byte loads; every tap is then a shared-memory read.  The arithmetic is the spec's (oracle/
// csc_ref.c fetch_bgr): per channel top/bottom horizontal blends at full precision (B and R ride in the two 16-bit halves of one
// word: 255*256 fits), one vertical blend, one rounding.  Roofline: 4 B per source pixel read + 1.5 B per output pixel written.
constexpr int SC_TW = 64, SC_TH = 8, SC_THREADS = (SC_TW / 2) * (SC_TH / 2);

__device__ __forceinline__ void blend_px(const uint32_t* r0, const uint32_t* r1, int x0, int x1, int fx, int fy, int& B, int& G, int& R) {
  const uint32_t p00 = r0[x0], p01 = r0[x1], p10 = r1[x0], p11 = r1[x1];
  const uint32_t M = 0x00ff00ffu;
  const uint32_t wx1 = (uint32_t)fx, wx0 = 256u - wx1;
  const uint32_t tbr = (p00 & M) * wx0 + (p01 & M) * wx1, bbr = (p10 & M) * wx0 + (p11 & M) * wx1;        // [B | R << 16], each <= 65280
  const uint32_t tg = ((p00 >> 8) & 255u) * wx0 + ((p01 >> 8) & 255u) * wx1, bg = ((p10 >> 8) & 255u) * wx0 + ((p11 >> 8) & 255u) * wx1;
  const uint32_t wy1 = (uint32_t)fy, wy0 = 256u - wy1;
  B = (int)(((tbr & 0xffffu) * wy0 + (bbr & 0xffffu) * wy1 + (1u << 15)) >> 16);
  R = (int)(((tbr >> 16) * wy0 + (bbr >> 16) * wy1 + (1u << 15)) >> 16);
  G = (int)((tg * wy0 + bg * wy1 + (1u << 15)) >> 16);
}

__global__ void __launch_bounds__(SC_THREADS) csc_bgra_nv12_scaled(CscParams p, int fw_cap, int fh_cap) {
  extern __shared__ __align__(16) uint32_t sc_tile[];            // fh_cap rows of fw_cap pixels (fw_cap % 4 == 0)
  const int tid = threadIdx.x;
  const int ox0 = blockIdx.x * SC_TW, oy0 = blockIdx.y * SC_TH;
  // footprint of this tile in the source (output coordinates beyond the visible picture replicate its last row / column)
  const int xf = min(ox0, p.dst_w - 1), xl = min(ox0 + SC_TW - 1, p.dst_w - 1);
  const int yf = min(oy0, p.dst_h - 1), yl = min(oy0 + SC_TH - 1, p.dst_h - 1);
  const int xs0 = p.tx[xf].i0 & ~3, xs1 = p.tx[xl].i1, ys0 = p.ty[yf].i0, ys1 = p.ty[yl].i1;
  const int fw4 = (xs1 - xs0 + 4) >> 2, fh = ys1 - ys0 + 1;      // quads per row, rows
  for (int i = tid; i < fh * fw4; i += SC_THREADS) {
    const int r = i / fw4, c = i - r * fw4, sx = xs0 + 4 * c;
    const uint8_t* g = p.src + (size_t)(ys0 + r) * p.src_stride + (size_t)sx * 4;
    uint4 v;
    if (sx + 3 < p.src_w) v = ld_stream(g);
    else {                                                      // last quad of a row whose width is not a multiple of 4
      v.x = *reinterpret_cast<const uint32_t*>(g);
      v.y = sx + 1 < p.src_w ? *reinterpret_cast<const uint32_t*>(g + 4) : 0u;
      v.z = sx + 2 < p.src_w ? *reinterpret_cast<const uint32_t*>(g + 8) : 0u;
      v.w = 0u;
    }
    *reinterpret_cast<uint4*>(&sc_tile[r * fw_cap + 4 * c]) = v;
  }
  (void)fh_cap;
  __syncthreads();
  const int bx = tid % (SC_TW / 2), by = tid / (SC_TW / 2);
  const int ox = ox0 + 2 * bx, oy = oy0 + 2 * by;
  if (ox >= p.coded_w || oy >= p.coded_h) return;
  const int* mx = c_mx[p.matrix];
  int sb = 0, sg = 0, sr = 0;
  unsigned yy[4];
#pragma unroll
  for (int k = 0; k < 4; k++) {
    const int x = min(ox + (k & 1), p.dst_w - 1), y = min(oy + (k >> 1), p.dst_h - 1);
    const Tap ax = p.tx[x], ay = p.ty[y];
    int B, G, R;
    blend_px(&sc_tile[(ay.i0 - ys0) * fw_cap], &sc_tile[(ay.i1 - ys0) * fw_cap], ax.i0 - xs0, ax.i1 - xs0, ax.f, ay.f, B, G, R);
    yy[k] = (unsigned)(mx[0] * R + mx[1] * G + mx[2] * B + (mx[9] << 14) + (1 << 13)) >> 14;
    sb += B; sg += G; sr += R;
  }
  const unsigned cb = (unsigned)(mx[3] * sr + mx[4] * sg + mx[5] * sb + C_SEED) >> 16;
  const unsigned cr = (unsigned)(mx[6] * sr + mx[7] * sg + mx[8] * sb + C_SEED) >> 16;
  *reinterpret_cast<uint16_t*>(p.out_y + (size_t)oy * p.coded_w + ox) = (uint16_t)(yy[0] | (yy[1] << 8));
  *reinterpret_cast<uint16_t*>(p.out_y + (size_t)(oy + 1) * p.coded_w + ox) = (uint16_t)(yy[2] | (yy[3] << 8));
  *reinterpret_cast<uint16_t*>(p.out_uv + (size_t)(oy >> 1) * p.coded_w + ox) = (uint16_t)(cb | (cr << 8));
}

// host side ---------------------------------------------------------------------------------
void make_taps_host(Tap* t, int dn, int sn) {
  for (int d = 0; d < dn; d++) {
    if (dn == sn) { t[d] = Tap{d, d, 0, 0}; continue; }
    int64_t pos = (((int64_t)(2 * d + 1) * sn) << 15) / dn - (1 << 15);
    int64_t hi = (int64_t)(sn - 1) << 16;
    if (pos < 0) pos = 0;
    if (pos > hi) pos = hi;
    int i0 = (int)(pos >> 16);
    t[d] = Tap{i0, i0 + 1 < sn ? i0 + 1 : sn - 1, (int)((pos >> 8) & 255), 0};
  }
}

int launch_csc(const CscParams& p, cudaStream_t st) {
  const bool fast = p.tx == nullptr && p.ty == nullptr && p.dst_w == p.src_w && p.dst_h == p.src_h && p.coded_w == p.dst_w &&
                    (p.coded_w % 4) == 0 && (p.src_stride % 16) == 0 && ((uintptr_t)p.src % 16) == 0 &&
                    ((uintptr_t)p.out_y % 4) == 0 && ((uintptr_t)p.out_uv % 4) == 0;
  if (fast) {
    int quads = p.coded_w / 4, pairs = p.coded_h / 2;
    int block = CSC_BLOCK;
    while (quads % block != 0 && block > 64) block -= 32;   // prefer a divisor of the row
    if (quads % block != 0) block = CSC_BLOCK;
    int gx = (quads + block - 1) / block;
    int gy = (pairs + CSC_U - 1) / CSC_U;                    // one U-group per block
    if (gy > 65535) gy = 65535;
    dim3 grid(gx, gy);
    if (p.matrix == 1) csc_bgra_nv12_fast<1><<<grid, block, 0, st>>>(p, quads, pairs);
    else csc_bgra_nv12_fast<0><<<grid, block, 0, st>>>(p, quads, pairs);
  } else {
    // scaled: the tiled kernel when the tile's source footprint fits shared memory (any sane scale factor), else the general one
    if (p.tx && p.ty && (p.src_stride % 16) == 0 && ((uintptr_t)p.src % 16) == 0) {
      const long long fw = ((long long)SC_TW * p.src_w + p.dst_w - 1) / p.dst_w + 8, fh = ((long long)SC_TH * p.src_h + p.dst_h - 1) / p.dst_h + 3;
      const int fw_cap = (int)((fw + 3) & ~3LL), fh_cap = (int)fh;
      const long long smem = (long long)fw_cap * fh_cap * 4;
      if (smem <= 96 * 1024) {
        static int attr = 0;
        if (smem > 48 * 1024 && smem > attr) { cudaFuncSetAttribute(csc_bgra_nv12_scaled, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); attr = (int)smem; }
        dim3 grid((p.coded_w + SC_TW - 1) / SC_TW, (p.coded_h + SC_TH - 1) / SC_TH);
        csc_bgra_nv12_scaled<<<grid, SC_THREADS, (size_t)smem, st>>>(p, fw_cap, fh_cap);
        return 1;
      }
    }
    dim3 block(32, 8);
    dim3 grid((p.coded_w / 2 + 31) / 32, (p.coded_h / 2 + 7) / 8);
    csc_bgra_nv12_general<<<grid, block, 0, st>>>(p);
  }
  return 1;
}

}  // namespace b2v
