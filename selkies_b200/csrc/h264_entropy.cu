// h264_entropy.cu — CAVLC entropy coding and byte-stream assembly (ITU-T H.264 7.3.4/7.3.5, 9.2, Annex B).
//
// Entropy coding is serial per slice in the bitstream, but nothing a macroblock writes depends on the
// BITS of its neighbours — only on their coefficient counts (nC) and motion vectors, which the
// analysis kernels already left in HBM.  So it is split into three data-parallel kernels:
//   k_cavlc_mb    one warp per macroblock, one LANE per residual block (27 blocks): each lane sizes its
//                 block, a warp prefix-sum places it, then it writes its codes with shared-memory atomicOr;
//                 result: a private bit string per macroblock (+ P_Skip decision, mvd from 8.4.1.3 prediction)
//   k_slice_build one block per chunk of up to 256 macroblocks of a slice: local scans + a decoupled look-back over the chunks of
//                 the slice give every macroblock its bit offset and its mb_skip_run; 8 threads per macroblock shift the bit
//                 strings into the slice RBSP (atomicOr); the chunk that finishes last counts the slice's emulation-prevention
//                 bytes; the last block of the picture runs the rate-control step
//   k_pack_au     one block per slice: prefix over slice sizes, emulation prevention (H264Escape; the count in k_slice_build
//                 and this copy share it, bitstream.cuh), start codes + NAL headers, parameter sets, AuHeader, band table.
// CPU restatement: oracle/h264_ref.c cavlc_block(), code_slice(), nal_write(), rc_update().
#include "h264_common.cuh"
#include "h264_cavlc.cuh"
#include "b2v_internal.h"
#include "h264_kernels.h"

namespace b2v {

// ------------------------------------------------------------------------------------------------ mv prediction (8.4.1.3, 8.4.1.1)
__device__ __forceinline__ int median3(int a, int b, int c) { return max(min(a, b), min(max(a, b), c)); }

// avX: neighbour partition available (inside the slice); rX: it is an inter macroblock with refIdx 0.
// Intra (I_PCM) and unavailable neighbours contribute mv 0 / refIdx -1.
struct MvCtx { bool avA, avB, avC, rA, rB, rC; int ax, ay, bx, by, cx, cy; };
__device__ __forceinline__ MvCtx mv_ctx(const FrameCtx& f, int mbx, int mby) {
  MvCtx m;
  const bool top = top_in_slice(f, mby);
  m.avA = left_in_slice(f, mbx); m.avB = top; m.avC = top && mbx + 1 < f.mbw;
  int cxi = mbx + 1;
  if (!m.avC) { cxi = mbx - 1; m.avC = top && mbx > 0; }      // C unavailable -> D
  m.ax = m.ay = m.bx = m.by = m.cx = m.cy = 0;
  m.rA = m.rB = m.rC = false;
  if (m.avA) { const MbInfo a = f.mbinfo[mby * f.mbw + mbx - 1]; if (a.type == MB_P16) { m.rA = true; m.ax = a.mvx; m.ay = a.mvy; } }
  if (m.avB) { const MbInfo b = f.mbinfo[(mby - 1) * f.mbw + mbx]; if (b.type == MB_P16) { m.rB = true; m.bx = b.mvx; m.by = b.mvy; } }
  if (m.avC) { const MbInfo c = f.mbinfo[(mby - 1) * f.mbw + cxi]; if (c.type == MB_P16) { m.rC = true; m.cx = c.mvx; m.cy = c.mvy; } }
  return m;
}
__device__ __forceinline__ void mv_pred16(const MvCtx& m, int& px, int& py) {
  if (!m.avB && !m.avC && m.avA) { px = m.ax; py = m.ay; return; }
  const int cnt = (int)m.rA + (int)m.rB + (int)m.rC;
  if (cnt == 1) { px = m.rA ? m.ax : m.rB ? m.bx : m.cx; py = m.rA ? m.ay : m.rB ? m.by : m.cy; return; }
  px = median3(m.ax, m.bx, m.cx); py = median3(m.ay, m.by, m.cy);
}
__device__ __forceinline__ void mv_pred_skip(const MvCtx& m, int& px, int& py) {
  px = py = 0;
  if (!m.avA || !m.avB) return;
  if ((m.rA && m.ax == 0 && m.ay == 0) || (m.rB && m.bx == 0 && m.by == 0)) return;
  mv_pred16(m, px, py);
}

// I_NxN macroblock header (7.3.5, 7.3.5.1): mb_type, 16 x (prev_intra4x4_pred_mode_flag [rem_intra4x4_pred_mode]),
// intra_chroma_pred_mode, coded_block_pattern (intra me(v) mapping), mb_qp_delta
template <class S>
__device__ __forceinline__ void mb_header_i4(S& h, const FrameCtx& f, const MbInfo& mi, int mb, int mbx, int mby) {
  put_ue(h, f.idr ? 0u : 5u);
  const uint8_t* own = f.i4modes + (size_t)mb * 16;
  const bool availA = left_in_slice(f, mbx), availB = top_in_slice(f, mby);
  const bool a_i4 = availA && f.mbinfo[mb - 1].type == MB_I4, b_i4 = availB && f.mbinfo[mb - f.mbw].type == MB_I4;
  for (int blk = 0; blk < 16; blk++) {
    const int bx = blk_x[blk], by = blk_y[blk], mode = own[by * 4 + bx];
    const int ma = bx > 0 ? (int)own[by * 4 + bx - 1] : !availA ? -1 : a_i4 ? (int)f.i4modes[(size_t)(mb - 1) * 16 + by * 4 + 3] : 2;
    const int mbm = by > 0 ? (int)own[(by - 1) * 4 + bx] : !availB ? -1 : b_i4 ? (int)f.i4modes[(size_t)(mb - f.mbw) * 16 + 12 + bx] : 2;
    const int pm = (ma < 0 || mbm < 0) ? 2 : min(ma, mbm);
    if (mode == pm) h.put(1, 1);
    else { h.put(1, 0); h.put(3, (uint32_t)(mode < pm ? mode : mode - 1)); }
  }
  put_ue(h, mi.chroma_mode);
  put_ue(h, cbp_to_codenum_intra[mi.cbp]);
  if (mi.cbp) put_se(h, 0);
}

// macroblock header of a coded (not P_Skip, not I_PCM) macroblock: I_NxN above; I_16x16: mb_type, intra_chroma_pred_mode,
// mb_qp_delta; P_L0_16x16: mb_type, mvd_l0, coded_block_pattern (inter me(v) mapping) [, mb_qp_delta]
template <class S>
__device__ __forceinline__ void mb_header(S& h, const FrameCtx& f, const MbInfo& mi, int mb, int mbx, int mby, int mvdx, int mvdy,
                                          int cbp_l, int cbp_c) {
  if (mi.type == MB_I4) mb_header_i4(h, f, mi, mb, mbx, mby);
  else if (mi.type == MB_I16) {
    const int tcode = 1 + mi.i16_mode + 4 * cbp_c + (cbp_l ? 12 : 0);
    put_ue(h, (uint32_t)(f.idr ? tcode : tcode + 5)); put_ue(h, mi.chroma_mode); put_se(h, 0);
  } else {
    put_ue(h, 0); put_se(h, mvdx); put_se(h, mvdy); put_ue(h, cbp_to_codenum_inter[mi.cbp]);
    if (mi.cbp) put_se(h, 0);
  }
}

// ------------------------------------------------------------------------------------------------ k_cavlc_mb
constexpr int CAVLC_WARPS = 4;

__global__ void __launch_bounds__(32 * CAVLC_WARPS) k_cavlc_mb(FrameCtx f) {
  __shared__ __align__(16) uint32_t s_words[CAVLC_WARPS][MB_WORDS];
  __shared__ __align__(16) int16_t s_lv[CAVLC_WARPS][32][16];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int mb = blockIdx.x * CAVLC_WARPS + warp;
  if (mb >= f.mbw * f.mbh) return;
  const int mbx = mb % f.mbw, mby = mb / f.mbw;
  const MbInfo mi = f.mbinfo[mb];
  uint32_t* words = s_words[warp];

  // ---- macroblock header fields ---------------------------------------------------------------------
  // (most macroblocks of a desktop picture leave through the P_Skip exit: nothing that only a coded macroblock needs — the bit
  // scratch, the mvd — is touched before it)
  const int cbp_l = mi.cbp & 15, cbp_c = mi.cbp >> 4;
  int mvdx = 0, mvdy = 0;
  if (!f.idr) {
    const MvCtx mc = mv_ctx(f, mbx, mby);
    if (mi.type == MB_P16 && mi.cbp == 0) {
      int sx, sy;
      mv_pred_skip(mc, sx, sy);
      if (mi.mvx == sx && mi.mvy == sy) {        // P_Skip: no bits; the slice scan folds it into mb_skip_run
        if (lane == 0) f.mb_nbits[mb] = 0x80000000u;
        return;
      }
    }
    int px, py;
    mv_pred16(mc, px, py);
    mvdx = mi.mvx - px; mvdy = mi.mvy - py;
  }
#pragma unroll
  for (int i = lane; i < MB_WORDS; i += 32) words[i] = 0;
  if (mi.type == MB_PCM) {                       // I_PCM: only mb_type here; alignment + 384 raw samples are placed by k_slice_bits
    if (lane == 0) {
      const uint32_t code = f.idr ? 25u : 30u;
      const int len = 2 * (31 - __clz(code + 1)) + 1;
      f.mb_words[(size_t)mb * MB_WORDS] = (code + 1) << (32 - len);
      f.mb_nbits[mb] = (uint32_t)len | 0x40000000u;
    }
    return;
  }
  // ---- which block does this lane code, and with which nC ---------------------------------------------
  // lane 0: Intra16x16 DC | 1..16: luma blkIdx lane-1 | 17,18: chroma DC | 19..26: chroma AC
  const uint8_t* nz_own = f.nnz + (size_t)mb * 32;
  const bool availA = left_in_slice(f, mbx), availB = top_in_slice(f, mby);
  const uint8_t* nz_a = f.nnz + (size_t)(mb - 1) * 32;
  const uint8_t* nz_b = f.nnz + (size_t)(mb - f.mbw) * 32;
  bool coded = false; int start = 0, maxc = 16, nC = 0, cblk = lane;
  if (lane == 0) { coded = mi.type == MB_I16; }
  else if (lane <= 16) { coded = (cbp_l >> ((lane - 1) >> 2)) & 1; if (mi.type == MB_I16) { start = 1; maxc = 15; } }
  else if (lane <= 18) { coded = cbp_c != 0; maxc = 4; nC = -1; }
  else if (lane <= 26) { coded = cbp_c == 2; start = 1; maxc = 15; }
  if (coded && nC == 0) {
    int na = 0, nb = 0; bool oka, okb;
    if (lane <= 16) {
      const int b = lane == 0 ? 0 : lane - 1, bx = blk_x[b], by = blk_y[b];
      oka = bx > 0 || availA; okb = by > 0 || availB;
      if (bx > 0) na = nz_own[by * 4 + bx - 1]; else if (availA) na = nz_a[by * 4 + 3];
      if (by > 0) nb = nz_own[(by - 1) * 4 + bx]; else if (availB) nb = nz_b[12 + bx];
    } else {
      const int c = (lane - 19) >> 2, b = (lane - 19) & 3, bx = b & 1, by = b >> 1;
      oka = bx > 0 || availA; okb = by > 0 || availB;
      if (bx > 0) na = nz_own[16 + c * 4 + by * 2]; else if (availA) na = nz_a[16 + c * 4 + by * 2 + 1];
      if (by > 0) nb = nz_own[16 + c * 4 + bx]; else if (availB) nb = nz_b[16 + c * 4 + 2 + bx];
    }
    nC = oka && okb ? (na + nb + 1) >> 1 : oka ? na : okb ? nb : 0;
  }
  // stage this lane's 16 levels in shared memory (dynamic indexing without local memory)
  if (lane < COEF_BLOCKS) {
    const uint4* src = reinterpret_cast<const uint4*>(f.coef + ((size_t)mb * COEF_BLOCKS + cblk) * 16);
    uint4* dst = reinterpret_cast<uint4*>(&s_lv[warp][lane][0]);
    if (coded) { dst[0] = src[0]; dst[1] = src[1]; }
  }
  __syncwarp();
  const int16_t* lv = &s_lv[warp][lane][start];

  // ---- pass 1: sizes ---------------------------------------------------------------------------------
  CountSink cs;
  if (coded) cavlc_block(cs, lv, maxc, nC);
  int hdr_bits;
  { CountSink h; mb_header(h, f, mi, mb, mbx, mby, mvdx, mvdy, cbp_l, cbp_c); hdr_bits = h.n; }
  int incl = cs.n;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(FULL, incl, d); if (lane >= d) incl += o; }
  const int total_bits = hdr_bits + __shfl_sync(FULL, incl, 31);
  const int my_off = hdr_bits + incl - cs.n;

  // ---- pass 2: write -----------------------------------------------------------------------------------
  if (lane == 0) { SmemSink h{words, 0, MB_WORDS * 32}; mb_header(h, f, mi, mb, mbx, mby, mvdx, mvdy, cbp_l, cbp_c); }
  if (coded) { SmemSink ws{words, my_off, MB_WORDS * 32}; cavlc_block(ws, lv, maxc, nC); }
  __syncwarp();
  int nb = total_bits;
  if (nb > MB_WORDS * 32) { nb = MB_WORDS * 32; if (lane == 0) atomicExch(f.overflow, 1); }
  uint32_t* dst = f.mb_words + (size_t)mb * MB_WORDS;
  for (int i = lane; i < (nb + 31) >> 5; i += 32) dst[i] = words[i];
  if (lane == 0) f.mb_nbits[mb] = (uint32_t)nb;
}

// ------------------------------------------------------------------------------------------------ slice header (7.3.3)
// of the slice at geo; first_mb_in_slice and frame_num count within its band (each band is a picture of its own when striped)
template <class S>
__device__ __forceinline__ void slice_header(S& s, const FrameCtx& f, const SliceGeo& geo, int qp) {
  const int band = geo.row0 / f.band_rows;
  const int first_mb = geo.mb0 - band * f.band_rows * f.mbw, frame_num = f.idr ? 0 : f.striped ? f.band_fn[band] : f.frame_num;
  put_ue(s, (uint32_t)first_mb);
  put_ue(s, f.idr ? 7u : 5u);
  put_ue(s, 0);
  s.put(8, (uint32_t)(frame_num & 255));
  if (f.idr) put_ue(s, (uint32_t)(f.idr_pic_id & 15));
  if (!f.idr) { s.put(1, 0); s.put(1, 0); }
  if (f.idr) { s.put(1, 0); s.put(1, 0); } else s.put(1, 0);
  put_se(s, qp - 26);
  put_ue(s, 1);
}

constexpr int SLICE_THREADS = 256;
static_assert(SLICE_THREADS == STUFF_THREADS, "the last chunk of a slice counts its emulation-prevention bytes");

// ---- rate-control / paint-over step, run by the LAST slice-scan block of the picture (thread 0).  The picture's RBSP bit count
// is known at that point (the byte stream adds emulation prevention, which the controller does not need), so the feedback
// record advances here while the rest of the byte-stream assembly is still to come.  Same integer arithmetic as
// oracle/h264_ref.c rc_step: prev = the record after picture k-1, used = the record picture k was coded from (after k-2).
__device__ __forceinline__ void rc_step(const FrameCtx& f, int qp_used, long long rbsp_bits) {
  RcState* rc = f.rc;
  const RcFb prev = rc->fb[(f.pic & 1) ^ 1], used = rc->fb[f.pic & 1];
  const int coded = __ldcg(&rc->pic_coded);      // stored by other blocks of this launch: read through L2
  rc->pic_coded = 0;
  rc->last_qp = qp_used; rc->frames++; rc->pic_bits = rbsp_bits;
  RcFb n = prev;
  const bool was_paint = f.paint_trigger > 0 && !f.idr && used.paint;
  if (f.idr || (coded && !was_paint)) { n.static_run = 0; n.remaining = 0; }
  else if (!coded) {
    n.static_run = min(prev.static_run + 1, RC_STATIC_PARK);
    if (f.paint_trigger > 0 && n.static_run == f.paint_trigger) n.remaining = f.paint_burst > 0 ? f.paint_burst : 1;
  }
  n.paint = n.remaining > 0;
  if (n.paint) n.remaining--;
  if (f.rc_mode == 0) {
    const long long bits = rbsp_bits + 40LL * f.n_slices;      // + start code and NAL header of every slice
    const long long T = f.target_bits < 1 ? 1 : f.target_bits;
    long long full = prev.fullness + bits - T;
    if (full < -4 * T) full = -4 * T;
    if (full > 64 * T) full = 64 * T;
    n.fullness = full;
    long long budget = T - full / 16;
    if (budget < T / 2) budget = T / 2;
    if (budget > 2 * T) budget = 2 * T;
    const int base = prev.qp < 0 ? rc_initial_qp(T, f.mbw * f.mbh) : prev.qp;
    int q = base;
    n.X = f.idr ? 0 : bits * rc_qs[qp_used];
    if (!f.idr) {
      const long long lim = budget * rc_qs[qp_used];
      const long long lo = prev.X > 0 && prev.X < n.X ? prev.X : n.X, hi = prev.X > n.X ? prev.X : n.X;
      const long long eff = hi > 3 * lo ? lo : (lo + hi) / 2;
      int qt = base;
      if (eff * 100 > lim * 104) {
        const int thr[9] = {104, 119, 133, 150, 168, 189, 238, 300, 378}, stp[9] = {1, 2, 3, 4, 5, 6, 8, 10, 12};
        int dq = 1;
#pragma unroll
        for (int i = 0; i < 9; i++) if (eff * 100 > lim * thr[i]) dq = stp[i];
        qt = qp_used + dq;
      } else if (hi * 100 < lim * 88 && full <= 0) {
        qt = qp_used - ((hi * 2 < lim && full < -2 * T) ? 2 : 1);
      }
      // debt (oracle rc_step): while the bucket holds more than RC_DEBT_PICTURES pictures' worth of overspend — recurring spikes the
      // two-picture rule lets through — a picture that coded anything makes the quantiser one step coarser
      if (full > (long long)RC_DEBT_PICTURES * T && coded && qt <= qp_used) qt = qp_used + 1;
      q = clip3i(base - 2, base + 4, qt);
    }
    n.qp = clip3i(RC_QP_MIN, RC_QP_MAX, q);
  }
  rc->fb[f.pic & 1] = n;
}

// ---- slice_ep_body: one block counts the emulation-prevention bytes slice s needs and publishes its NAL size
__device__ __forceinline__ void slice_ep_body(const FrameCtx& f, int s) {
  __shared__ int s_red[SLICE_THREADS / 32];
  const long long rbsp_bytes = __ldcg(&f.slice_rbsp[s]);
  const int t = count_escapes<H264Escape>(f.slice_buf + (size_t)s * f.slice_words, rbsp_bytes, s_red);
  if (threadIdx.x == 0) {
    const SliceGeo geo = slice_geo(f, s);
    const int start_len = (geo.row0 % f.band_rows == 0 && geo.x0 == 0 && !f.idr) ? 4 : 3;     // 4-byte start code on the first NAL of (each band's) access unit
    f.slice_size[s] = (uint32_t)(start_len + 1 + rbsp_bytes + t);
  }
}

// ---- k_slice_build: one block per CHUNK of up to 256 consecutive macroblocks of a slice, so a slice of many rows is built
// by many blocks instead of one long loop.  What a chunk needs from the chunks in front of it is (a) the bit position where it starts
// and (b) the mb_skip_run still open at that point — the first coded macroblock of a chunk codes ue(open run + its own leading skips),
// whose LENGTH is the only thing in a chunk that depends on the carry.  Decoupled look-back (the chunks of a slice are consecutive
// blocks of this grid, lower-numbered blocks never wait for higher ones): every chunk publishes its AGGREGATE as soon as its local
// scans are done (has a coded macroblock?  skips in front of the first / behind the last one, bits of everything but that one ue),
// folds the aggregates of its predecessors — or starts from the nearest published INCLUSIVE state — and publishes its own inclusive
// state.  A chunk that holds an I_PCM macroblock (byte alignment: its length depends on its position) publishes no usable aggregate;
// its successors wait for its inclusive state instead.  Then every chunk shifts its macroblocks' bit strings into the slice RBSP
// (8 threads per macroblock, offsets from shared memory), the chunk that holds the slice's last macroblock appends the trailing
// skip run + rbsp_trailing_bits, and the last chunk of a slice to FINISH counts the slice's emulation-prevention bytes.
struct ChunkAgg { int flag; int has; int first_run; int trailing; long long rest_bits; };   // has: bit 0 coded macroblock present, bit 1 I_PCM inside (no aggregate)
struct ChunkInc { int flag; int trailing; long long bits; };
constexpr int CHUNK_MAX_POLLS = 1 << 22;
constexpr int COPY_LANES = 8;      // threads per macroblock in the bit-string copy

__device__ __forceinline__ bool wait_flag(const volatile int* flag, int tag) {
  int spins = 0;
  while (*flag != tag) if (++spins > CHUNK_MAX_POLLS) return false;
  __threadfence();
  return true;
}

__global__ void __launch_bounds__(SLICE_THREADS, 8) k_slice_build(FrameCtx f) {
  __shared__ long long s_warp_sum[SLICE_THREADS / 32];
  __shared__ int s_warp_max[SLICE_THREADS / 32];
  __shared__ uint32_t s_nb[SLICE_THREADS];       // nbits | I_PCM flag (bit 30), 0xffffffff = skipped
  __shared__ int s_run[SLICE_THREADS];
  __shared__ long long s_off[SLICE_THREADS];
  __shared__ long long s_bits_in, s_bits_out;
  __shared__ int s_trail_in, s_trail_out, s_first, s_flag;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int cps = f.chunks_per_slice, s = blockIdx.x / cps, k = blockIdx.x - s * cps;
  const SliceGeo geo = slice_geo(f, s);
  const int n_chunks = (geo.n_mb + SLICE_THREADS - 1) / SLICE_THREADS;
  const int tag = f.pic + 1, qp = frame_qp(f);
  uint32_t* out = f.slice_buf + (size_t)s * f.slice_words;
  bool active = k < n_chunks;
  const int idx0 = k * SLICE_THREADS, n = active ? min(SLICE_THREADS, geo.n_mb - idx0) : 0, mb_first = geo.mb0 + idx0;
  const bool last_chunk = active && k == n_chunks - 1;
  if (active) {
    // ---- local scans -------------------------------------------------------------------------------------------------------
    uint32_t nbits = 0; bool skip = true, pcm = false;
    if (tid < n) { const uint32_t v = f.mb_nbits[mb_first + tid]; skip = (v >> 31) != 0; pcm = ((v >> 30) & 1u) != 0; nbits = v & 0x3fffffffu; }
    const bool any_pcm = __syncthreads_or(pcm) != 0;
    int incl_max = skip ? -1 : tid;            // last coded macroblock (local index) up to and including this one
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int o = __shfl_up_sync(FULL, incl_max, d); if (lane >= d) incl_max = max(incl_max, o); }
    if (lane == 31) s_warp_max[warp] = incl_max;
    __syncthreads();
    int prev_max = -1, last_coded = -1;
    for (int w = 0; w < SLICE_THREADS / 32; w++) { if (w < warp) prev_max = max(prev_max, s_warp_max[w]); last_coded = max(last_coded, s_warp_max[w]); }
    int excl_max = __shfl_up_sync(FULL, incl_max, 1);
    if (lane == 0) excl_max = -1;
    excl_max = max(excl_max, prev_max);
    const bool first_coded = !skip && excl_max < 0;
    if (tid == 0) s_first = n;                 // skips in front of the first coded macroblock (n: none coded)
    __syncthreads();
    if (first_coded) s_first = tid;
    const int run_local = tid - 1 - excl_max;  // for every coded macroblock but the first: its mb_skip_run
    const int pre = (!skip && !first_coded && !f.idr) ? ue_len((uint32_t)run_local) : 0;
    const long long tot = skip ? 0 : (long long)pre + nbits;
    long long incl = tot;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const long long o = __shfl_up_sync(FULL, incl, d); if (lane >= d) incl += o; }
    if (lane == 31) s_warp_sum[warp] = incl;
    __syncthreads();
    long long woff = 0, rest = 0;
    for (int w = 0; w < SLICE_THREADS / 32; w++) { if (w < warp) woff += s_warp_sum[w]; rest += s_warp_sum[w]; }
    const long long off_local = woff + incl - tot;       // bits of this chunk in front of the macroblock, without the first ue
    const int first = s_first, trailing_local = last_coded >= 0 ? n - 1 - last_coded : n;
    // ---- publish the aggregate, get the carry --------------------------------------------------------------------------------
    if (tid == 0) {
      ChunkAgg* a = f.chunk_agg + blockIdx.x;
      a->has = (last_coded >= 0 ? 1 : 0) | (any_pcm ? 2 : 0); a->first_run = first; a->trailing = trailing_local; a->rest_bits = rest;
      __threadfence();
      *reinterpret_cast<volatile int*>(&a->flag) = tag;
    }
    if (warp == 0) {
      // base state in front of chunk 0: the slice header (every chunk can size it: no waiting for chunk 0)
      long long bits; int trail = 0; bool ok = true;
      { CountSink h; slice_header(h, f, geo, qp); bits = h.n; }
      int start = 0;
      // nearest predecessor whose inclusive state is already there (32 at a time, nearest first)
      for (int hi = k - 1; hi >= 0 && start == 0; hi -= 32) {
        const int j = hi - lane;
        const bool ready = j >= 0 && *reinterpret_cast<const volatile int*>(&f.chunk_inc[blockIdx.x - k + j].flag) == tag;
        const unsigned m = __ballot_sync(FULL, ready);
        if (m) {
          const int jj = hi - (__ffs(m) - 1);
          __threadfence();
          const ChunkInc* c = f.chunk_inc + (blockIdx.x - k + jj);
          bits = *reinterpret_cast<const volatile long long*>(&c->bits); trail = *reinterpret_cast<const volatile int*>(&c->trailing);
          start = jj + 1;
        }
      }
      // fold the aggregates of chunks start .. k-1, 32 loads at a time
      for (int base = start; base < k; base += 32) {
        const int j = base + lane;
        int has = 0, fr = 0, tr = 0; long long rb = 0, ib = 0; int it = 0;
        if (j < k) {
          const ChunkAgg* a = f.chunk_agg + (blockIdx.x - k + j);
          ok &= wait_flag(&a->flag, tag);
          has = *reinterpret_cast<const volatile int*>(&a->has);
          if (has & 2) {                       // I_PCM inside: only its inclusive state will do
            const ChunkInc* c = f.chunk_inc + (blockIdx.x - k + j);
            ok &= wait_flag(&c->flag, tag);
            ib = *reinterpret_cast<const volatile long long*>(&c->bits); it = *reinterpret_cast<const volatile int*>(&c->trailing);
          } else {
            fr = *reinterpret_cast<const volatile int*>(&a->first_run); tr = *reinterpret_cast<const volatile int*>(&a->trailing);
            rb = *reinterpret_cast<const volatile long long*>(&a->rest_bits);
          }
        }
        const int cnt = min(32, k - base);
        for (int t = 0; t < cnt; t++) {
          const int h2 = __shfl_sync(FULL, has, t), fr2 = __shfl_sync(FULL, fr, t), tr2 = __shfl_sync(FULL, tr, t);
          const long long rb2 = __shfl_sync(FULL, rb, t), ib2 = __shfl_sync(FULL, ib, t); const int it2 = __shfl_sync(FULL, it, t);
          const int n_j = min(SLICE_THREADS, geo.n_mb - (base + t) * SLICE_THREADS);
          if (h2 & 2) { bits = ib2; trail = it2; }
          else if (h2 & 1) { bits += (f.idr ? 0 : ue_len((uint32_t)(trail + fr2))) + rb2; trail = tr2; }
          else trail += n_j;
        }
      }
      ok = __all_sync(FULL, ok);
      if (lane == 0) { s_bits_in = bits; s_trail_in = trail; if (!ok) atomicExch(f.overflow, 4); }
    }
    __syncthreads();
    const long long bits_in = s_bits_in; const int trail_in = s_trail_in;
    // ---- final offsets ----------------------------------------------------------------------------------------------------------
    const int run_first = trail_in + first;
    const int pre_first = (last_coded >= 0 && !f.idr) ? ue_len((uint32_t)run_first) : 0;
    int run = first_coded ? run_first : run_local;
    long long my_off = bits_in + off_local + ((!skip && !first_coded) ? pre_first : 0);
    s_nb[tid] = skip ? 0xffffffffu : (nbits | (pcm ? 0x40000000u : 0u)); s_run[tid] = run; s_off[tid] = my_off;
    if (tid == 0) { s_bits_out = bits_in + rest + pre_first; s_trail_out = last_coded >= 0 ? trailing_local : trail_in + n; }
    __syncthreads();
    if (any_pcm && tid == 0) {                   // byte alignment of the raw samples: serial walk (pathological content only)
      long long pos = bits_in;
      for (int j = 0; j < n; j++) {
        const uint32_t nb = s_nb[j];
        if (nb == 0xffffffffu) continue;
        s_off[j] = pos;
        pos += (f.idr ? 0 : ue_len((uint32_t)s_run[j])) + (nb & 0x3fffffffu);
        if (nb & 0x40000000u) pos = ((pos + 7) & ~7LL) + 384 * 8;
      }
      s_bits_out = pos;
    }
    __syncthreads();
    if (tid == 0) {
      ChunkInc* c = f.chunk_inc + blockIdx.x;
      c->bits = s_bits_out; c->trailing = s_trail_out;
      __threadfence();
      *reinterpret_cast<volatile int*>(&c->flag) = tag;
      if (k == 0) { GlobalSink g{out, 0}; slice_header(g, f, geo, qp); }     // (the bits it occupies were counted above)
      if (last_chunk) {                          // trailing mb_skip_run, rbsp_trailing_bits
        GlobalSink g{out, s_bits_out};
        const int runt = s_trail_out;
        if (!f.idr && runt > 0) put_ue(g, (uint32_t)runt);
        f.slice_bits[s] = g.pos;
        if (runt < geo.n_mb) {                   // the slice holds a coded macroblock (benign races: every writer stores the same value)
          f.rc->pic_coded = 1;
          if (f.striped) f.band_coded[geo.row0 / f.band_rows] = 1;
        }
        g.put(1, 1);
        f.slice_rbsp[s] = (uint32_t)((g.pos + 7) >> 3);
      }
    }
  }
  // ---- the last block of the picture to get here runs the rate-control step (every block read its QP at its start) --------------
  if (tid == 0) {
    __threadfence();
    s_flag = atomicAdd(&f.rc->scan_done, 1) == (int)gridDim.x - 1;
  }
  __syncthreads();
  if (s_flag) {
    __threadfence();
    long long bits = 0;
    for (int j = tid; j < f.n_slices; j += SLICE_THREADS) bits += __ldcg(&f.slice_bits[j]);
    __syncthreads();
    const long long t = block_sum<SLICE_THREADS>(bits, s_warp_sum);
    if (tid == 0) {
      f.rc->scan_done = 0;
      rc_step(f, qp, t);
    }
  }
  if (!active) return;
  // ---- copy: COPY_LANES threads per macroblock shift its bit string into the slice RBSP ----------------------------------------
  {
    const int sub = tid % COPY_LANES;
    for (int i = tid / COPY_LANES; i < n; i += SLICE_THREADS / COPY_LANES) {
      const uint32_t v = s_nb[i];
      if (v == 0xffffffffu) continue;            // P_Skip: folded into a later mb_skip_run
      const bool pcm = (v & 0x40000000u) != 0;
      const uint32_t nbits = v & 0x3fffffffu;
      const int mb = mb_first + i, mby = mb / f.mbw, mbx = mb - mby * f.mbw;
      long long pos = s_off[i];
      if (!f.idr) {
        const uint32_t run = (uint32_t)s_run[i];
        if (sub == 0) { GlobalSink g{out, pos}; put_ue(g, run); }
        pos += ue_len(run);
      }
      const uint32_t* src = f.mb_words + (size_t)mb * MB_WORDS;
      for (int w = sub; w < (int)((nbits + 31) >> 5); w += COPY_LANES) or_word(out, pos + 32LL * w, src[w]);
      if (pcm) {     // I_PCM payload: 256 luma, 64 Cb, 64 Cr samples from the reconstruction (== source), byte aligned
        const long long pp = (pos + nbits + 7) & ~7LL;
        const int px = mbx * 16, py = mby * 16;
        const uint8_t* ry = f.recon; const uint8_t* ruv = f.recon + (size_t)f.cw * f.ch;
        for (int w = sub; w < 96; w += COPY_LANES) {
          uint32_t q;
          if (w < 64) q = __byte_perm(__ldcg(reinterpret_cast<const uint32_t*>(ry + (size_t)(py + (w >> 2)) * f.cw + px + (w & 3) * 4)), 0, 0x0123);
          else {
            const int kk = (w - 64) & 15, comp = (w - 64) >> 4;
            const uint2 c2 = __ldcg(reinterpret_cast<const uint2*>(ruv + (size_t)(py / 2 + (kk >> 1)) * f.cw + px + (kk & 1) * 8));
            q = comp == 0 ? __byte_perm(c2.x, c2.y, 0x0246) : __byte_perm(c2.x, c2.y, 0x1357);
          }
          or_word(out, pp + 32LL * w, q);
        }
      }
    }
  }
  // ---- the chunk of a slice that finishes last counts the slice's emulation-prevention bytes --------------------------------------
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    const bool lastf = atomicAdd(&f.slice_done[s], 1) == n_chunks - 1;
    if (lastf) f.slice_done[s] = 0;
    s_flag = lastf;
  }
  __syncthreads();
  if (s_flag) { __threadfence(); slice_ep_body(f, s); }
}

// ------------------------------------------------------------------------------------------------ k_pack_au
constexpr int PACK_THREADS = STUFF_THREADS;

__global__ void __launch_bounds__(PACK_THREADS) k_pack_au(FrameCtx f, long long au_cap) {
  __shared__ long long s_base;
  __shared__ long long s_part[PACK_THREADS / 32];
  __shared__ int s_wsum[PACK_THREADS / 32];
  __shared__ int s_carry;
  const int s = blockIdx.x, tid = threadIdx.x;
  // the controller has already moved on to the next picture (rc_step ran in k_slice_build, before this kernel and possibly on another
  // stream): this picture's QP is the one it recorded
  const int qp = f.rc->last_qp;
  // byte offset of this slice's NAL inside the access unit
  long long part = 0;
  for (int j = tid; j < s; j += PACK_THREADS) part += f.slice_size[j];
  part = block_sum<PACK_THREADS>(part, s_part);
  const SliceGeo geo = slice_geo(f, s);
  const int row0 = geo.row0, band = row0 / f.band_rows;
  const bool band_first = row0 == band * f.band_rows && geo.x0 == 0;      // this slice opens its band's access unit
  const int plen = (f.striped && band == f.n_bands - 1) ? f.param_len_last : f.param_len;
  if (tid == 0) s_base = part + (f.idr ? (long long)band * f.param_len + plen : 0);     // parameter sets of bands 0..band precede this NAL
  __syncthreads();
  uint8_t* au = f.au + f.au_data_off;
  const long long cap = au_cap - (long long)f.au_data_off;
  const long long base = s_base;
  uint32_t* rbsp = f.slice_buf + (size_t)s * f.slice_words;
  const long long n = f.slice_rbsp[s];
  const int start_len = (band_first && !f.idr) ? 4 : 3;
  if (tid == 0 && base + start_len + 1 <= cap) {
    long long o = base;
    if (start_len == 4) au[o++] = 0;
    au[o++] = 0; au[o++] = 0; au[o++] = 1;
    au[o++] = (uint8_t)(((f.idr ? 3 : 2) << 5) | (f.idr ? 5 : 1));
  }
  const long long out0 = base + start_len + 1;
  stuff_copy<H264Escape>(rbsp, n, au + out0, cap - out0, s_wsum, s_carry);
  clear_bits<PACK_THREADS>(rbsp, n, f.slice_words);
  if (band_first) {
    if (f.idr && base <= cap) {
      const uint8_t* ps = f.param_sets + ((f.striped && band == f.n_bands - 1) ? f.param_len : 0);
      for (int i = tid; i < plen; i += PACK_THREADS) au[base - plen + i] = ps[i];
    }
    if (f.striped && tid == 0) {      // band table entry; the band's frame_num advances only if it is delivered
      long long sz = f.idr ? plen : 0;
      const int band_row1 = min(f.mbh, (band + 1) * f.band_rows);
      const int s1 = min(f.n_slices, f.seg_cols ? band_row1 * segs_per_row(f) : (band_row1 + f.slice_rows - 1) / f.slice_rows);
      for (int j = s; j < s1; j++) sz += f.slice_size[j];
      const int coded = f.idr ? 1 : f.band_coded[band];
      const int fn = f.idr ? 0 : f.band_fn[band];
      BandEntry* be = reinterpret_cast<BandEntry*>(f.au + sizeof(AuHeader)) + band;
      be->off = (int32_t)(base - (f.idr ? plen : 0)); be->size = (int32_t)sz; be->coded = coded; be->frame_num = fn;
      f.band_fn[band] = (fn + (coded ? 1 : 0)) & 255;
      f.band_coded[band] = 0;
    }
  }
  if (s == 0) {
    if (tid == 0) {
      long long total = f.idr ? (long long)(f.n_bands - 1) * f.param_len + (f.striped ? f.param_len_last : f.param_len) : 0, bits = 0;
      for (int j = 0; j < f.n_slices; j++) { total += f.slice_size[j]; bits += f.slice_bits[j]; }
      AuHeader* h = reinterpret_cast<AuHeader*>(f.au);
      int ovf = *f.overflow;
      if (total > cap) { ovf |= 2; total = cap; }
      h->size = (int32_t)total; h->qp = qp; h->is_idr = f.idr; h->n_slices = f.n_slices; h->total_bits = bits;
      h->overflow = ovf;
      h->next_qp = f.rc->fb[f.pic & 1].qp;         // the controller's decision for the picture two ahead
      h->csc_t0 = f.csc_ts ? f.csc_ts[0] : 0; h->csc_t1 = f.csc_ts ? f.csc_ts[1] : 0;
    }
  }
}

int launch_cavlc(const FrameCtx& f, cudaStream_t st) {
  const int mbs = f.mbw * f.mbh;
  k_cavlc_mb<<<(mbs + CAVLC_WARPS - 1) / CAVLC_WARPS, 32 * CAVLC_WARPS, 0, st>>>(f);
  return 1;
}
int launch_slice_build(const FrameCtx& f, cudaStream_t st) {
  FrameCtx g = f;
  const int full = f.seg_cols ? f.seg_cols : f.slice_rows * f.mbw;       // macroblocks of a full-size slice of this picture
  g.chunks_per_slice = (full + SLICE_THREADS - 1) / SLICE_THREADS;
  k_slice_build<<<f.n_slices * g.chunks_per_slice, SLICE_THREADS, 0, st>>>(g);      // scan + copy + emulation-prevention count
  return 1;
}
int launch_pack_cap(const FrameCtx& f, long long au_cap, cudaStream_t st) {
  k_pack_au<<<f.n_slices, PACK_THREADS, 0, st>>>(f, au_cap);
  return 1;
}

}  // namespace b2v
