// h264_cavlc.cuh — the CAVLC residual-block coder (ITU-T H.264 9.2), shared by the entropy kernels (which write bits) and
// the analysis kernels (which only SIZE a macroblock to decide I_PCM).
#pragma once
#include "bitstream.cuh"
#include "h264_tables.cuh"

namespace b2v {

constexpr int NC_CHROMA_DC = -1;   // coeff_token table for chroma DC
constexpr int NC_WORST = -2;       // size estimate: the longest coeff_token of the four nC tables

// lv: scan-order levels of the block, already offset by its first coded position; maxc = 16, 15 or 4
template <class S>
__device__ __forceinline__ void cavlc_block(S& s, const int16_t* lv, int maxc, int nC) {
  uint32_t nz = 0, ones = 0;
  for (int k = 0; k < maxc; k++) { const int v = lv[k]; nz |= (uint32_t)(v != 0) << k; ones |= (uint32_t)(v == 1 || v == -1) << k; }
  const int total = __popc(nz);
  int t1 = 0;
  { uint32_t m = nz; while (m && t1 < 3) { const int top = 31 - __clz(m); if (!((ones >> top) & 1)) break; t1++; m ^= 1u << top; } }
  const int ti = 4 * total + t1;
  if (nC == NC_CHROMA_DC) s.put(chroma_dc_coeff_token_len[ti], chroma_dc_coeff_token_bits[ti]);
  else if (nC == NC_WORST) s.put(max(max((int)coeff_token_len[0][ti], (int)coeff_token_len[1][ti]), max((int)coeff_token_len[2][ti], (int)coeff_token_len[3][ti])), 0);
  else { const int tab = nC < 2 ? 0 : nC < 4 ? 1 : nC < 8 ? 2 : 3; s.put(coeff_token_len[tab][ti], coeff_token_bits[tab][ti]); }
  if (!total) return;
  uint32_t m = nz;
  for (int i = 0; i < t1; i++) { const int top = 31 - __clz(m); s.put(1, lv[top] < 0 ? 1u : 0u); m ^= 1u << top; }
  int suffix_len = (total > 10 && t1 < 3) ? 1 : 0;
  bool first = true;
  while (m) {
    const int top = 31 - __clz(m); m ^= 1u << top;
    const int level = lv[top];
    int code = level > 0 ? 2 * level - 2 : -2 * level - 1;
    if (first && t1 < 3) code -= 2;
    first = false;
    if (suffix_len == 0) {
      if (code < 14) s.put(code + 1, 1);
      else if (code < 30) { s.put(15, 1); s.put(4, (uint32_t)(code - 14)); }
      else { s.put(16, 1); s.put(12, (uint32_t)(code - 30)); }
    } else {
      if (code < (15 << suffix_len)) { s.put((code >> suffix_len) + 1, 1); s.put(suffix_len, (uint32_t)(code & ((1 << suffix_len) - 1))); }
      else { s.put(16, 1); s.put(12, (uint32_t)(code - (15 << suffix_len))); }
    }
    if (suffix_len == 0) suffix_len = 1;
    if (abs(level) > (3 << (suffix_len - 1)) && suffix_len < 6) suffix_len++;
  }
  const int zeros = (31 - __clz(nz)) + 1 - total;
  if (total < maxc) {
    if (nC == NC_CHROMA_DC) s.put(chroma_dc_total_zeros_len[total - 1][zeros], chroma_dc_total_zeros_bits[total - 1][zeros]);
    else s.put(total_zeros_len[total - 1][zeros], total_zeros_bits[total - 1][zeros]);
  }
  int left = zeros;
  m = nz;
  while (left > 0 && (m & (m - 1))) {
    const int top = 31 - __clz(m); m ^= 1u << top;
    const int run = top - (31 - __clz(m)) - 1;
    const int tix = min(left, 7) - 1;
    s.put(run_len[tix][run], run_bits[tix][run]);
    left -= run;
  }
}

}  // namespace b2v
