// bitstream.cuh — what the H.264 (h264_entropy.cu) and JPEG (jpeg.cu) byte-stream back ends share: bit sinks, the escape rule
// of each codec, and the block-wide helpers.  A unit (slice, stripe) is coded into a zeroed bit string of big-endian u32 words
// (atomicOr), sized by count_escapes() and written by stuff_copy(); both apply the codec's rule through escape_mask(), so a
// unit's size and its bytes cannot disagree.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace b2v {

// ------------------------------------------------------------------------------------------------ bit sinks
struct CountSink {          // sizes what a writer would write
  int n = 0;
  __device__ __forceinline__ void put(int len, uint32_t) { n += len; }
};
// MSB-first, concurrent writers use atomicOr; v must fit in len bits.  CHECKED: bits past cap_bits are counted, not written.
template <class Pos, bool CHECKED>
struct BitSink {
  uint32_t* w; Pos pos; Pos cap_bits;
  __device__ __forceinline__ void put(int len, uint32_t v) {
    if (len == 0) return;
    if (!CHECKED || pos + len <= cap_bits) {
      const Pos wi = pos >> 5; const int o = (int)(pos & 31), space = 32 - o;
      if (len <= space) atomicOr(&w[wi], v << (space - len));
      else { atomicOr(&w[wi], v >> (len - space)); atomicOr(&w[wi + 1], v << (32 - (len - space))); }
    }
    pos += len;
  }
};
using SmemSink = BitSink<int, true>;           // per-macroblock scratch in shared memory
using GlobalSink = BitSink<long long, false>;  // a unit's bit string in global memory

template <class S> __device__ __forceinline__ void put_ue(S& s, uint32_t v) { const int len = 31 - __clz(v + 1); s.put(2 * len + 1, v + 1); }
template <class S> __device__ __forceinline__ void put_se(S& s, int v) { put_ue(s, v > 0 ? (uint32_t)(2 * v - 1) : (uint32_t)(-2 * v)); }
__device__ __forceinline__ int ue_len(uint32_t v) { return 2 * (31 - __clz(v + 1)) + 1; }

// a whole word at any bit position (a bit string copied into another one)
__device__ __forceinline__ void or_word(uint32_t* out, long long bitpos, uint32_t v) {
  if (!v) return;
  const long long wi = bitpos >> 5; const int o = (int)(bitpos & 31);
  if (o == 0) atomicOr(&out[wi], v);
  else { atomicOr(&out[wi], v >> o); atomicOr(&out[wi + 1], v << (32 - o)); }
}

// byte i of a bit string, through L2 (other blocks of the same launch may have written it)
__device__ __forceinline__ uint32_t stream_byte(const uint32_t* w, long long i) { return (__ldcg(&w[i >> 2]) >> (24 - 8 * (int)(i & 3))) & 255u; }

// ------------------------------------------------------------------------------------------------ block helpers
// Sum of v over a block of THREADS threads, returned to thread 0; s_warp: THREADS / 32 shared slots no thread still reads.
template <int THREADS, class T>
__device__ __forceinline__ T block_sum(T v, T* s_warp) {
  if constexpr (sizeof(T) == 4) v = __reduce_add_sync(0xffffffffu, v);
  else {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  }
  if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = v;
  __syncthreads();
  T t = 0;
  if (threadIdx.x == 0) for (int w = 0; w < THREADS / 32; w++) t += s_warp[w];
  return t;
}

// Exclusive prefix sum of v over a block of THREADS threads, starting at s_carry, which then advances by the block's total.
template <int THREADS, class T>
__device__ __forceinline__ T block_scan(T v, T* s_warp, T& s_carry) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  T incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { const T o = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += o; }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  T before = s_carry;
  for (int w = 0; w < warp; w++) before += s_warp[w];
  before += incl - v;
  __syncthreads();
  if (threadIdx.x == THREADS - 1) s_carry = before + v;
  __syncthreads();
  return before;
}

// Zero the words a unit of nbytes used (and the one behind), so the next picture can OR into its bit string again.
template <int THREADS>
__device__ __forceinline__ void clear_bits(uint32_t* w, long long nbytes, long long words) {
  const long long nw = min(words, (nbytes >> 2) + 2);
  for (long long i = threadIdx.x; i < nw; i += THREADS) w[i] = 0;
}

// ------------------------------------------------------------------------------------------------ escapes
// A policy is made at byte i of a bit string, then sees the bytes from i on; true: the byte gets CODE in front (BEFORE) or behind.
struct H264Escape {         // emulation prevention (7.4.1): 03 in front of a byte <= 3 that follows an even run of >= 2 zero bytes
  static constexpr bool BEFORE = true; static constexpr uint8_t CODE = 3;
  int z = 0;                // zero bytes in front of the next byte
  __device__ __forceinline__ H264Escape(const uint32_t* w, long long i) { while (i - 1 - z >= 0 && stream_byte(w, i - 1 - z) == 0u) z++; }
  __device__ __forceinline__ bool operator()(uint32_t b) { const bool e = b <= 3u && z >= 2 && (z & 1) == 0; z = b == 0u ? z + 1 : 0; return e; }
};
struct JpegEscape {         // byte stuffing (T.81 B.1.1.5): 00 behind every FF of entropy-coded data
  static constexpr bool BEFORE = false; static constexpr uint8_t CODE = 0;
  __device__ __forceinline__ JpegEscape(const uint32_t*, long long) {}
  __device__ __forceinline__ bool operator()(uint32_t b) const { return b == 255u; }
};

constexpr int STUFF_THREADS = 256;     // block size of the count and the copy
constexpr int STUFF_CH = 16;           // bytes per thread per round

__device__ __forceinline__ uint32_t byte_of(const uint32_t (&words)[STUFF_CH / 4], int k) { return (words[k >> 2] >> (24 - 8 * (k & 3))) & 255u; }

// words: bytes i0 .. i0 + STUFF_CH - 1 of a unit of n bytes; returns the mask of those (< n) the policy escapes
template <class P>
__device__ __forceinline__ uint32_t escape_mask(const uint32_t* w, long long i0, long long n, uint32_t (&words)[STUFF_CH / 4]) {
  uint32_t m = 0;
  if (i0 < n) {
#pragma unroll
    for (int j = 0; j < STUFF_CH / 4; j++) words[j] = i0 + 4 * j < n ? __ldcg(&w[(i0 >> 2) + j]) : 0u;
    P esc(w, i0);
#pragma unroll
    for (int k = 0; k < STUFF_CH; k++) if (esc(byte_of(words, k)) && i0 + k < n) m |= 1u << k;
  }
  return m;
}

// escape bytes a unit of n bytes needs, returned to thread 0 (a block of STUFF_THREADS threads)
template <class P>
__device__ __forceinline__ int count_escapes(const uint32_t* w, long long n, int* s_warp) {
  int cnt = 0;
  for (long long i0 = (long long)threadIdx.x * STUFF_CH; i0 < n; i0 += (long long)STUFF_THREADS * STUFF_CH) {
    uint32_t words[STUFF_CH / 4];
    cnt += __popc(escape_mask<P>(w, i0, n, words));
  }
  return block_sum<STUFF_THREADS>(cnt, s_warp);
}

// Copies a unit of n bytes to out[0 ..) with its escapes, dropping stores at or past cap; returns the escapes inserted.
template <class P>
__device__ __forceinline__ int stuff_copy(const uint32_t* in, long long n, uint8_t* out, long long cap, int* s_warp, int& s_carry) {
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (long long cb = 0; cb < n; cb += (long long)STUFF_THREADS * STUFF_CH) {
    const long long i0 = cb + (long long)threadIdx.x * STUFF_CH;
    uint32_t words[STUFF_CH / 4];
    const uint32_t esc = escape_mask<P>(in, i0, n, words);
    long long o = i0 + block_scan<STUFF_THREADS>(__popc(esc), s_warp, s_carry);
#pragma unroll
    for (int k = 0; k < STUFF_CH; k++) {
      if (i0 + k < n) {
        const bool e = (esc >> k) & 1u;
        if (P::BEFORE && e) { if (o < cap) out[o] = P::CODE; o++; }
        if (o < cap) out[o] = (uint8_t)byte_of(words, k);
        o++;
        if (!P::BEFORE && e) { if (o < cap) out[o] = P::CODE; o++; }
      }
    }
  }
  return s_carry;
}

}  // namespace b2v
