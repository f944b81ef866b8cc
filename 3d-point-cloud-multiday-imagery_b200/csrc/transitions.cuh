// Day-pair transition counts of a cluster map (mdkm_bind_day_transitions): for every pair (a, b)
// the number of pixels whose state is s on day a and t on day b, with state = label + 1 where the
// pixel produced a point and 0 where it did not -- exactly the values of the cluster map.
#pragma once
#include "common.cuh"

namespace mdkm {

constexpr int kTransPx = 16;  // pixels per lane and round: one 16-byte load per day at uint8

// where a CTA accumulates the (k+1)^2 bins of a pair before they reach the global ones
enum { kTransWarpBins = 0, kTransCtaBins = 1, kTransGlobalBins = 2 };

struct TransParams {
  const void* map;           // [D][HW] states, 1 or 2 bytes each: the whole stack
  long long HW;
  long long q_begin, q_end;  // the pixels of every day this rank bins
  const int* pairs;          // [n_pairs][2] days
  int n_pairs;
  int k1;                    // states: k + 1
  unsigned long long* bins;  // [n_pairs][k1 * k1], cleared by the host
};

// the 16 bytes at byte offset s (0..15, warp-uniform) of the 32 bytes lo:hi
__device__ __forceinline__ uint4 realign16(const uint4& lo, const uint4& hi, int s) {
  const unsigned int w[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
  const int ws = s >> 2;
  const unsigned int sh = (unsigned int)(s & 3) * 8u;
  unsigned int u[5];
#pragma unroll
  for (int i = 0; i < 5; ++i) u[i] = ws == 0 ? w[i] : (ws == 1 ? w[i + 1] : (ws == 2 ? w[i + 2] : w[i + 3]));
  return make_uint4(__funnelshift_r(u[0], u[1], sh), __funnelshift_r(u[1], u[2], sh),
                    __funnelshift_r(u[2], u[3], sh), __funnelshift_r(u[3], u[4], sh));
}

// kTransPx states of type T starting at p (any element address) as 32-bit words; `s` is p's
// offset from 16-byte alignment: 0 loads aligned vectors, otherwise one more vector is loaded
// and the bytes are shifted into place (the extra bytes lie in the same aligned 16-byte block
// as the last state read, so they are inside the map's allocation)
template <typename T>
__device__ __forceinline__ void load_states(const T* p, int s, unsigned int (&w)[kTransPx * sizeof(T) / 4]) {
  constexpr int kVec = kTransPx * sizeof(T) / 16;
  const uint4* v = reinterpret_cast<const uint4*>(reinterpret_cast<const unsigned char*>(p) - s);
  uint4 r[kVec];
  if (s == 0) {
#pragma unroll
    for (int i = 0; i < kVec; ++i) r[i] = __ldg(v + i);
  } else {
    uint4 a[kVec + 1];
#pragma unroll
    for (int i = 0; i <= kVec; ++i) a[i] = __ldg(v + i);
#pragma unroll
    for (int i = 0; i < kVec; ++i) r[i] = realign16(a[i], a[i + 1], s);
  }
#pragma unroll
  for (int i = 0; i < kVec; ++i) {
    w[4 * i] = r[i].x; w[4 * i + 1] = r[i].y; w[4 * i + 2] = r[i].z; w[4 * i + 3] = r[i].w;
  }
}

// state of pixel e (0..15) of packed words (a select over the words: no local-memory indexing)
template <typename T>
__device__ __forceinline__ int state_at(const unsigned int (&w)[kTransPx * sizeof(T) / 4], int e) {
  const int wi = e * (int)sizeof(T) / 4;
  unsigned int v = w[0];
#pragma unroll
  for (int i = 1; i < kTransPx * (int)sizeof(T) / 4; ++i) v = wi == i ? w[i] : v;
  return (int)((v >> ((e * 8 * (int)sizeof(T)) & 31)) & (sizeof(T) == 1 ? 0xffu : 0xffffu));
}

// bit e set: pixel e has state sa on day a and sb on day b (SIMD compares of the packed words;
// the multiply gathers the top bit of every byte / half-word into the top bits of the word)
template <typename T>
__device__ __forceinline__ unsigned int pair_mask(const unsigned int (&wa)[kTransPx * sizeof(T) / 4],
                                                  const unsigned int (&wb)[kTransPx * sizeof(T) / 4], int sa, int sb) {
  unsigned int m = 0u;
  if (sizeof(T) == 1) {
    const unsigned int ba = (unsigned int)sa * 0x01010101u, bb = (unsigned int)sb * 0x01010101u;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const unsigned int e = __vcmpeq4(wa[i], ba) & __vcmpeq4(wb[i], bb) & 0x80808080u;
      m |= ((e * 0x00204081u) >> 28) << (4 * i);
    }
  } else {
    const unsigned int ba = (unsigned int)sa * 0x00010001u, bb = (unsigned int)sb * 0x00010001u;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const unsigned int e = __vcmpeq2(wa[i], ba) & __vcmpeq2(wb[i], bb) & 0x80008000u;
      m |= ((e * 0x00008001u) >> 30) << (2 * i);
    }
  }
  return m;
}

// Adds this lane's pixels to the bins: bit e of `rem` set = pixel e, with its states packed in
// wa (day a) and wb (day b), bin key = state_a * k1 + state_b.  Warp-synchronous.  The pixels of
// a lane with equal keys are counted together first (neighbouring pixels nearly always share
// one: one round for a uniform chunk), then the lanes holding the same key (__match_any_sync,
// one key per lane and round) are summed and their leader adds the total: a round costs one
// update per distinct key.  kTransWarpBins: `s_bins` is this warp's own copy, updated without
// atomics -- the keys of one round are distinct, and __syncwarp orders the rounds;
// kTransCtaBins: the CTA's copy, shared atomics; kTransGlobalBins: `g_bins`, 64-bit global
// atomics.
template <typename T, int kMode>
__device__ __forceinline__ void trans_add(unsigned int* s_bins, unsigned long long* g_bins,
                                          const unsigned int (&wa)[kTransPx * sizeof(T) / 4],
                                          const unsigned int (&wb)[kTransPx * sizeof(T) / 4], int k1, unsigned int rem,
                                          int lane) {
  while (__any_sync(0xffffffffu, rem != 0)) {
    int mine = -1, cnt = 0;
    if (rem) {
      const int e = __ffs(rem) - 1;
      const int sa = state_at<T>(wa, e), sb = state_at<T>(wb, e);
      const unsigned int hit = pair_mask<T>(wa, wb, sa, sb) & rem;
      mine = sa * k1 + sb;
      cnt = __popc(hit);
      rem &= ~hit;
    }
    const unsigned int peers = __match_any_sync(0xffffffffu, mine);
    cnt = __reduce_add_sync(peers, cnt);
    if (mine >= 0 && lane == __ffs(peers) - 1) {
      if (kMode == kTransWarpBins) s_bins[mine] += (unsigned int)cnt;
      else if (kMode == kTransCtaBins) atomicAdd(&s_bins[mine], (unsigned int)cnt);
      else atomicAdd(&g_bins[mine], (unsigned long long)cnt);
    }
    if (kMode == kTransWarpBins) __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------
// Transition counts of the requested day pairs.  blockIdx.y strides over the pairs, blockIdx.x
// over 16-pixel chunks of [q_begin, q_end) aligned to 16 bytes in day a; day b is read at the
// same pixels (its vectors shifted into place when (b - a) * HW is not a multiple of 16 bytes);
// the head and tail of the range (fewer than 16 pixels each) are read element by element.  Bin
// key = state_a * k1 + state_b.  With shared bins (32-bit: the host sizes the grid so that no
// CTA bins 2^31 pixels of a pair) every CTA flushes the non-zero bins of a pair with 64-bit
// global atomics before it moves on to the next pair.
// ---------------------------------------------------------------------------------------
template <typename T, int kMode>
__global__ void __launch_bounds__(kThreads, 4) day_transitions_kernel(const TransParams p) {
  extern __shared__ __align__(16) unsigned int s_trans[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nb = p.k1 * p.k1;
  constexpr int kCopies = kMode == kTransWarpBins ? kThreads / 32 : 1;
  unsigned int* s_bins = kMode == kTransWarpBins ? s_trans + warp * nb : s_trans;
  if (kMode != kTransGlobalBins) {
    for (int i = tid; i < kCopies * nb; i += kThreads) s_trans[i] = 0u;
    __syncthreads();
  }
  const T* map = static_cast<const T*>(p.map);
  for (int pr = blockIdx.y; pr < p.n_pairs; pr += gridDim.y) {
    const T* ma = map + (long long)__ldg(p.pairs + 2 * pr) * p.HW;
    const T* mb = map + (long long)__ldg(p.pairs + 2 * pr + 1) * p.HW;
    unsigned long long* g_bins = p.bins + (size_t)pr * nb;
    const long long len = p.q_end - p.q_begin;
    const long long head = min(len, (long long)((16u - ((unsigned int)(size_t)(ma + p.q_begin) & 15u)) & 15u) / (long long)sizeof(T));
    const long long q0 = p.q_begin + head;
    const long long n_chunks = (p.q_end - q0) / kTransPx;
    const long long q_tail = q0 + n_chunks * kTransPx;
    const int sb = (int)((unsigned int)(size_t)(mb + q0) & 15u);
    constexpr int kWords = kTransPx * sizeof(T) / 4;
    unsigned int wa[kWords], wb[kWords];
    for (long long c = (long long)blockIdx.x * kThreads + tid; c - lane < n_chunks; c += (long long)gridDim.x * kThreads) {
      unsigned int rem = 0u;
      if (c < n_chunks) {
        load_states<T>(ma + q0 + c * kTransPx, 0, wa);
        load_states<T>(mb + q0 + c * kTransPx, sb, wb);
        rem = (1u << kTransPx) - 1u;
      }
      trans_add<T, kMode>(s_bins, g_bins, wa, wb, p.k1, rem, lane);
    }
    if (blockIdx.x == 0 && warp == 0) {  // lane 0: the head, lane 1: the tail
      const long long lo = lane == 0 ? p.q_begin : q_tail, hi = lane == 0 ? q0 : p.q_end;
      unsigned int rem = 0u;
#pragma unroll
      for (int i = 0; i < kWords; ++i) wa[i] = wb[i] = 0u;
#pragma unroll
      for (int e = 0; e < kTransPx; ++e) {
        if (lane < 2 && lo + e < hi) {
          const int sh = (e % (4 / sizeof(T))) * 8 * sizeof(T);
          wa[e * sizeof(T) / 4] |= (unsigned int)ma[lo + e] << sh;
          wb[e * sizeof(T) / 4] |= (unsigned int)mb[lo + e] << sh;
          rem |= 1u << e;
        }
      }
      trans_add<T, kMode>(s_bins, g_bins, wa, wb, p.k1, rem, lane);
    }
    if (kMode != kTransGlobalBins) {
      __syncthreads();
      for (int i = tid; i < nb; i += kThreads) {
        unsigned long long v = 0ull;
#pragma unroll
        for (int w = 0; w < kCopies; ++w) {
          v += s_trans[w * nb + i];
          s_trans[w * nb + i] = 0u;
        }
        if (v) atomicAdd(&g_bins[i], v);
      }
      __syncthreads();
    }
  }
}

}  // namespace mdkm
