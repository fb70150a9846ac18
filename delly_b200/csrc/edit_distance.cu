// edit_distance.cu — batched Myers bit-vector edit distance (NW / SHW / HW, distance + first end
// location), the device replacement for edlibAlign(..., EDLIB_TASK_DISTANCE).
//
// Reference semantics reproduced (results only; the Ukkonen band schedule of the CPU code is an
// optimisation that does not change results):
//   src/edlib.cpp:139-294  edlibAlign driver: empty-sequence rules, k auto-doubling, NW end location
//   src/edlib.cpp:407-442  calculateBlock (Myers/Hyyro advance-block)
//   src/edlib.cpp:545-702  HW/SHW: min over target columns of D[m][c], k=min(k,|q|) for HW, -1 if > k,
//                          positions in increasing order (we return the first)
//   src/edlib.cpp:728-929  NW: -1 if k < |n-m|, k=min(k,max(m,n)), D[m][n] if <= k
//
// Device design (B200, integer-ALU bound; HBM traffic is ~(|q|+|t|)/2..1 byte per 30+ int ops):
//   * jobs are binned on the device by ceil(|q|/32) (counting sort: count -> offsets -> scatter),
//   * |q| <= 128: ONE THREAD PER JOB. The whole DP column is one multi-word bit-vector held in
//     registers (NW = 1..4 x 32 bit, add-with-carry chain, funnel shifts), the score is read at bit
//     |q|-1 so no padding/wildcard columns are needed. The per-job match masks Peq[5][NW] live in a
//     per-thread-private, bank-conflict-free slice of shared memory; the target is streamed with
//     aligned LDG.128 + PRMT realignment (ChunkReader).
//   * HW distance without end locations: ed_hw_kernel, the same thread-per-job scheme with the query top-aligned over padding
//     rows (score from the sign bits), and the two probes of a read (jobs 2j, 2j+1 over the same target) in one thread.
//   * |q| > 128: ONE WARP PER JOB, anti-diagonal wavefront: lane l owns a 64-row block and processes
//     column t-l at step t; the horizontal delta (hout) crosses lanes by shuffle. Queries longer
//     than 2048 rows are processed in 2048-row stripes, the stripe's bottom hout per column being
//     parked in a per-warp L2-resident scratch row.
//   * bytes other than ACGTN take an exact slow path (byte equality against the query), so the
//     reference's "equality is byte equality" contract holds for IUPAC / lower case too.
#include "common.cuh"
#include "myers.cuh"
#include <algorithm>
#include <cstdio>

namespace {

constexpr int ED_THREADS = 128;
// job classes: 0 trivial, 1..4 = words per thread-job, 5 = warp-per-job

struct EdArgs {
  const uint8_t* seqs;
  const uint8_t* seqs_end;
  const uint32_t* q_off;
  const uint32_t* q_len;
  const uint32_t* t_off;
  const uint32_t* t_len;
  const int32_t* k;
  uint32_t n;
  int32_t* dist;
  int32_t* end_loc;
  uint32_t* perm;
  uint32_t* counts;  // [0..7] class counts, [8..15] class starts, [16..23] scatter cursors, [24] max t_len of multi-stripe jobs, [32..37] band pass queues,
                     // [41..44], [49..52], [57..60] pair class counts, starts, cursors (ED_PAIR_*)
  int last_pos;      // HW/SHW: report the LAST optimal end position instead of the first (edlib's positionsSHW.back(), src/edlib.cpp:250)
  uint8_t* hbuf;     // per-warp scratch rows for multi-stripe jobs
  uint32_t hbuf_stride;
  // generalised equality (edlib's additionalEqualities, src/edlib.cpp:58-79); all jobs then take the warp-per-job kernel
  const uint32_t* eq_f;  // [256] bitmask of the pairs in which the byte is the first member (null: plain byte equality)
  const uint32_t* eq_s;  // [256] ... the second member
  const uint8_t* eq_cls; // [256] bitmask over {A,C,G,T,N} of the class symbols the byte is equal to
  int force_long;
  uint32_t two;      // = 2, read at run time so that ptxas keeps the multiply forms of ed_hw_kernel's shifts on the FMA pipe
};

__device__ __forceinline__ int ed_class(uint32_t ql, uint32_t tl, int force_long) {
  if (ql == 0 || tl == 0) return 0;
  if (force_long) return 5;
  if (ql <= 128) return (int) ((ql + 31) >> 5);
  return 5;
}

// Apply edlib's k rules to the exact distance. mode: DGPU_MODE_*.
__device__ __forceinline__ int apply_k(int d, int k, int mode, int m, int n) {
  if (k < 0) return d;  // auto-doubling k always finds the exact distance (src/edlib.cpp:192-210)
  if (mode == DGPU_MODE_HW) {
    int kk = min(k, m);  // src/edlib.cpp:563-565
    return d <= kk ? d : -1;
  } else if (mode == DGPU_MODE_SHW) {
    return d <= k ? d : -1;
  } else {
    int diff = n > m ? n - m : m - n;
    if (k < diff) return -1;           // src/edlib.cpp:740-743
    int kk = min(k, max(m, n));        // src/edlib.cpp:745
    return d <= kk ? d : -1;
  }
}

// Pair classes (HW, distance only): jobs 2j and 2j+1 that align two probes against the same read run in one thread, which streams
// and decodes the read once for both (ed_hw_kernel<NW, 2>). counts[ED_PAIR_CNT + c] = pairs of class c (c = NW of the longer probe,
// 1..4), [ED_PAIR_START + c] their start in perm, [ED_PAIR_CUR + c] the scatter cursors; a pair takes one perm entry (its first job).
constexpr int ED_PAIR_CNT = 40, ED_PAIR_START = 48, ED_PAIR_CUR = 56;

// Pair class of job i's pair (0: job i runs alone). Depends only on the job arrays: both jobs of the pair are thread-per-job jobs
// over the same target bytes (equal t_off and t_len), the mode is HW, there are no equality tables and no end locations are wanted.
__device__ __forceinline__ int ed_pair_class(const EdArgs& a, int mode, uint32_t i) {
  if (mode != DGPU_MODE_HW || a.force_long || a.end_loc) return 0;
  const uint32_t j = i & ~1u;
  if (j + 1 >= a.n) return 0;
  const uint32_t q0 = a.q_len[j], q1 = a.q_len[j + 1], t0 = a.t_len[j], t1 = a.t_len[j + 1];
  if (q0 == 0 || q1 == 0 || q0 > 128 || q1 > 128 || t0 == 0 || t0 != t1 || a.t_off[j] != a.t_off[j + 1]) return 0;
  return (int) ((max(q0, q1) + 31) >> 5);
}

__global__ void ed_count_kernel(EdArgs a, int mode) {
  __shared__ uint32_t h[16];   // [0..7] single-job classes, [8 + c] pair classes
  __shared__ uint32_t hmax;
  if (threadIdx.x < 16) h[threadIdx.x] = 0;
  if (threadIdx.x == 0) hmax = 0;
  __syncthreads();
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < a.n) {
    const int pc = ed_pair_class(a, mode, i);
    if (pc) {
      if (!(i & 1u)) atomicAdd(&h[8 + pc], 1u);
    } else {
      uint32_t ql = a.q_len[i], tl = a.t_len[i];
      int c = ed_class(ql, tl, a.force_long);
      atomicAdd(&h[c], 1u);
      if (c == 5 && ql > 2048) atomicMax(&hmax, tl);
      if (c == 0) {
        // src/edlib.cpp:158-177: NW -> max(len), endLocations[0] = n-1; HW/SHW -> |q|, endLocations[0] = -1.
        // (this special case is taken before k is looked at)
        int d = (mode == DGPU_MODE_NW) ? (int) max(ql, tl) : (int) ql;
        a.dist[i] = d;
        if (a.end_loc) a.end_loc[i] = (mode == DGPU_MODE_NW) ? (int) tl - 1 : -1;
      }
    }
  }
  __syncthreads();
  if (threadIdx.x < 8 && h[threadIdx.x]) atomicAdd(&a.counts[threadIdx.x], h[threadIdx.x]);
  if (threadIdx.x >= 9 && threadIdx.x < 13 && h[threadIdx.x]) atomicAdd(&a.counts[ED_PAIR_CNT + threadIdx.x - 8], h[threadIdx.x]);
  if (threadIdx.x == 0 && hmax) atomicMax(&a.counts[24], hmax);
}

__global__ void ed_offsets_kernel(uint32_t* counts) {
  uint32_t s = 0;
  for (int c = 0; c < 8; ++c) {
    counts[8 + c] = s;
    counts[16 + c] = s;
    s += counts[c];
  }
  for (int c = 1; c <= 4; ++c) {
    counts[ED_PAIR_START + c] = s;
    counts[ED_PAIR_CUR + c] = s;
    s += counts[ED_PAIR_CNT + c];
  }
}

__global__ void ed_scatter_kernel(EdArgs a, int mode) {
  __shared__ uint32_t h[16];
  __shared__ uint32_t base[16];
  if (threadIdx.x < 16) h[threadIdx.x] = 0;
  __syncthreads();
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  int c = -1;
  uint32_t r = 0;
  if (i < a.n) {
    const int pc = ed_pair_class(a, mode, i);
    if (!pc) c = ed_class(a.q_len[i], a.t_len[i], a.force_long);
    else if (!(i & 1u)) c = 8 + pc;
    if (c >= 0) r = atomicAdd(&h[c], 1u);
  }
  __syncthreads();
  if (threadIdx.x < 16) {
    const uint32_t cur = threadIdx.x < 8 ? 16 + threadIdx.x : ED_PAIR_CUR + threadIdx.x - 8;
    base[threadIdx.x] = h[threadIdx.x] ? atomicAdd(&a.counts[cur], h[threadIdx.x]) : 0;
  }
  __syncthreads();
  if (c >= 0) a.perm[base[c] + r] = i;
}

// ---- multi-word add with carry ---------------------------------------------------------
template <int NW> struct AddChain;
template <> struct AddChain<1> {
  static __device__ __forceinline__ void run(uint32_t* s, const uint32_t* x, const uint32_t* y) { s[0] = x[0] + y[0]; }
};
template <> struct AddChain<2> {
  static __device__ __forceinline__ void run(uint32_t* s, const uint32_t* x, const uint32_t* y) {
    asm("add.cc.u32 %0, %2, %4;\n\taddc.u32 %1, %3, %5;"
        : "=r"(s[0]), "=r"(s[1]) : "r"(x[0]), "r"(x[1]), "r"(y[0]), "r"(y[1]));
  }
};
template <> struct AddChain<3> {
  static __device__ __forceinline__ void run(uint32_t* s, const uint32_t* x, const uint32_t* y) {
    asm("add.cc.u32 %0, %3, %6;\n\taddc.cc.u32 %1, %4, %7;\n\taddc.u32 %2, %5, %8;"
        : "=r"(s[0]), "=r"(s[1]), "=r"(s[2])
        : "r"(x[0]), "r"(x[1]), "r"(x[2]), "r"(y[0]), "r"(y[1]), "r"(y[2]));
  }
};
template <> struct AddChain<4> {
  static __device__ __forceinline__ void run(uint32_t* s, const uint32_t* x, const uint32_t* y) {
    asm("add.cc.u32 %0, %4, %8;\n\taddc.cc.u32 %1, %5, %9;\n\taddc.cc.u32 %2, %6, %10;\n\taddc.u32 %3, %7, %11;"
        : "=r"(s[0]), "=r"(s[1]), "=r"(s[2]), "=r"(s[3])
        : "r"(x[0]), "r"(x[1]), "r"(x[2]), "r"(x[3]), "r"(y[0]), "r"(y[1]), "r"(y[2]), "r"(y[3]));
  }
};

// One DP column of the single-block Myers recurrence over NW 32-bit words.
// HIN = horizontal delta entering the top row: 0 for HW (free start), +1 for NW/SHW.
template <int NW, int HIN>
__device__ __forceinline__ int myers_column(uint32_t (&Pv)[NW], uint32_t (&Mv)[NW], const uint32_t (&Eq)[NW], uint32_t topbit) {
  uint32_t Xv[NW], t[NW], sum[NW], Ph[NW], Mh[NW];
#pragma unroll
  for (int w = 0; w < NW; ++w) {
    Xv[w] = Eq[w] | Mv[w];
    t[w] = Eq[w] & Pv[w];
  }
  AddChain<NW>::run(sum, t, Pv);
#pragma unroll
  for (int w = 0; w < NW; ++w) {
    uint32_t Xh = (sum[w] ^ Pv[w]) | Eq[w];
    Ph[w] = Mv[w] | ~(Xh | Pv[w]);
    Mh[w] = Pv[w] & Xh;
  }
  int d = (int) ((Ph[NW - 1] >> topbit) & 1u) - (int) ((Mh[NW - 1] >> topbit) & 1u);
#pragma unroll
  for (int w = NW - 1; w >= 0; --w) {
    uint32_t ph = (w == 0) ? ((Ph[0] << 1) | (uint32_t) HIN) : __funnelshift_l(Ph[w - 1], Ph[w], 1);
    uint32_t mh = (w == 0) ? (Mh[0] << 1) : __funnelshift_l(Mh[w - 1], Mh[w], 1);
    Pv[w] = mh | ~(Xv[w] | ph);
    Mv[w] = ph & Xv[w];
  }
  return d;
}

// symbol slot in the shared Peq table: A0 C1 T2 G3 N4 — the order ((c >> 1) & 3) yields for ACGT, so the fast path
// can turn four target bytes into four table offsets with packed arithmetic
__device__ __forceinline__ uint32_t peq_slot(uint32_t code) { return code < 4 ? (code ^ (code >> 1)) : code; }

template <int NW, int MODE, bool WANT_END>
__global__ void __launch_bounds__(ED_THREADS) ed_small_kernel(EdArgs a) {
  __shared__ uint32_t peq[5 * NW * ED_THREADS];
  constexpr int HIN = (MODE == DGPU_MODE_HW) ? 0 : 1;
  const uint32_t cnt = a.counts[NW];
  const uint32_t start = a.counts[8 + NW];
  const uint32_t tid = threadIdx.x;
  for (uint32_t idx = blockIdx.x * ED_THREADS + tid; idx < cnt; idx += gridDim.x * ED_THREADS) {
    const uint32_t job = a.perm[start + idx];
    const uint32_t m = a.q_len[job], n = a.t_len[job];
    const uint8_t* q = a.seqs + a.q_off[job];
    const uint8_t* t = a.seqs + a.t_off[job];

    // ---- build Peq (match masks) for A,C,G,T,N -----------------------------------
    {
      ChunkReader qr;
      qr.init(q, a.seqs_end);
#pragma unroll
      for (int w = 0; w < NW; ++w) {
        uint32_t pm[5] = {0, 0, 0, 0, 0};
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const uint32_t i0 = w * 32 + half * 16;
          if (i0 < m) {
            uint4 v = qr.next();
#pragma unroll
            for (int b = 0; b < 16; ++b) {
              if (i0 + b < m) {
                uint32_t code = dna_code(byte_of(v, b));
                uint32_t bit = 1u << (half * 16 + b);
#pragma unroll
                for (int s = 0; s < 5; ++s) pm[s] |= (code == (uint32_t) s) ? bit : 0u;
              }
            }
          }
        }
#pragma unroll
        for (int s = 0; s < 5; ++s) peq[(peq_slot(s) * NW + w) * ED_THREADS + tid] = pm[s];
      }
    }

    uint32_t Pv[NW], Mv[NW];
#pragma unroll
    for (int w = 0; w < NW; ++w) { Pv[w] = 0xffffffffu; Mv[w] = 0; }
    int score = (int) m;
    // candidate end position -1 (score m) exists iff |q| % 64 != 0 (edlib's padding columns)
    int best = (m & 63u) ? (int) m : 0x7fffffff;
    int bpos = -1;
    const uint32_t topbit = (m - 1) & 31u;

    auto step = [&](uint32_t c, uint32_t col) {
      uint32_t Eq[NW];
      uint32_t code = dna_code(c);
      if (code < 5) {
#pragma unroll
        for (int w = 0; w < NW; ++w) Eq[w] = peq[(peq_slot(code) * NW + w) * ED_THREADS + tid];
      } else {
        // exact slow path: byte equality against the query
#pragma unroll
        for (int w = 0; w < NW; ++w) Eq[w] = 0;
        for (uint32_t i = 0; i < m; ++i) {
          if (__ldg(q + i) == (uint8_t) c) {
#pragma unroll
            for (int w = 0; w < NW; ++w)
              if ((int) (i >> 5) == w) Eq[w] |= 1u << (i & 31);
          }
        }
      }
      score += myers_column<NW, HIN>(Pv, Mv, Eq, topbit);
      if (MODE != DGPU_MODE_NW) {
        if (WANT_END) { if (score < best || (a.last_pos && score == best)) { best = score; bpos = (int) col; } }
        else best = min(best, score);
      }
    };

    ChunkReader tr;
    tr.init(t, a.seqs_end);
    uint32_t c0 = 0;
    const uint32_t base2 = (tid * 4u) * 0x00010001u;  // this thread's slot offset in both 16-bit halves
    for (; c0 + 16 <= n; c0 += 16) {
      uint4 v = tr.next();
      const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int q4 = 0; q4 < 4; ++q4) {
        const uint32_t wd = wv[q4];
        // four bytes at once: x = slot of each byte if it is one of ACGT; `expected` rebuilds the bytes from the slots
        const uint32_t x = (wd >> 1) & 0x03030303u;
        uint32_t sel = x | (x >> 4);
        sel = (sel & 0xffu) | ((sel >> 8) & 0xff00u);
        const uint32_t expected = __byte_perm(0x47544341u, 0u, sel);
        if (wd == expected) {
          // byte offsets of the four Peq rows, two per register: slot * (NW*512) + tid*4
          const uint32_t offA = (x & 0x00ff00ffu) * (uint32_t) (NW * 4 * ED_THREADS) + base2;          // columns 0 and 2
          const uint32_t offB = ((x >> 8) & 0x00ff00ffu) * (uint32_t) (NW * 4 * ED_THREADS) + base2;   // columns 1 and 3
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            const uint32_t pk = (b & 1) ? offB : offA;
            const uint32_t off = (b & 2) ? (pk >> 16) : (pk & 0xffffu);
            uint32_t Eq[NW];
#pragma unroll
            for (int w = 0; w < NW; ++w) Eq[w] = *(const uint32_t*) ((const char*) peq + off + w * 4 * ED_THREADS);
            score += myers_column<NW, HIN>(Pv, Mv, Eq, topbit);
            if (MODE != DGPU_MODE_NW) {
              if (WANT_END) { if (score < best || (a.last_pos && score == best)) { best = score; bpos = (int) (c0 + q4 * 4 + b); } }
              else best = min(best, score);
            }
          }
        } else {
#pragma unroll
          for (int b = 0; b < 4; ++b) step((wd >> (b * 8)) & 0xffu, c0 + q4 * 4 + b);
        }
      }
    }
    if (c0 < n) {
      uint4 v = tr.next();
      uint32_t wv[4] = {v.x, v.y, v.z, v.w};
      for (uint32_t b = 0; c0 + b < n; ++b) {
        uint32_t w = wv[0];
        w = (b >> 2) == 1 ? wv[1] : w;
        w = (b >> 2) == 2 ? wv[2] : w;
        w = (b >> 2) == 3 ? wv[3] : w;
        step((w >> ((b & 3) * 8)) & 0xffu, c0 + b);
      }
    }

    int d, e;
    if (MODE == DGPU_MODE_NW) { d = score; e = (int) n - 1; }
    else { d = best; e = bpos; }
    const int kk = a.k ? a.k[job] : -1;
    d = apply_k(d, kk, MODE, (int) m, (int) n);
    a.dist[job] = d;
    if (a.end_loc) a.end_loc[job] = (d < 0) ? -1 : e;
  }
}

// ---- HW distance: top-aligned query, one or two jobs per thread -----------------------------------------
// The query of m rows sits in the TOP m bits of its NW words: below it are P = 32*NW - m padding rows that match every byte and start
// with vertical delta 0 (Pv = Mv = 0). HW's top border is D[0][j] = 0 for every column, so D of a padding row is min(0 + 0, ...) = 0 in
// every column (induction over rows and columns, all D >= 0): the last padding row is a copy of the border, and the query rows see the
// same free start as without padding. Row m-1 is then bit 31 of the top word and the score delta is the two sign bits, with no shift
// by a per-job amount; and two queries of different lengths in one pair need the same word count only.

// 4-bit mask of the bytes of w equal to the byte splatted in s (bit b = byte b)
__device__ __forceinline__ uint32_t byte_eq_nibble(uint32_t w, uint32_t s) {
  const uint32_t t = w ^ s;
  const uint32_t z = ~(((t & 0x7f7f7f7fu) + 0x7f7f7f7fu) | t | 0x7f7f7f7fu);   // 0x80 in each zero byte, exact per byte
  return (z * 0x00204081u) >> 28;                                               // bit 8b+7 -> bit 28+b, no other product term lands there
}

// word w of a mask of the low P bits (the padding rows, for P padding rows)
__device__ __forceinline__ uint32_t pad_word(uint32_t P, int w) {
  const uint32_t lo = 32u * (uint32_t) w;
  return P >= lo + 32 ? 0xffffffffu : P <= lo ? 0u : (1u << (P - lo)) - 1u;
}

// Top-aligned match masks of the query q (m rows, 1 <= m <= 32*NW) for the slots A0 C1 T2 G3 N4, padding rows set in all of them.
template <int NW>
__device__ __forceinline__ void build_peq_top(const uint8_t* q, uint32_t m, const uint8_t* seqs_end, uint32_t (&pm)[5][NW]) {
  uint32_t raw[5][NW];
#pragma unroll
  for (int s = 0; s < 5; ++s)
#pragma unroll
    for (int w = 0; w < NW; ++w) raw[s][w] = 0;
  ChunkReader qr;
  qr.init(q, seqs_end);
#pragma unroll
  for (int w = 0; w < NW; ++w) {
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      if ((uint32_t) (w * 32 + half * 16) < m) {
        const uint4 v = qr.next();
        const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int sh = half * 16 + k * 4;
          raw[0][w] |= byte_eq_nibble(wv[k], 0x41414141u) << sh;   // A
          raw[1][w] |= byte_eq_nibble(wv[k], 0x43434343u) << sh;   // C
          raw[2][w] |= byte_eq_nibble(wv[k], 0x54545454u) << sh;   // T
          raw[3][w] |= byte_eq_nibble(wv[k], 0x47474747u) << sh;   // G
          raw[4][w] |= byte_eq_nibble(wv[k], 0x4e4e4e4eu) << sh;   // N
        }
      }
    }
  }
  // keep rows < m, then shift up by P = 32*NW - m rows: first by P % 32 bits, then by P / 32 words
  const uint32_t P = 32u * NW - m, bs = P & 31u, ws = P >> 5;
#pragma unroll
  for (int s = 0; s < 5; ++s) {
    uint32_t b[NW];
#pragma unroll
    for (int w = 0; w < NW; ++w) raw[s][w] &= pad_word(m, w);   // rows < m (pad_word(m, w) = the low m bits of the words)
#pragma unroll
    for (int w = 0; w < NW; ++w) b[w] = (w == 0) ? (raw[s][0] << bs) : __funnelshift_l(raw[s][w - 1], raw[s][w], bs);
#pragma unroll
    for (int w = 0; w < NW; ++w) {
      uint32_t o = 0;
#pragma unroll
      for (int d = 0; d <= w; ++d) o = (ws == (uint32_t) d) ? b[w - d] : o;
      pm[s][w] = o | pad_word(P, w);
    }
  }
}

// One DP column over NW top-aligned words, HW (no horizontal delta enters the top): adds the delta of row m-1, read from the sign
// bits, to score.
template <int NW>
__device__ __forceinline__ void myers_column_top(uint32_t (&Pv)[NW], uint32_t (&Mv)[NW], const uint32_t (&Eq)[NW], int& score, uint32_t two) {
  uint32_t Xv[NW], t[NW], sum[NW], Ph[NW], Mh[NW];
#pragma unroll
  for (int w = 0; w < NW; ++w) {
    Xv[w] = Eq[w] | Mv[w];
    t[w] = Eq[w] & Pv[w];
  }
  AddChain<NW>::run(sum, t, Pv);
#pragma unroll
  for (int w = 0; w < NW; ++w) {
    uint32_t Xh = (sum[w] ^ Pv[w]) | Eq[w];
    Ph[w] = Mv[w] | ~(Xh | Pv[w]);
    Mh[w] = Pv[w] & Xh;
  }
  // Written as multiply-highs and multiply-adds so that ptxas can issue them on the FMA pipe (the ALU pipe carries the LOP3s):
  // score += sign bit of Ph (unsigned high word of Ph * 2) and -(sign bit of Mh) (signed high word of Mh * 2);
  // the one-row shift of word w >= 1 is Ph[w] * 2 + the top bit of Ph[w-1] (bits that do not overlap, so + is |).
  score = __umulhi(Ph[NW - 1], two) + score;
  score = __mulhi((int) Mh[NW - 1], (int) two) + score;
#pragma unroll
  for (int w = NW - 1; w >= 0; --w) {
    const uint32_t ph = (w == 0) ? (Ph[0] * two) : (Ph[w] * two + __umulhi(Ph[w - 1], two));
    const uint32_t mh = (w == 0) ? (Mh[0] * two) : (Mh[w] * two + __umulhi(Mh[w - 1], two));
    Pv[w] = mh | ~(Xv[w] | ph);
    Mv[w] = ph & Xv[w];
  }
}

// J = 1: the HW distance-only single-job class NW (counts[NW]); J = 2: the pair class NW (counts[ED_PAIR_CNT + NW]). Shared Peq:
// entry ((slot * NW + w) * ED_THREADS + tid) holds J words, one per job, so a pair reads both of its jobs' words with one LDS.64.
template <int NW, int J>
__global__ void __launch_bounds__(ED_THREADS, J == 1 ? 8 : NW == 4 ? 5 : 6) ed_hw_kernel(EdArgs a) {
  __shared__ uint32_t peq[5 * NW * J * ED_THREADS];
  const uint32_t cnt = (J == 2) ? a.counts[ED_PAIR_CNT + NW] : a.counts[NW];
  const uint32_t start = (J == 2) ? a.counts[ED_PAIR_START + NW] : a.counts[8 + NW];
  const uint32_t tid = threadIdx.x;
  char* const peqb = (char*) peq;
  for (uint32_t idx = blockIdx.x * ED_THREADS + tid; idx < cnt; idx += gridDim.x * ED_THREADS) {
    const uint32_t job0 = a.perm[start + idx];
    const uint32_t n = a.t_len[job0];
    const uint8_t* t = a.seqs + a.t_off[job0];
    uint32_t m[J];
    const uint8_t* q[J];
#pragma unroll
    for (int j = 0; j < J; ++j) { m[j] = a.q_len[job0 + j]; q[j] = a.seqs + a.q_off[job0 + j]; }

#pragma unroll
    for (int j = 0; j < J; ++j) {
      uint32_t pm[5][NW];
      build_peq_top<NW>(q[j], m[j], a.seqs_end, pm);
#pragma unroll
      for (int s = 0; s < 5; ++s)
#pragma unroll
        for (int w = 0; w < NW; ++w) peq[((s * NW + w) * ED_THREADS + tid) * J + j] = pm[s][w];
    }

    uint32_t Pv[J][NW], Mv[J][NW];
    int score[J], best[J];
#pragma unroll
    for (int j = 0; j < J; ++j) {
#pragma unroll
      for (int w = 0; w < NW; ++w) { Pv[j][w] = ~pad_word(32u * NW - m[j], w); Mv[j][w] = 0; }
      score[j] = (int) m[j];
      best[j] = (m[j] & 63u) ? (int) m[j] : 0x7fffffff;   // candidate end position -1 exists iff |q| % 64 != 0
    }

    auto column = [&](const uint32_t (&Eq)[J][NW]) {
#pragma unroll
      for (int j = 0; j < J; ++j) {
        myers_column_top<NW>(Pv[j], Mv[j], Eq[j], score[j], a.two);
        best[j] = min(best[j], score[j]);
      }
    };
    auto load_eq = [&](uint32_t off, uint32_t (&Eq)[J][NW]) {
#pragma unroll
      for (int w = 0; w < NW; ++w) {
        const char* p = peqb + off + w * 4 * J * ED_THREADS;
        if (J == 2) { const uint2 e = *(const uint2*) p; Eq[0][w] = e.x; Eq[J - 1][w] = e.y; }
        else Eq[0][w] = *(const uint32_t*) p;
      }
    };
    // one column whose byte is not A, C, G or T
    auto step = [&](uint32_t c) {
      uint32_t Eq[J][NW];
      const uint32_t code = dna_code(c);
      if (code < 5) {
        load_eq((peq_slot(code) * NW * ED_THREADS + tid) * 4 * J, Eq);
      } else {
        // exact slow path: byte equality against the query, padding rows match everything
#pragma unroll
        for (int j = 0; j < J; ++j) {
          const uint32_t P = 32u * NW - m[j];
#pragma unroll
          for (int w = 0; w < NW; ++w) Eq[j][w] = pad_word(P, w);
          for (uint32_t i = 0; i < m[j]; ++i) {
            if (__ldg(q[j] + i) == (uint8_t) c) {
              const uint32_t r = P + i;
#pragma unroll
              for (int w = 0; w < NW; ++w)
                if ((r >> 5) == (uint32_t) w) Eq[j][w] |= 1u << (r & 31);
            }
          }
        }
      }
      column(Eq);
    };
    const uint32_t base2 = (tid * 4u * J) * 0x00010001u;  // this thread's entry offset in both 16-bit halves
    // four target columns (bytes of wd), the first ncols of them inside the target
    auto group = [&](uint32_t wd, uint32_t ncols) {
      // four bytes at once: x = slot of each byte if it is one of ACGT; `expected` rebuilds the bytes from the slots
      const uint32_t x = (wd >> 1) & 0x03030303u;
      uint32_t sel = x | (x >> 4);
      sel = (sel & 0xffu) | ((sel >> 8) & 0xff00u);
      const uint32_t expected = __byte_perm(0x47544341u, 0u, sel);
      const uint32_t live = ncols >= 4 ? 0xffffffffu : (1u << (ncols * 8)) - 1u;
      if (((wd ^ expected) & live) == 0) {
        // byte offsets of the four Peq entries, two per register: slot * (NW*J*512) + tid*4*J
        const uint32_t offA = (x & 0x00ff00ffu) * (uint32_t) (NW * 4 * J * ED_THREADS) + base2;          // columns 0 and 2
        const uint32_t offB = ((x >> 8) & 0x00ff00ffu) * (uint32_t) (NW * 4 * J * ED_THREADS) + base2;   // columns 1 and 3
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          if ((uint32_t) b < ncols) {
            const uint32_t pk = (b & 1) ? offB : offA;
            uint32_t Eq[J][NW];
            load_eq((b & 2) ? (pk >> 16) : (pk & 0xffffu), Eq);
            column(Eq);
          }
        }
      } else {
#pragma unroll
        for (int b = 0; b < 4; ++b)
          if ((uint32_t) b < ncols) step((wd >> (b * 8)) & 0xffu);
      }
    };

    ChunkReader tr;
    tr.init(t, a.seqs_end);
    uint32_t c0 = 0;
    for (; c0 + 16 <= n; c0 += 16) {
      const uint4 v = tr.next();
      group(v.x, 4); group(v.y, 4); group(v.z, 4); group(v.w, 4);
    }
    if (c0 < n) {
      // the last partial chunk through the same path, columns past the target masked
      const uint4 v = tr.next();
      const uint32_t rem = n - c0;
      group(v.x, min(rem, 4u));
      if (rem > 4) group(v.y, min(rem - 4, 4u));
      if (rem > 8) group(v.z, min(rem - 8, 4u));
      if (rem > 12) group(v.w, rem - 12);
    }

#pragma unroll
    for (int j = 0; j < J; ++j) {
      const int kk = a.k ? a.k[job0 + j] : -1;
      a.dist[job0 + j] = apply_k(best[j], kk, DGPU_MODE_HW, (int) m[j], (int) n);
    }
  }
}

// ---- warp-per-job wavefront for |q| > 128 -------------------------------------------
constexpr int EDL_WARPS = 4;  // warps per CTA in the long kernel

template <int MODE, bool EQ>
__global__ void __launch_bounds__(EDL_WARPS * 32) ed_long_kernel(EdArgs a, const uint32_t* list, const uint32_t* list_cnt) {
  __shared__ uint64_t peq_s[EDL_WARPS][5][32];
  constexpr int HIN0 = (MODE == DGPU_MODE_HW) ? 0 : 1;
  // job list: the class-5 segment of perm, or (NW with band passes in front) what the band passes left over
  const uint32_t cnt = list ? *list_cnt : a.counts[5];
  if (!list) list = a.perm + a.counts[8 + 5];
  const int lane = threadIdx.x & 31;
  const int wib = threadIdx.x >> 5;
  const uint32_t gwarp = blockIdx.x * EDL_WARPS + wib;
  const uint32_t nwarps = gridDim.x * EDL_WARPS;
  volatile uint8_t* hrow = a.hbuf ? a.hbuf + (size_t) gwarp * a.hbuf_stride : nullptr;

  for (uint32_t idx = gwarp; idx < cnt; idx += nwarps) {
    const uint32_t job = list[idx];
    const uint32_t m = a.q_len[job], n = a.t_len[job];
    const uint8_t* q = a.seqs + a.q_off[job];
    const uint8_t* t = a.seqs + a.t_off[job];
    const uint32_t nstripes = (m + 2047) / 2048;
    int score = (int) m;  // D[m][0]; only meaningful on the lane that owns row m-1
    int best = (m & 63u) ? (int) m : 0x7fffffff, bpos = -1;  // end position -1 exists iff |q| % 64 != 0

    for (uint32_t s = 0; s < nstripes; ++s) {
      const uint32_t row0 = s * 2048 + (uint32_t) lane * 64;  // first query row of this lane's block
      const uint32_t rows_left = m - s * 2048;
      const int nb = (int) min(32u, (rows_left + 63) / 64);   // active lanes in this stripe
      const bool last_stripe = (s + 1 == nstripes);
      const bool active = lane < nb;
      const int topbit = (int) ((m - 1) & 63u);

      // Peq for this lane's 64 rows
      uint64_t pm_other = 0;  // EQ: rows holding a byte outside ACGTN (compared exactly, pair tables included)
      {
        uint64_t pm[5] = {0, 0, 0, 0, 0};
        pm_other = 0;
        if (active) {
          for (uint32_t i = 0; i < 64 && row0 + i < m; ++i) {
            uint32_t code = dna_code(__ldg(q + row0 + i));
#pragma unroll
            for (int sy = 0; sy < 5; ++sy) pm[sy] |= (code == (uint32_t) sy) ? (1ull << i) : 0ull;
            if (EQ && code == 5u) pm_other |= 1ull << i;
          }
        }
        __syncwarp();
#pragma unroll
        for (int sy = 0; sy < 5; ++sy) peq_s[wib][sy][lane] = pm[sy];
        __syncwarp();
      }

      uint64_t Pv = ~0ull, Mv = 0;
      int hout = 0;
      uint32_t cbuf = 0;   // 32 target bytes, one per lane, refreshed every 32 steps
      uint32_t cchar = 0;  // this lane's current column byte
      const uint32_t nsteps = n + (uint32_t) nb - 1;
      for (uint32_t st = 0; st < nsteps; ++st) {
        if ((st & 31u) == 0) {
          uint32_t p = st + (uint32_t) lane;
          cbuf = (p < n) ? (uint32_t) __ldg(t + p) : 0u;
        }
        uint32_t newc = __shfl_sync(0xffffffffu, cbuf, (int) (st & 31u));
        uint32_t upc = __shfl_up_sync(0xffffffffu, cchar, 1);
        cchar = (lane == 0) ? newc : upc;
        int hin_sh = __shfl_up_sync(0xffffffffu, hout, 1);
        const int col = (int) st - lane;
        if (active && col >= 0 && col < (int) n) {
          int hin;
          if (lane == 0) hin = (s == 0) ? HIN0 : (int) (int8_t) hrow[col];
          else hin = hin_sh;
          uint32_t code = dna_code(cchar);
          uint64_t Eq;
          if (EQ) {
            const uint32_t cm = a.eq_cls[cchar & 0xffu];
            Eq = 0;
#pragma unroll
            for (int sy = 0; sy < 5; ++sy)
              if ((cm >> sy) & 1u) Eq |= peq_s[wib][sy][lane];
            uint64_t rest = pm_other;
            const uint32_t cf = a.eq_f[cchar & 0xffu], cs = a.eq_s[cchar & 0xffu];
            while (rest) {
              const int i = __ffsll((long long) rest) - 1;
              rest &= rest - 1;
              const uint32_t qb = __ldg(q + row0 + i);
              if (qb == (cchar & 0xffu) || (a.eq_f[qb] & cs) || (a.eq_s[qb] & cf)) Eq |= 1ull << i;
            }
          } else if (code < 5) Eq = peq_s[wib][code][lane];
          else {
            Eq = 0;
            for (uint32_t i = 0; i < 64 && row0 + i < m; ++i)
              if (__ldg(q + row0 + i) == (uint8_t) cchar) Eq |= 1ull << i;
          }
          uint64_t Ph, Mh;
          hout = block64(Pv, Mv, Eq, hin, Ph, Mh);
          if (lane == nb - 1 && last_stripe) {
            // delta of row m-1 (inside this block)
            score += (int) ((Ph >> topbit) & 1ull) - (int) ((Mh >> topbit) & 1ull);
            if (MODE != DGPU_MODE_NW) {
              if (score < best || (a.last_pos && score == best)) { best = score; bpos = col; }
            }
          }
          if (lane == nb - 1 && !last_stripe) hrow[col] = (uint8_t) (int8_t) hout;
        }
      }
      __syncwarp();
      __threadfence_block();
    }
    // broadcast the result from the lane that owns row m-1
    const int owner = (int) (((m - 1) & 2047u) >> 6);
    int d = (MODE == DGPU_MODE_NW) ? score : best;
    int e = (MODE == DGPU_MODE_NW) ? (int) n - 1 : bpos;
    d = __shfl_sync(0xffffffffu, d, owner);
    e = __shfl_sync(0xffffffffu, e, owner);
    if (lane == 0) {
      const int kk = a.k ? a.k[job] : -1;
      d = apply_k(d, kk, MODE, (int) m, (int) n);
      a.dist[job] = d;
      if (a.end_loc) a.end_loc[job] = (d < 0) ? -1 : e;
    }
  }
}

// ---- banded passes for long NW jobs (Ukkonen band, src/edlib.cpp:728-929 computes the same cells block-wise) ------------------------
// The reference computes, for a threshold k, only the blocks that intersect the diagonals a path of cost <= k can touch, and doubles
// k (from 64) until the result is <= k (src/edlib.cpp:192-210). The device form of the same idea:
//   * a band pass of class G gives a job to G lanes (32/G jobs per warp). The band is a STAIRCASE of G 64-row blocks: during the 64
//     target columns of chunk J lane p holds block J - A + p (A = blocks above the diagonal, chosen per job from |t| - |q|); lanes
//     are skewed by one step so that a block's horizontal delta reaches the block below by shuffle; after the chunk every lane takes
//     over the block of the lane below (Pv, Mv and the absolute score of the block's last row travel through shared memory), the
//     last lane opens a new block with Pv = 1..1 (the cells left of it are outside the band: +1 per row is an upper bound).
//   * the pass covers every diagonal in [-64(G-1-A), 64A] at every column, so its result s is the exact distance whenever
//     s <= kvalid = 2 * min(64A - max(0,d), 64(G-1-A) - max(0,-d)) + |d|, d = |t| - |q| (Ukkonen's argument), or when the
//     staircase covers the whole matrix. Otherwise the job goes to the next class (band twice as wide), finally to ed_long_kernel.
//   * the first class of a job comes from a cheap upper bound (mismatches on the main diagonal + |d|, ed_band_plan_kernel): when it
//     fits a class that class is certain to succeed; otherwise classes are tried from kvalid >= 64 upwards like the reference does.
// counts[32 + c] = jobs queued for band class c (c < EDB_CLASSES), counts[32 + EDB_CLASSES] = jobs left to ed_long_kernel
__device__ __forceinline__ void band_queue(const EdArgs& a, uint32_t* lists, uint32_t cap, int c, uint32_t job) {
  lists[(size_t) c * cap + atomicAdd(&a.counts[32 + c], 1u)] = job;
}

// first class, from c0 on, that can hold the job and (need >= 0) certifies distances up to `need`, or covers the whole matrix
__device__ __forceinline__ int band_first_class(int c0, int m, int n, int need) {
  const int nblk = (m + 63) >> 6;
  for (int c = c0; c < EDB_CLASSES; ++c) {
    if (nblk > edb_block_cap(c)) continue;
    const BandPlan b = band_plan(edb_lanes(c), m, n);
    if (b.whole || b.kvalid >= need) return c;
  }
  return EDB_CLASSES;
}

__global__ void __launch_bounds__(256) ed_band_plan_kernel(EdArgs a, uint32_t* lists, uint32_t cap) {
  const uint32_t cnt = a.counts[5], start = a.counts[8 + 5];
  const int lane = threadIdx.x & 31;
  const uint32_t gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t idx = gwarp; idx < cnt; idx += nwarps) {
    const uint32_t job = a.perm[start + idx];
    const int m = (int) a.q_len[job], n = (int) a.t_len[job];
    const uint8_t* q = a.seqs + a.q_off[job];
    const uint8_t* t = a.seqs + a.t_off[job];
    const int d = n > m ? n - m : m - n;
    int kk = a.k ? a.k[job] : -1;
    if (kk >= 0 && kk < d) {                      // src/edlib.cpp:740-743
      if (lane == 0) { a.dist[job] = -1; if (a.end_loc) a.end_loc[job] = -1; }
      continue;
    }
    const int len = min(m, n);
    int mis = 0;
    for (int i = lane; i < len; i += 32) mis += __ldg(q + i) != __ldg(t + i);
    for (int o = 16; o; o >>= 1) mis += __shfl_xor_sync(0xffffffffu, mis, o);
    int need = mis + d;                           // cost of the gap-free alignment + end gap: an upper bound of the distance
    if (kk >= 0) need = min(need, min(kk, max(m, n)));   // beyond the caller's k the answer is -1 whatever the distance is
    if (lane == 0) {
      int c = band_first_class(0, m, n, need);
      if (c == EDB_CLASSES) c = band_first_class(0, m, n, 64);   // no class certifies the bound: widen step by step like the reference
      band_queue(a, lists, cap, c, job);
    }
  }
}

template <int G, bool EQ>
__global__ void __launch_bounds__(EDB_WARPS * 32) ed_band_kernel(EdArgs a, uint32_t* lists, uint32_t cap) {
  constexpr int CLS = (G == 2) ? 0 : (G == 4) ? 1 : (G == 8) ? 2 : (G == 16) ? 3 : 4;
  constexpr int JPW = 32 / G;                      // jobs per warp
  constexpr int PEQ_JOB = EDB_PEQ_WORDS / JPW;     // Peq words per job
  __shared__ uint64_t peq_s[EDB_WARPS][EDB_PEQ_WORDS];
  __shared__ uint64_t hoP[EDB_WARPS][32], hoM[EDB_WARPS][32];
  __shared__ int hoS[EDB_WARPS][32];
  const uint32_t cnt = a.counts[32 + CLS];
  const uint32_t* list = lists + (size_t) CLS * cap;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int p = lane & (G - 1), grp = lane / G;
  const uint32_t gwarp = blockIdx.x * EDB_WARPS + wib, nwarps = gridDim.x * EDB_WARPS;
  uint64_t* peq = &peq_s[wib][grp * PEQ_JOB];
  const EqTabs tabs = {a.eq_f, a.eq_s, a.eq_cls};

  for (uint32_t base = gwarp * JPW; base < cnt; base += nwarps * JPW) {
    const bool have = base + grp < cnt;
    const uint32_t job = have ? list[base + grp] : 0;
    const int m = have ? (int) a.q_len[job] : 0, n = have ? (int) a.t_len[job] : 0;
    const uint8_t* q = a.seqs + (have ? a.q_off[job] : 0);
    const uint8_t* t = a.seqs + (have ? a.t_off[job] : 0);
    const int nblk = (m + 63) >> 6;
    const BandPlan bp = band_plan(G, max(m, 1), max(n, 1));

    __syncwarp();
    band_build_peq<G>(peq, q, m, false, p);
    __syncwarp();

    const int Jend = (n - 1) >> 6;
    int steps = have ? 65 * Jend + ((n - 1) & 63) + G : 0;
    for (int o = 16; o; o >>= 1) steps = max(steps, __shfl_xor_sync(0xffffffffu, steps, o));

    uint64_t Pv = ~0ull, Mv = 0;
    int blk = p - bp.A, J = 0, c = -p;             // c < 0: waiting for the skew; 0..63: column 64J + c; 64: hand-over slot
    int sc = 64 * (blk + 1);                        // D[last row of the block][column before the current one]
    int hout = 1;
    uint32_t chn = (have && n > 0) ? __ldg(t) : 0u;
    for (int st = 0; st < steps; ++st) {
      const int hin_sh = __shfl_up_sync(0xffffffffu, hout, 1, G);
      if (c >= 0 && c < 64) {
        const int col = (J << 6) + c;
        if (col < n) {
          const uint32_t ch = chn;
          if (col + 1 < n) chn = __ldg(t + col + 1);
          if (blk >= 0 && blk < nblk) {
            const uint64_t Eq = band_eq<EQ>(peq, blk, ch, q, m, false, tabs);
            const int hin = (p == 0 || blk == 0) ? 1 : hin_sh;   // above: the matrix border or a cell outside the band
            uint64_t Ph, Mh;
            hout = block64(Pv, Mv, Eq, hin, Ph, Mh);
            sc += hout;
          }
        }
      }
      const bool give = (c == 63), take = (c == 64) && (((J + 1) << 6) < n);
      if (__any_sync(0xffffffffu, give || take)) {
        if (give) { hoP[wib][lane] = Pv; hoM[wib][lane] = Mv; hoS[wib][lane] = sc; }
        __syncwarp();
        if (take) {
          if (p < G - 1) { Pv = hoP[wib][lane + 1]; Mv = hoM[wib][lane + 1]; sc = hoS[wib][lane + 1]; }
          else { Pv = ~0ull; Mv = 0; sc += 64; }
          ++blk; ++J; c = -1;
        }
        __syncwarp();
      }
      ++c;
    }

    // D[m][n]: the block holding row m-1, corrected by the vertical deltas of the rows below it inside the block
    const int tb = (m - 1) & 63;
    const uint64_t below = tb == 63 ? 0ull : (~0ull << (tb + 1));
    int s = sc - __popcll(Pv & below) + __popcll(Mv & below);
    const int plast = (nblk - 1) - (Jend - bp.A);
    s = __shfl_sync(0xffffffffu, s, (grp * G) + (plast & (G - 1)));
    if (have && p == 0) {
      const int kk = a.k ? a.k[job] : -1;
      if (plast >= 0 && plast < G && (bp.whole || s <= bp.kvalid)) {
        const int dd = apply_k(s, kk, DGPU_MODE_NW, m, n);
        a.dist[job] = dd;
        if (a.end_loc) a.end_loc[job] = dd < 0 ? -1 : n - 1;
      } else if (kk >= 0 && min(kk, max(m, n)) <= bp.kvalid) {
        a.dist[job] = -1;                          // every path of cost <= k lies inside the band, and the band found none
        if (a.end_loc) a.end_loc[job] = -1;
      } else {
        band_queue(a, lists, cap, band_first_class(CLS + 1, m, n, bp.kvalid + 1), job);
      }
    }
  }
}

// ---- pipelined host-pointer call: arena prefix needed by each job index range ----------------------------------
constexpr int ED_PIPE_MAX_CHUNKS = 16;          // job index ranges per call
constexpr uint64_t ED_PIPE_MIN_JOBS = 1u << 18; // smallest range worth a separate launch
constexpr int ED_PIPE_PIECES = 32;              // arena upload pieces

__global__ void ed_extent_kernel(const uint32_t* __restrict__ q_off, const uint32_t* __restrict__ q_len,
                                 const uint32_t* __restrict__ t_off, const uint32_t* __restrict__ t_len,
                                 uint32_t n, uint32_t jobs_per, uint32_t arena_bytes, uint32_t* __restrict__ ext) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t e = 0, c = 0;
  if (i < n) {
    const uint64_t a = (uint64_t) q_off[i] + q_len[i], b = (uint64_t) t_off[i] + t_len[i];
    const uint64_t m = a > b ? a : b;
    if (m > arena_bytes) ext[ED_PIPE_MAX_CHUNKS] = 1;   // a sequence outside the caller's arena: the call is refused before any kernel reads it
    e = (uint32_t) (m < arena_bytes ? m : arena_bytes);
    c = i / jobs_per;
  }
  // a block of 256 consecutive jobs spans at most two ranges: reduce per warp when the warp is uniform
  const uint32_t c0 = __shfl_sync(0xffffffffu, c, 0);
  if (__all_sync(0xffffffffu, c == c0 || i >= n)) {
    for (int o = 16; o; o >>= 1) e = max(e, __shfl_xor_sync(0xffffffffu, e, o));
    if ((threadIdx.x & 31) == 0 && e) atomicMax(&ext[c0], e);
  } else if (i < n && e) atomicMax(&ext[c], e);
}

int dgpu_pipe_init(dgpu_ctx* ctx) {
  if (!ctx->copy_stream) DGPU_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  if (!ctx->out_stream) DGPU_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->out_stream, cudaStreamNonBlocking));
  const size_t want = 1 + ED_PIPE_PIECES + ED_PIPE_MAX_CHUNKS;
  while (ctx->pipe_events.size() < want) {
    cudaEvent_t e;
    DGPU_CUDA(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    ctx->pipe_events.push_back(e);
  }
  return DGPU_OK;
}

template <int MODE>
int launch_mode(dgpu_ctx* ctx, EdArgs& a, const uint32_t* hc, cudaStream_t st) {
  const int sms = ctx->num_sms;
  auto grid_for = [&](uint32_t cnt, int per_block, int max_per_sm) {
    uint32_t need = (cnt + per_block - 1) / per_block;
    uint32_t cap = (uint32_t) (sms * max_per_sm);
    return need < cap ? need : cap;
  };
  dgpu_prof_begin(ctx, st);
  const bool want_end = (a.end_loc != nullptr);
  // HW distance without end locations: the top-aligned kernel (single jobs and pairs); everything else: ed_small_kernel
#define ED_LAUNCH_SMALL(NWV)                                                                                              \
  if (hc[NWV]) {                                                                                                          \
    if (want_end) ed_small_kernel<NWV, MODE, true><<<grid_for(hc[NWV], ED_THREADS, 16), ED_THREADS, 0, st>>>(a);          \
    else if constexpr (MODE == DGPU_MODE_HW) ed_hw_kernel<NWV, 1><<<grid_for(hc[NWV], ED_THREADS, 16), ED_THREADS, 0, st>>>(a);     \
    else ed_small_kernel<NWV, MODE, false><<<grid_for(hc[NWV], ED_THREADS, 16), ED_THREADS, 0, st>>>(a);                  \
    DGPU_LAUNCH_CHECK(ctx, "ed_small");                                                                                   \
  }                                                                                                                       \
  if (hc[ED_PAIR_CNT + NWV]) {                                                                                            \
    ed_hw_kernel<NWV, 2><<<grid_for(hc[ED_PAIR_CNT + NWV], ED_THREADS, 16), ED_THREADS, 0, st>>>(a);                      \
    DGPU_LAUNCH_CHECK(ctx, "ed_pair");                                                                                    \
  }
  ED_LAUNCH_SMALL(1)
  ED_LAUNCH_SMALL(2)
  ED_LAUNCH_SMALL(3)
  ED_LAUNCH_SMALL(4)
#undef ED_LAUNCH_SMALL
  if (hc[5]) {
    uint32_t g = grid_for(hc[5], EDL_WARPS, 8);
    a.hbuf = nullptr;
    a.hbuf_stride = 0;
    if (hc[24]) {
      a.hbuf_stride = (hc[24] + 255u) & ~255u;
      void* hb;
      int rc = dgpu_reserve(ctx, SLOT_WORK0, (size_t) g * EDL_WARPS * a.hbuf_stride, &hb);
      if (rc) return rc;
      a.hbuf = (uint8_t*) hb;
    }
    if (MODE == DGPU_MODE_NW && !ctx->no_band) {
      // band passes first (narrowest class first: a pass queues what it could not certify for the next one), the full matrix last
      const uint32_t cap = hc[5];
      void* lp;
      int rc = dgpu_reserve(ctx, SLOT_EDBAND, (size_t) (EDB_CLASSES + 1) * cap * sizeof(uint32_t), &lp);
      if (rc) return rc;
      uint32_t* lists = (uint32_t*) lp;
      ed_band_plan_kernel<<<grid_for(hc[5], 8, 8), 256, 0, st>>>(a, lists, cap);
      DGPU_LAUNCH_CHECK(ctx, "ed_band_plan");
#define ED_LAUNCH_BAND(GV)                                                                                                    \
      if (a.eq_cls) ed_band_kernel<GV, true><<<grid_for(hc[5], EDB_WARPS * (32 / GV), 5), EDB_WARPS * 32, 0, st>>>(a, lists, cap);  \
      else ed_band_kernel<GV, false><<<grid_for(hc[5], EDB_WARPS * (32 / GV), 5), EDB_WARPS * 32, 0, st>>>(a, lists, cap);         \
      DGPU_LAUNCH_CHECK(ctx, "ed_band");
      ED_LAUNCH_BAND(2)
      ED_LAUNCH_BAND(4)
      ED_LAUNCH_BAND(8)
      ED_LAUNCH_BAND(16)
      ED_LAUNCH_BAND(32)
#undef ED_LAUNCH_BAND
      if (a.eq_cls) ed_long_kernel<MODE, true><<<g, EDL_WARPS * 32, 0, st>>>(a, lists + (size_t) EDB_CLASSES * cap, a.counts + 32 + EDB_CLASSES);
      else ed_long_kernel<MODE, false><<<g, EDL_WARPS * 32, 0, st>>>(a, lists + (size_t) EDB_CLASSES * cap, a.counts + 32 + EDB_CLASSES);
      DGPU_LAUNCH_CHECK(ctx, "ed_long");
    } else if (a.eq_cls) {
      ed_long_kernel<MODE, true><<<g, EDL_WARPS * 32, 0, st>>>(a, nullptr, nullptr);
      DGPU_LAUNCH_CHECK(ctx, "ed_long");
    } else {
      ed_long_kernel<MODE, false><<<g, EDL_WARPS * 32, 0, st>>>(a, nullptr, nullptr);
      DGPU_LAUNCH_CHECK(ctx, "ed_long");
    }
  }
  dgpu_prof_end(ctx, st);
  return DGPU_OK;
}

}  // namespace

// Internal entry shared with edit_path.cu: last_pos selects the last optimal end position.
int dgpu_edit_distance_impl(dgpu_ctx* ctx, const uint8_t* seqs, uint64_t seqs_bytes,
                            const uint32_t* q_off, const uint32_t* q_len,
                            const uint32_t* t_off, const uint32_t* t_len,
                            const int32_t* k, int mode, uint64_t n,
                            int32_t* dist, int32_t* end_loc, void* stream, int last_pos, const uint32_t* eq_tabs);

extern "C" {

int dgpu_edit_distance_dev(dgpu_ctx* ctx, const uint8_t* seqs, uint64_t seqs_bytes,
                           const uint32_t* q_off, const uint32_t* q_len,
                           const uint32_t* t_off, const uint32_t* t_len,
                           const int32_t* k, int mode, uint64_t n,
                           int32_t* dist, int32_t* end_loc, void* stream) {
  return dgpu_edit_distance_impl(ctx, seqs, seqs_bytes, q_off, q_len, t_off, t_len, k, mode, n, dist, end_loc, stream, 0, nullptr);
}

}  // extern "C"

int dgpu_edit_distance_impl(dgpu_ctx* ctx, const uint8_t* seqs, uint64_t seqs_bytes,
                            const uint32_t* q_off, const uint32_t* q_len,
                            const uint32_t* t_off, const uint32_t* t_len,
                            const int32_t* k, int mode, uint64_t n,
                            int32_t* dist, int32_t* end_loc, void* stream, int last_pos, const uint32_t* eq_tabs) {
  if (!ctx) return DGPU_ERR_ARG;
  if (mode != DGPU_MODE_NW && mode != DGPU_MODE_SHW && mode != DGPU_MODE_HW) return DGPU_ERR_ARG;
  if (n == 0) return DGPU_OK;
  if (n >= (1ull << 31) || seqs_bytes >= (1ull << 32)) return DGPU_ERR_ARG;
  if (!seqs || !q_off || !q_len || !t_off || !t_len || !dist) return DGPU_ERR_ARG;
  DGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = stream ? (cudaStream_t) stream : ctx->stream;

  EdArgs a;
  a.seqs = seqs; a.seqs_end = seqs + seqs_bytes;
  a.q_off = q_off; a.q_len = q_len; a.t_off = t_off; a.t_len = t_len; a.k = k;
  a.n = (uint32_t) n; a.dist = dist; a.end_loc = end_loc;
  a.hbuf = nullptr; a.hbuf_stride = 0;
  a.last_pos = last_pos;
  // eq_tabs (device): uint32 f[256], uint32 s[256], then uint8 cls[256]
  a.eq_f = eq_tabs; a.eq_s = eq_tabs ? eq_tabs + 256 : nullptr; a.eq_cls = eq_tabs ? (const uint8_t*) (eq_tabs + 512) : nullptr;
  a.force_long = eq_tabs ? 1 : 0;
  a.two = 2;
  void* p;
  int rc = dgpu_reserve(ctx, SLOT_PERM, n * sizeof(uint32_t), &p);
  if (rc) return rc;
  a.perm = (uint32_t*) p;
  rc = dgpu_reserve(ctx, SLOT_COUNTS, 64 * sizeof(uint32_t), &p);
  if (rc) return rc;
  a.counts = (uint32_t*) p;

  DGPU_CUDA(ctx, cudaMemsetAsync(a.counts, 0, 64 * sizeof(uint32_t), st));
  const uint32_t cb = (uint32_t) ((n + 255) / 256);
  ed_count_kernel<<<cb, 256, 0, st>>>(a, mode);
  DGPU_LAUNCH_CHECK(ctx, "ed_count");
  ed_offsets_kernel<<<1, 1, 0, st>>>(a.counts);
  DGPU_LAUNCH_CHECK(ctx, "ed_offsets");
  ed_scatter_kernel<<<cb, 256, 0, st>>>(a, mode);
  DGPU_LAUNCH_CHECK(ctx, "ed_scatter");
  uint32_t hc[64];
  if (ctx->async_bound) {
    // Asynchronous form (dgpu_set_async_bound): no host round trip. Every class is launched with a grid sized from the job count (the kernels
    // read their own class counts on the device and an empty class returns at once), the stripe scratch of long targets from the caller's bound.
    for (int c = 0; c < 64; ++c) hc[c] = 0;
    const uint32_t bound = ctx->async_bound;
    hc[1] = hc[2] = (uint32_t) n;
    if (bound > 64) hc[3] = (uint32_t) n;
    if (bound > 96) hc[4] = (uint32_t) n;
    if (bound > 128 || a.force_long) { hc[5] = (uint32_t) n; if (bound > 2048) hc[24] = bound; }
    if (mode == DGPU_MODE_HW && !a.force_long && !end_loc && n > 1)   // pair classes (ed_pair_class): at most n / 2 pairs
      for (int c = 1; c <= 4; ++c) hc[ED_PAIR_CNT + c] = hc[c] ? (uint32_t) (n / 2) : 0;
  } else {
    // One small D2H so that launches are sized exactly and empty classes cost nothing.
    DGPU_CUDA(ctx, cudaMemcpyAsync(hc, a.counts, sizeof(hc), cudaMemcpyDeviceToHost, st));
    DGPU_CUDA(ctx, cudaStreamSynchronize(st));
  }

  if (mode == DGPU_MODE_HW) return launch_mode<DGPU_MODE_HW>(ctx, a, hc, st);
  if (mode == DGPU_MODE_SHW) return launch_mode<DGPU_MODE_SHW>(ctx, a, hc, st);
  return launch_mode<DGPU_MODE_NW>(ctx, a, hc, st);
}

extern "C" {

int dgpu_edit_distance(dgpu_ctx* ctx, const uint8_t* seqs, uint64_t seqs_bytes,
                       const uint32_t* q_off, const uint32_t* q_len,
                       const uint32_t* t_off, const uint32_t* t_len,
                       const int32_t* k, int mode, uint64_t n,
                       int32_t* dist, int32_t* end_loc) {
  DgpuCallTrace trace_("dgpu_edit_distance", n);
  if (!ctx) return DGPU_ERR_ARG;
  if (n == 0) return DGPU_OK;
  if (!seqs || !q_off || !q_len || !t_off || !t_len || !dist) return DGPU_ERR_ARG;
  if (n >= (1ull << 31) || seqs_bytes >= (1ull << 32)) return DGPU_ERR_ARG;
  // caller buffers: every sequence inside the arena. Small batches are checked here; the pipelined path below checks on the device while it
  // reduces the arena extents (a host loop over 10 M jobs reads 160 MB and cost 11 ms of an 18 ms call)
  const uint64_t njc0 = std::min<uint64_t>(ED_PIPE_MAX_CHUNKS, n / ED_PIPE_MIN_JOBS);
  if (njc0 < 2 || seqs_bytes < (32u << 20))
    for (uint64_t i = 0; i < n; ++i)
      if ((uint64_t) q_off[i] + q_len[i] > seqs_bytes || (uint64_t) t_off[i] + t_len[i] > seqs_bytes) { ctx->last_error = "dgpu_edit_distance: a sequence lies outside the arena"; return DGPU_ERR_ARG; }
  DGPU_CUDA(ctx, cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  void *d_seqs, *d_qoff, *d_qlen, *d_toff, *d_tlen, *d_k = nullptr, *d_dist, *d_end = nullptr;
  int rc;
  if ((rc = dgpu_reserve(ctx, SLOT_SEQS, seqs_bytes + 64, &d_seqs))) return rc;
  if ((rc = dgpu_reserve(ctx, SLOT_QOFF, n * 4, &d_qoff))) return rc;
  if ((rc = dgpu_reserve(ctx, SLOT_QLEN, n * 4, &d_qlen))) return rc;
  if ((rc = dgpu_reserve(ctx, SLOT_TOFF, n * 4, &d_toff))) return rc;
  if ((rc = dgpu_reserve(ctx, SLOT_TLEN, n * 4, &d_tlen))) return rc;
  if (k && (rc = dgpu_reserve(ctx, SLOT_K, n * 4, &d_k))) return rc;
  if ((rc = dgpu_reserve(ctx, SLOT_DIST, n * 4, &d_dist))) return rc;
  if (end_loc && (rc = dgpu_reserve(ctx, SLOT_ENDLOC, n * 4, &d_end))) return rc;

  // Small batches: one copy-in, one pass, one copy-out on the context stream.
  const uint64_t njc = std::min<uint64_t>(ED_PIPE_MAX_CHUNKS, n / ED_PIPE_MIN_JOBS);
  if (njc < 2 || seqs_bytes < (32u << 20)) {
    DGPU_CUDA(ctx, cudaMemcpyAsync(d_seqs, seqs, seqs_bytes, cudaMemcpyHostToDevice, st));
    DGPU_CUDA(ctx, cudaMemcpyAsync(d_qoff, q_off, n * 4, cudaMemcpyHostToDevice, st));
    DGPU_CUDA(ctx, cudaMemcpyAsync(d_qlen, q_len, n * 4, cudaMemcpyHostToDevice, st));
    DGPU_CUDA(ctx, cudaMemcpyAsync(d_toff, t_off, n * 4, cudaMemcpyHostToDevice, st));
    DGPU_CUDA(ctx, cudaMemcpyAsync(d_tlen, t_len, n * 4, cudaMemcpyHostToDevice, st));
    if (k) DGPU_CUDA(ctx, cudaMemcpyAsync(d_k, k, n * 4, cudaMemcpyHostToDevice, st));
    rc = dgpu_edit_distance_dev(ctx, (const uint8_t*) d_seqs, seqs_bytes, (const uint32_t*) d_qoff, (const uint32_t*) d_qlen,
                                (const uint32_t*) d_toff, (const uint32_t*) d_tlen, (const int32_t*) d_k, mode, n,
                                (int32_t*) d_dist, (int32_t*) d_end, st);
    if (rc) return rc;
    DGPU_CUDA(ctx, cudaMemcpyAsync(dist, d_dist, n * 4, cudaMemcpyDeviceToHost, st));
    if (end_loc) DGPU_CUDA(ctx, cudaMemcpyAsync(end_loc, d_end, n * 4, cudaMemcpyDeviceToHost, st));
    DGPU_CUDA(ctx, cudaStreamSynchronize(st));
    return DGPU_OK;
  }

  // Large batches (the genotyping batch of src/coverage.h:412-454 is 131072 x threads jobs): the call is PCIe-bound
  // (about 100 input bytes per job against 0.5 ns of kernel time), so the arena upload is pipelined against the
  // kernels. The job metadata goes first; the arena follows in ED_PIPE_PIECES pieces on a copy stream; the jobs
  // are cut into njc index ranges, and range c is launched as soon as the arena prefix it reads (its largest
  // q_off+q_len / t_off+t_len, reduced on the device from the uploaded metadata) has arrived. Results of a
  // finished range go back on a third stream. Any job order is correct; arena-ordered jobs (the way batches are
  // built: reads appended as they are scanned) overlap fully.
  if ((rc = dgpu_pipe_init(ctx))) return rc;
  cudaStream_t cs = ctx->copy_stream, os = ctx->out_stream;
  cudaEvent_t* ev = ctx->pipe_events.data();  // [0] metadata, [1..PIECES] arena pieces, [1+PIECES..] range done
  DGPU_CUDA(ctx, cudaMemcpyAsync(d_qoff, q_off, n * 4, cudaMemcpyHostToDevice, cs));
  DGPU_CUDA(ctx, cudaMemcpyAsync(d_qlen, q_len, n * 4, cudaMemcpyHostToDevice, cs));
  DGPU_CUDA(ctx, cudaMemcpyAsync(d_toff, t_off, n * 4, cudaMemcpyHostToDevice, cs));
  DGPU_CUDA(ctx, cudaMemcpyAsync(d_tlen, t_len, n * 4, cudaMemcpyHostToDevice, cs));
  if (k) DGPU_CUDA(ctx, cudaMemcpyAsync(d_k, k, n * 4, cudaMemcpyHostToDevice, cs));
  DGPU_CUDA(ctx, cudaEventRecord(ev[0], cs));
  const uint64_t piece = (((seqs_bytes + ED_PIPE_PIECES - 1) / ED_PIPE_PIECES) + 0xfffffull) & ~0xfffffull;  // 1 MiB multiple
  int npieces = 0;
  for (uint64_t o = 0; o < seqs_bytes; o += piece, ++npieces) {
    const uint64_t len = std::min<uint64_t>(piece, seqs_bytes - o);
    DGPU_CUDA(ctx, cudaMemcpyAsync((uint8_t*) d_seqs + o, seqs + o, len, cudaMemcpyHostToDevice, cs));
    DGPU_CUDA(ctx, cudaEventRecord(ev[1 + npieces], cs));
  }
  const uint64_t jobs_per = (n + njc - 1) / njc;
  void* p;
  if ((rc = dgpu_reserve(ctx, SLOT_WORK1, (ED_PIPE_MAX_CHUNKS + 1) * sizeof(uint32_t), &p))) return rc;
  uint32_t* d_ext = (uint32_t*) p;
  DGPU_CUDA(ctx, cudaStreamWaitEvent(st, ev[0], 0));
  DGPU_CUDA(ctx, cudaMemsetAsync(d_ext, 0, (ED_PIPE_MAX_CHUNKS + 1) * sizeof(uint32_t), st));
  ed_extent_kernel<<<(unsigned) ((n + 255) / 256), 256, 0, st>>>((const uint32_t*) d_qoff, (const uint32_t*) d_qlen, (const uint32_t*) d_toff,
                                                                 (const uint32_t*) d_tlen, (uint32_t) n, (uint32_t) jobs_per, (uint32_t) seqs_bytes, d_ext);
  DGPU_LAUNCH_CHECK(ctx, "ed_extent");
  uint32_t h_ext[ED_PIPE_MAX_CHUNKS + 1];
  DGPU_CUDA(ctx, cudaMemcpyAsync(h_ext, d_ext, sizeof(h_ext), cudaMemcpyDeviceToHost, st));
  DGPU_CUDA(ctx, cudaStreamSynchronize(st));
  if (h_ext[ED_PIPE_MAX_CHUNKS]) {
    cudaStreamSynchronize(cs);   // the arena upload reads the caller's buffer only inside seqs_bytes; let it drain
    ctx->last_error = "dgpu_edit_distance: a sequence lies outside the arena";
    return DGPU_ERR_ARG;
  }
  for (uint64_t c = 0; c < njc; ++c) {
    const uint64_t j0 = c * jobs_per;
    if (j0 >= n) break;
    const uint64_t cnt = std::min<uint64_t>(jobs_per, n - j0);
    const int need = h_ext[c] ? (int) ((h_ext[c] - 1) / piece) : 0;   // last arena piece this range reads
    DGPU_CUDA(ctx, cudaStreamWaitEvent(st, ev[1 + std::min(need, npieces - 1)], 0));
    rc = dgpu_edit_distance_dev(ctx, (const uint8_t*) d_seqs, seqs_bytes, (const uint32_t*) d_qoff + j0, (const uint32_t*) d_qlen + j0,
                                (const uint32_t*) d_toff + j0, (const uint32_t*) d_tlen + j0, d_k ? (const int32_t*) d_k + j0 : nullptr, mode, cnt,
                                (int32_t*) d_dist + j0, d_end ? (int32_t*) d_end + j0 : nullptr, st);
    if (rc) { cudaStreamSynchronize(cs); return rc; }
    cudaEvent_t done = ev[1 + ED_PIPE_PIECES + c];
    DGPU_CUDA(ctx, cudaEventRecord(done, st));
    DGPU_CUDA(ctx, cudaStreamWaitEvent(os, done, 0));
    DGPU_CUDA(ctx, cudaMemcpyAsync(dist + j0, (int32_t*) d_dist + j0, cnt * 4, cudaMemcpyDeviceToHost, os));
    if (end_loc) DGPU_CUDA(ctx, cudaMemcpyAsync(end_loc + j0, (int32_t*) d_end + j0, cnt * 4, cudaMemcpyDeviceToHost, os));
  }
  DGPU_CUDA(ctx, cudaStreamSynchronize(cs));
  DGPU_CUDA(ctx, cudaStreamSynchronize(st));
  DGPU_CUDA(ctx, cudaStreamSynchronize(os));
  return DGPU_OK;
}

}  // extern "C"
