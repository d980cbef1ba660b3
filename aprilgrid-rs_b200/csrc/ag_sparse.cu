// Sparse stages of the aprilgrid front end, sm_100a: everything between the threshold mask
// and the refined saddle list.  One CTA per frame; the data are a few hundred KB per frame
// and live in L2.
//
//   K3  k_label_clusters   4-connected components of the mask by union-find whose roots are
//                          the minimum raster index of each component, numbered in ascending
//                          root order (== the reference's raster-scan discovery order), plus
//                          the per-cluster centroid.
//                          reference: src/detector.rs:171-187 (init_saddle_clusters),
//                          src/image_util.rs:208-236 (pixel_bfs), src/detector.rs:421-429.
//   K4  k_refine_filter    one warp per candidate: 9x9 window of the blurred image -> 5x5
//                          cone convolution -> 6-parameter quadratic fit -> saddle test;
//                          then the k / phi filter with order-preserving compaction.
//                          reference: src/detector.rs:194-361 (rochade_refine), :432-445.
#include "ag_common.cuh"
#include "ag_kernels.h"
#include "ag_libm.h"

namespace ag {

// ----------------------------------------------------------------------------------------
// union-find helpers on the sparse parent array (only mask pixels are ever touched).
// Loads bypass L1 (ld.cg): parents are modified concurrently with atomicMin at L2.
// ----------------------------------------------------------------------------------------
AG_D int uf_find(const int* P, int p) {
  int q;
  while ((q = __ldcg(P + p)) != p) p = q;
  return p;
}
AG_D void uf_union(int* P, int a, int b) {
  while (true) {
    a = uf_find(P, a);
    b = uf_find(P, b);
    if (a == b) return;
    if (a < b) { int t = a; a = b; b = t; }
    int old = atomicMin(P + a, b);  // hang the larger root under the smaller one
    if (old == a) return;
    a = old;
  }
}

constexpr int kCclThreads = 1024;

// Block-wide exclusive scan of one int per thread (kCclThreads threads). Returns the
// exclusive prefix; *total receives the block sum.
AG_D int block_exclusive_scan(int v, int* s_warp /*[32]*/, int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int w = (lane < (int)(blockDim.x >> 5)) ? s_warp[lane] : 0;
    int winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= o) winc += t;
    }
    s_warp[lane] = winc - w;  // exclusive prefix of warp sums
    if (lane == 31) *total = winc;
  }
  __syncthreads();
  int r = s_warp[warp] + inc - v;
  __syncthreads();
  return r;
}

// Word-oriented version: every thread walks the set bits of its own mask words.  Works for any
// image and any fill of the mask; used when the compact pixel list below does not apply.
AG_D void label_clusters_words(const uint32_t* __restrict__ mask, const FrameGeom& g, int* __restrict__ parent,
                               int max_clusters, int* __restrict__ acc /*[F][max_clusters][3]*/,
                               float2* __restrict__ centers, int* __restrict__ n_clusters,
                               uint32_t* __restrict__ frame_status, int* s_warp, int& s_total) {
  const int f = blockIdx.x;
  const uint32_t* M = mask + (size_t)f * g.n_words;
  int* P = parent + (size_t)f * g.n_px;
  int* A = acc + (size_t)f * max_clusters * 3;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int wpr = g.wpr, w = g.w;

  // P0: every mask pixel points at its left neighbour if that is set, else at itself.
  for (int wi = tid; wi < g.n_words; wi += nt) {
    uint32_t m = M[wi];
    if (!m) continue;
    int row = wi / wpr, wc = wi - row * wpr;
    int base = row * w + wc * 32;
    uint32_t left = (m << 1) | (wc > 0 ? (M[wi - 1] >> 31) : 0u);
    while (m) {
      int b = __ffs(m) - 1;
      m &= m - 1;
      int p = base + b;
      P[p] = ((left >> b) & 1u) ? p - 1 : p;
    }
  }
  __syncthreads();
  // P1: union with the pixel above.  A pixel whose left and upper-left neighbours are both
  // set is already connected to its upper neighbour through them, so it is skipped.
  for (int wi = tid; wi < g.n_words; wi += nt) {
    uint32_t m = M[wi];
    if (!m || wi < wpr) continue;
    int row = wi / wpr, wc = wi - row * wpr;
    uint32_t up = M[wi - wpr];
    uint32_t u = m & up;
    if (!u) continue;
    uint32_t left = (m << 1) | (wc > 0 ? (M[wi - 1] >> 31) : 0u);
    uint32_t upleft = (up << 1) | (wc > 0 ? (M[wi - wpr - 1] >> 31) : 0u);
    u &= ~(left & upleft);
    int base = row * w + wc * 32;
    while (u) {
      int b = __ffs(u) - 1;
      u &= u - 1;
      uf_union(P, base + b, base + b - w);
    }
  }
  __syncthreads();
  // P2: flatten so that every pixel stores its root (= min raster index of the component).
  for (int wi = tid; wi < g.n_words; wi += nt) {
    uint32_t m = M[wi];
    if (!m) continue;
    int row = wi / wpr, wc = wi - row * wpr;
    int base = row * w + wc * 32;
    while (m) {
      int b = __ffs(m) - 1;
      m &= m - 1;
      int p = base + b;
      int r = uf_find(P, p);
      if (r != p) P[p] = r;
    }
  }
  __syncthreads();
  // P3: number the roots in ascending raster order.  Thread t owns a contiguous word range.
  const int per = (g.n_words + nt - 1) / nt;
  const int w_begin = min(tid * per, g.n_words), w_end = min(w_begin + per, g.n_words);
  int my_roots = 0;
  for (int wi = w_begin; wi < w_end; ++wi) {
    uint32_t m = M[wi];
    if (!m) continue;
    int row = wi / wpr, wc = wi - row * wpr;
    int base = row * w + wc * 32;
    while (m) {
      int b = __ffs(m) - 1;
      m &= m - 1;
      int p = base + b;
      if (__ldcg(P + p) == p) ++my_roots;
    }
  }
  int offset = block_exclusive_scan(my_roots, s_warp, &s_total);
  const int total = s_total;
  for (int wi = w_begin; wi < w_end; ++wi) {
    uint32_t m = M[wi];
    if (!m) continue;
    int row = wi / wpr, wc = wi - row * wpr;
    int base = row * w + wc * 32;
    while (m) {
      int b = __ffs(m) - 1;
      m &= m - 1;
      int p = base + b;
      if (__ldcg(P + p) == p) {
        P[p] = -(offset + 1);  // root now carries its cluster id, encoded negative
        ++offset;
      }
    }
  }
  const int n_used = min(total, max_clusters);
  for (int i = tid; i < n_used * 3; i += nt) A[i] = 0;
  __syncthreads();
  // P4: accumulate (sum x, sum y, count) per cluster with integer atomics.  The reference
  // sums the coordinates in f32 (detector.rs:424-426); integer sums below 2^24 are exact
  // in f32 whatever the order, so one int->float conversion reproduces them bit for bit.
  for (int wi = tid; wi < g.n_words; wi += nt) {
    uint32_t m = M[wi];
    if (!m) continue;
    int row = wi / wpr, wc = wi - row * wpr;
    int base = row * w + wc * 32;
    while (m) {
      int b = __ffs(m) - 1;
      m &= m - 1;
      int p = base + b;
      int v = __ldcg(P + p);
      int cid = v < 0 ? -v - 1 : -__ldcg(P + v) - 1;
      if (cid < max_clusters) {
        atomicAdd(A + 3 * cid + 0, wc * 32 + b);
        atomicAdd(A + 3 * cid + 1, row);
        atomicAdd(A + 3 * cid + 2, 1);
      }
    }
  }
  __syncthreads();
  float2* Cn = centers + (size_t)f * max_clusters;
  for (int c = tid; c < n_used; c += nt) {
    float n = (float)__ldcg(A + 3 * c + 2);
    float sx = (float)__ldcg(A + 3 * c + 0), sy = (float)__ldcg(A + 3 * c + 1);
    Cn[c] = make_float2(__fdiv_rn(sx, n), __fdiv_rn(sy, n));  // detector.rs:427
  }
  if (tid == 0) {
    n_clusters[f] = n_used;
    if (total > max_clusters) atomicOr(frame_status + f, (uint32_t)AG_FRAME_CLUSTER_OVERFLOW);
  }
}

// K3.  One CTA per frame.  The mask is 1-4 % full, so walking mask words leaves most lanes idle
// (4 of 32 active in the word-oriented version).  Here the set pixels are first COMPACTED into a
// list in raster order (count bits per thread, block scan, write (row << 16 | x) entries); every
// later pass runs over the list with all lanes busy:
//   P0 parent = left neighbour or self      P1 union with the pixel above (atomicMin hooking:
//   the root is the component's minimum raster index)      P2 flatten      P3 number the roots
//   in list (= raster) order with a block scan (= the reference's discovery order,
//   detector.rs:174-185)      P4 integer centroid sums.
// Falls back to the word-oriented version when the list does not fit or coordinates exceed 16 bits.
__global__ void __launch_bounds__(kCclThreads)
k_label_clusters(const uint32_t* __restrict__ mask, FrameGeom g, int* __restrict__ parent,
                 int max_clusters, int* __restrict__ acc /*[F][max_clusters][3]*/,
                 float2* __restrict__ centers, int* __restrict__ n_clusters,
                 uint32_t* __restrict__ frame_status, uint32_t* __restrict__ pixlist, int list_cap,
                 const int* __restrict__ only_if /*[F] or null: run only the frames flagged here*/) {
  __shared__ int s_warp[32];
  __shared__ int s_total;
  const int f = blockIdx.x;
  if (only_if && !only_if[f]) return;  // the run-based kernel handled this frame
  const uint32_t* M = mask + (size_t)f * g.n_words;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int wpr = g.wpr, w = g.w;
  // A: count the set pixels of this thread's contiguous word range
  const int per = (g.n_words + nt - 1) / nt;
  const int w_begin = min(tid * per, g.n_words), w_end = min(w_begin + per, g.n_words);
  int my_px = 0;
  for (int wi = w_begin; wi < w_end; ++wi) my_px += __popc(M[wi]);
  int offset = block_exclusive_scan(my_px, s_warp, &s_total);
  const int n_px = s_total;
  __syncthreads();
  if (!pixlist || n_px > list_cap || g.w > 65535 || g.h > 65535) {  // block-uniform
    label_clusters_words(mask, g, parent, max_clusters, acc, centers, n_clusters, frame_status, s_warp,
                         s_total);
    return;
  }
  uint32_t* L = pixlist + (size_t)f * list_cap;
  int* P = parent + (size_t)f * g.n_px;
  int* A = acc + (size_t)f * max_clusters * 3;
  if (my_px) {
    int row = w_begin / wpr, wc = w_begin - row * wpr;
    for (int wi = w_begin; wi < w_end; ++wi) {
      uint32_t m = M[wi];
      while (m) {
        const int b = __ffs(m) - 1;
        m &= m - 1;
        L[offset++] = ((uint32_t)row << 16) | (uint32_t)(wc * 32 + b);
      }
      if (++wc == wpr) { wc = 0; ++row; }
    }
  }
  __syncthreads();
  auto bit = [&](int row, int x) -> bool { return (M[row * wpr + (x >> 5)] >> (x & 31)) & 1u; };
  // P0: every mask pixel points at its left neighbour if that is set, else at itself.
  for (int i = tid; i < n_px; i += nt) {
    const uint32_t e = L[i];
    const int row = (int)(e >> 16), x = (int)(e & 0xffffu);
    const int p = row * w + x;
    P[p] = (x > 0 && bit(row, x - 1)) ? p - 1 : p;
  }
  __syncthreads();
  // P1: union with the pixel above.  A pixel whose left and upper-left neighbours are both
  // set is already connected to its upper neighbour through them, so it is skipped.
  for (int i = tid; i < n_px; i += nt) {
    const uint32_t e = L[i];
    const int row = (int)(e >> 16), x = (int)(e & 0xffffu);
    if (row == 0 || !bit(row - 1, x)) continue;
    if (x > 0 && bit(row, x - 1) && bit(row - 1, x - 1)) continue;
    const int p = row * w + x;
    uf_union(P, p, p - w);
  }
  __syncthreads();
  // P2: flatten so that every pixel stores its root (= min raster index of the component).
  for (int i = tid; i < n_px; i += nt) {
    const uint32_t e = L[i];
    const int p = (int)(e >> 16) * w + (int)(e & 0xffffu);
    const int r = uf_find(P, p);
    if (r != p) P[p] = r;
  }
  __syncthreads();
  // P3: number the roots in ascending raster order.  Thread t owns a contiguous part of the list.
  const int lper = (n_px + nt - 1) / nt;
  const int l_begin = min(tid * lper, n_px), l_end = min(l_begin + lper, n_px);
  int my_roots = 0;
  for (int i = l_begin; i < l_end; ++i) {
    const uint32_t e = L[i];
    const int p = (int)(e >> 16) * w + (int)(e & 0xffffu);
    if (__ldcg(P + p) == p) ++my_roots;
  }
  int roff = block_exclusive_scan(my_roots, s_warp, &s_total);
  const int total = s_total;
  for (int i = l_begin; i < l_end; ++i) {
    const uint32_t e = L[i];
    const int p = (int)(e >> 16) * w + (int)(e & 0xffffu);
    if (__ldcg(P + p) == p) {
      P[p] = -(roff + 1);  // root now carries its cluster id, encoded negative
      ++roff;
    }
  }
  const int n_used = min(total, max_clusters);
  for (int i = tid; i < n_used * 3; i += nt) A[i] = 0;
  __syncthreads();
  // P4: accumulate (sum x, sum y, count) per cluster with integer atomics.  The reference
  // sums the coordinates in f32 (detector.rs:424-426); integer sums below 2^24 are exact
  // in f32 whatever the order, so one int->float conversion reproduces them bit for bit.
  for (int i = tid; i < n_px; i += nt) {
    const uint32_t e = L[i];
    const int row = (int)(e >> 16), x = (int)(e & 0xffffu);
    const int p = row * w + x;
    const int v = __ldcg(P + p);
    const int cid = v < 0 ? -v - 1 : -__ldcg(P + v) - 1;
    if (cid < max_clusters) {
      atomicAdd(A + 3 * cid + 0, x);
      atomicAdd(A + 3 * cid + 1, row);
      atomicAdd(A + 3 * cid + 2, 1);
    }
  }
  __syncthreads();
  float2* Cn = centers + (size_t)f * max_clusters;
  for (int c = tid; c < n_used; c += nt) {
    float n = (float)__ldcg(A + 3 * c + 2);
    float sx = (float)__ldcg(A + 3 * c + 0), sy = (float)__ldcg(A + 3 * c + 1);
    Cn[c] = make_float2(__fdiv_rn(sx, n), __fdiv_rn(sy, n));  // detector.rs:427
  }
  if (tid == 0) {
    n_clusters[f] = n_used;
    if (total > max_clusters) atomicOr(frame_status + f, (uint32_t)AG_FRAME_CLUSTER_OVERFLOW);
  }
}

// ----------------------------------------------------------------------------------------
// K3, run-based.  One CTA per frame; the whole union-find lives in SHARED memory.
//
// The nodes are the maximal horizontal RUNS of set pixels (a few thousand per frame instead of
// ~20 k pixels), numbered in raster order, so the minimum run index of a component is the run
// that contains its minimum raster pixel:
//   A  count run starts per thread (contiguous word ranges), block scan -> run ids
//   B  write the runs (row << 16 | x0, x1) to a compact buffer; runs per row -> row starts
//   C  one thread per pair of adjacent rows merges their run lists (two pointers) and unites
//      overlapping runs with atomicMin hooking on the shared parent array
//   D  flatten; number the roots in run (= raster) order with a block scan -- the reference's
//      discovery order (detector.rs:174-185)
//   E  per run, closed-form sums (n, sum x, sum y) into the cluster accumulators
// No per-pixel parent array is written (the labels tap uses the pixel-list version).
// Falls back (returns false, block-uniform) when the frame has too many runs or rows.
// ----------------------------------------------------------------------------------------
constexpr int kRunCap = 12288;  // runs per frame held in shared memory (48 KB of parents)
constexpr int kRowCap = 4096;   // rows per frame (row starts in shared memory)

AG_D int suf_find(volatile int* P, int p) {
  int q;
  while ((q = P[p]) != p) p = q;
  return p;
}
AG_D void suf_union(int* P, int a, int b) {
  while (true) {
    a = suf_find(P, a);
    b = suf_find(P, b);
    if (a == b) return;
    if (a < b) { int t = a; a = b; b = t; }
    int old = atomicMin(P + a, b);  // hang the larger root under the smaller one
    if (old == a) return;
    a = old;
  }
}

__global__ void __launch_bounds__(kCclThreads)
k_label_runs(const uint32_t* __restrict__ mask, FrameGeom g, int max_clusters,
             int* __restrict__ acc /*[F][max_clusters][3]*/, float2* __restrict__ centers,
             int* __restrict__ n_clusters, uint32_t* __restrict__ frame_status,
             uint32_t* __restrict__ runbuf /*[F][2 * kRunCap]*/, int* __restrict__ fallback /*[F]*/) {
  extern __shared__ __align__(16) int s_dyn[];
  int* s_parent = s_dyn;                 // [kRunCap]
  int* s_rowstart = s_dyn + kRunCap;     // [kRowCap + 1]
  __shared__ int s_warp[32];
  __shared__ int s_total;
  const int f = blockIdx.x;
  const uint32_t* M = mask + (size_t)f * g.n_words;
  const int tid = threadIdx.x, nt = blockDim.x;
  const int wpr = g.wpr;
  // A: run starts in this thread's contiguous word range
  const int per = (g.n_words + nt - 1) / nt;
  const int w_begin = min(tid * per, g.n_words), w_end = min(w_begin + per, g.n_words);
  int my_runs = 0;
  {
    int wc = w_begin % wpr;
    for (int wi = w_begin; wi < w_end; ++wi) {
      const uint32_t m = M[wi];
      const uint32_t carry = wc > 0 ? (M[wi - 1] >> 31) : 0u;
      my_runs += __popc(m & ~((m << 1) | carry));
      if (++wc == wpr) wc = 0;
    }
  }
  int rid = block_exclusive_scan(my_runs, s_warp, &s_total);
  const int R = s_total;
  __syncthreads();
  if (R > kRunCap || g.h > kRowCap || g.w > 65535) {  // block-uniform
    if (tid == 0) fallback[f] = 1;
    return;
  }
  if (tid == 0) fallback[f] = 0;
  uint32_t* RB = runbuf + (size_t)f * 2 * kRunCap;
  for (int i = tid; i <= g.h; i += nt) s_rowstart[i] = 0;
  __syncthreads();
  // B: write the runs; count runs per row into s_rowstart[row + 1]
  if (my_runs) {
    int row = w_begin / wpr, wc = w_begin - row * wpr;
    for (int wi = w_begin; wi < w_end; ++wi) {
      const uint32_t m = M[wi];
      const uint32_t carry = wc > 0 ? (M[wi - 1] >> 31) : 0u;
      uint32_t starts = m & ~((m << 1) | carry);
      while (starts) {
        const int b = __ffs(starts) - 1;
        starts &= starts - 1;
        // end of the run: first clear bit at or after b, possibly in a following word of the row
        int x1;
        {
          uint32_t rest = ~(m >> b);  // bit k set <=> pixel b + k is clear (or beyond the word)
          int len = __ffs(rest) - 1;  // rest != 0 unless b == 0 and m == all ones
          if (rest == 0u) len = 32;
          int xe = wc * 32 + b + len;  // one past the run inside this word
          if (b + len == 32) {         // the run touches the word's end: follow it
            int wj = wi + 1, wcj = wc + 1;
            while (wcj < wpr) {
              const uint32_t mj = M[wj];
              if (mj == 0xffffffffu) { xe += 32; ++wj; ++wcj; continue; }
              xe += __ffs(~mj) - 1;
              break;
            }
          }
          x1 = xe - 1;
        }
        RB[2 * rid] = ((uint32_t)row << 16) | (uint32_t)(wc * 32 + b);
        RB[2 * rid + 1] = (uint32_t)x1;
        s_parent[rid] = rid;
        atomicAdd(&s_rowstart[row + 1], 1);
        ++rid;
      }
      if (++wc == wpr) { wc = 0; ++row; }
    }
  }
  __syncthreads();
  // exclusive scan of the per-row counts: s_rowstart[y] = first run of row y, [h] = R
  {
    const int rper = (g.h + 1 + nt - 1) / nt;
    const int r0 = min(tid * rper, g.h + 1), r1 = min(r0 + rper, g.h + 1);
    int sum = 0;
    for (int y = r0; y < r1; ++y) sum += s_rowstart[y];
    int off = block_exclusive_scan(sum, s_warp, &s_total);
    for (int y = r0; y < r1; ++y) {  // inclusive over the shifted counts == start of row y
      off += s_rowstart[y];
      s_rowstart[y] = off;
    }
  }
  __syncthreads();
  // C: unite overlapping runs of adjacent rows (4-connectivity: they share a column)
  for (int y = 1 + tid; y < g.h; y += nt) {
    int a = s_rowstart[y], a_end = s_rowstart[y + 1];
    int b = s_rowstart[y - 1], b_end = a;
    if (a == a_end || b == b_end) continue;
    uint32_t ax0 = RB[2 * a] & 0xffffu, ax1 = RB[2 * a + 1];
    uint32_t bx0 = RB[2 * b] & 0xffffu, bx1 = RB[2 * b + 1];
    while (true) {
      if (ax0 <= bx1 && bx0 <= ax1) suf_union(s_parent, a, b);
      if (ax1 <= bx1) {
        if (++a == a_end) break;
        ax0 = RB[2 * a] & 0xffffu;
        ax1 = RB[2 * a + 1];
      } else {
        if (++b == b_end) break;
        bx0 = RB[2 * b] & 0xffffu;
        bx1 = RB[2 * b + 1];
      }
    }
  }
  __syncthreads();
  // D: flatten, then number the roots in run order
  for (int i = tid; i < R; i += nt) {
    const int r = suf_find(s_parent, i);
    if (r != i) s_parent[i] = r;
  }
  __syncthreads();
  const int lper = (R + nt - 1) / nt;
  const int l_begin = min(tid * lper, R), l_end = min(l_begin + lper, R);
  int my_roots = 0;
  for (int i = l_begin; i < l_end; ++i) my_roots += s_parent[i] == i ? 1 : 0;
  int roff = block_exclusive_scan(my_roots, s_warp, &s_total);
  const int total = s_total;
  for (int i = l_begin; i < l_end; ++i)
    if (s_parent[i] == i) {
      s_parent[i] = -(roff + 1);  // root now carries its cluster id, encoded negative
      ++roff;
    }
  int* A = acc + (size_t)f * max_clusters * 3;
  const int n_used = min(total, max_clusters);
  for (int i = tid; i < n_used * 3; i += nt) A[i] = 0;
  __syncthreads();
  // E: per run, n = len, sum x = len * x0 + len (len - 1) / 2, sum y = len * row (exact integers;
  // the reference's f32 sums of integers below 2^24 equal them, detector.rs:424-426)
  for (int i = tid; i < R; i += nt) {
    const int v = s_parent[i];
    const int cid = v < 0 ? -v - 1 : -s_parent[v] - 1;
    if (cid < max_clusters) {
      const uint32_t e = RB[2 * i];
      const int row = (int)(e >> 16), x0 = (int)(e & 0xffffu), len = (int)RB[2 * i + 1] - x0 + 1;
      atomicAdd(A + 3 * cid + 0, len * x0 + len * (len - 1) / 2);
      atomicAdd(A + 3 * cid + 1, len * row);
      atomicAdd(A + 3 * cid + 2, len);
    }
  }
  __syncthreads();
  float2* Cn = centers + (size_t)f * max_clusters;
  for (int c = tid; c < n_used; c += nt) {
    float n = (float)__ldcg(A + 3 * c + 2);
    float sx = (float)__ldcg(A + 3 * c + 0), sy = (float)__ldcg(A + 3 * c + 1);
    Cn[c] = make_float2(__fdiv_rn(sx, n), __fdiv_rn(sy, n));  // detector.rs:427
  }
  if (tid == 0) {
    n_clusters[f] = n_used;
    if (total > max_clusters) atomicOr(frame_status + f, (uint32_t)AG_FRAME_CLUSTER_OVERFLOW);
  }
}

// Test tap: dense label image (cluster id or -1) from the mask and the parent array.
__global__ void k_labels_tap(const uint32_t* __restrict__ mask, FrameGeom g,
                             const int* __restrict__ parent, int32_t* __restrict__ labels,
                             uint8_t* __restrict__ mask_u8) {
  int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= g.n_px) return;
  int row = p / g.w, x = p - row * g.w;
  uint32_t m = mask[row * g.wpr + (x >> 5)];
  bool set = (m >> (x & 31)) & 1u;
  if (mask_u8) mask_u8[p] = set ? 1 : 0;
  if (labels) {
    int lab = -1;
    if (set) {
      int v = parent[p];
      lab = v < 0 ? -v - 1 : -parent[v] - 1;
    }
    labels[p] = lab;
  }
}

// ----------------------------------------------------------------------------------------
// K4: rochade refine + filter
// ----------------------------------------------------------------------------------------
__constant__ float c_cone[25];      // normalised cone kernel, detector.rs:240-254
__constant__ float c_pinv[6 * 25];  // pseudo-inverse of [x^2, xy, y^2, x, y, 1], :208-237

int upload_rochade_tables(const float* cone25, const float* pinv150) {
  cudaError_t e = cudaMemcpyToSymbol(c_cone, cone25, sizeof(float) * 25);
  if (e != cudaSuccess) return (int)e;
  e = cudaMemcpyToSymbol(c_pinv, pinv150, sizeof(float) * 150);
  return (int)e;
}

constexpr int kRefineThreads = 512;
constexpr int kRefineWarps = kRefineThreads / 32;

// f32::acos / f32::atan2 of the reference = the platform's acosf / atan2f: glibc's routines restated
// operation for operation (ag_libm.h), same bits as the oracle's libm calls.
AG_D float acosf_cr(float x) { return lm_acosf(x); }
AG_D float atan2f_cr(float y, float x) { return lm_atan2f(y, x); }

// Rust f32::round (half away from zero) followed by `as i32` (saturating).
AG_D int round_to_i32(float v) {
  float r = roundf(v);
  if (r != r) return 0;
  if (r >= 2147483648.0f) return 2147483647;
  if (r <= -2147483648.0f) return (int)0x80000000;
  return (int)r;
}

__global__ void __launch_bounds__(kRefineThreads)
k_refine_filter(const float* __restrict__ blur, FrameGeom g, const float2* __restrict__ centers,
                const int* __restrict__ n_clusters, int max_clusters,
                ag_saddle* __restrict__ raw, uint8_t* __restrict__ raw_valid,
                float min_angle, float max_angle, int max_saddles,
                ag_saddle* __restrict__ refined, int* __restrict__ n_refined,
                uint32_t* __restrict__ frame_status) {
  __shared__ float s_win[kRefineWarps][81];
  __shared__ float s_smooth[kRefineWarps][25];
  __shared__ float s_cone[25];
  __shared__ float s_pinv[150];
  __shared__ float s_redf[kRefineWarps];
  __shared__ int s_warp[32];
  __shared__ int s_total;
  __shared__ float s_kmax;

  const int f = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* B = blur + (size_t)f * g.n_px;
  const float2* Cn = centers + (size_t)f * max_clusters;
  ag_saddle* R = raw + (size_t)f * max_clusters;
  uint8_t* V = raw_valid + (size_t)f * max_clusters;
  const int n = n_clusters[f];
  if (tid < 25) s_cone[tid] = c_cone[tid];
  if (tid < 150) s_pinv[tid] = c_pinv[tid];
  __syncthreads();

  float kmax = -3.40282347e+38f;  // f32::MIN, detector.rs:436
  for (int c = warp; c < n; c += kRefineWarps) {
    const float2 ic = Cn[c];
    const float rxf = roundf(ic.x), ryf = roundf(ic.y);
    const int rx = round_to_i32(ic.x), ry = round_to_i32(ic.y);
    bool ok = !(ry - 4 < 0 || ry + 4 >= g.h || rx - 4 < 0 || rx + 4 >= g.w);  // :268-274
    ag_saddle out;
    bool valid = false;
    if (ok) {  // warp-uniform
      const float* src = B + (size_t)(ry - 4) * g.w + (rx - 4);
      for (int i = lane; i < 81; i += 32) {
        int r = i / 9, cc = i - r * 9;
        s_win[warp][i] = src[(size_t)r * g.w + cc];
      }
      __syncwarp();
      if (lane < 25) {  // 5x5 cone convolution, accumulation order of :283-297
        int r = lane / 5, cc = lane - r * 5;
        float conv = 0.0f;
#pragma unroll
        for (int pr = 0; pr < 5; ++pr)
#pragma unroll
          for (int pc = 0; pc < 5; ++pc)
            conv = __fadd_rn(conv, __fmul_rn(s_win[warp][(r + pr) * 9 + cc + pc], s_cone[pr * 5 + pc]));
        s_smooth[warp][lane] = conv;
      }
      __syncwarp();
      float prm = 0.0f;
      if (lane < 6) {  // params[j] = sum_i pinv[j][i] * smooth[i], i ascending (:321-328)
#pragma unroll
        for (int i = 0; i < 25; ++i)
          prm = __fadd_rn(prm, __fmul_rn(s_pinv[lane * 25 + i], s_smooth[warp][i]));
      }
      const float a1 = __shfl_sync(0xffffffffu, prm, 0), a2 = __shfl_sync(0xffffffffu, prm, 1),
                  a3 = __shfl_sync(0xffffffffu, prm, 2), a4 = __shfl_sync(0xffffffffu, prm, 3),
                  a5 = __shfl_sync(0xffffffffu, prm, 4);
      const float fxx = __fmul_rn(2.0f, a1), fyy = __fmul_rn(2.0f, a3), fxy = a2;
      const float d = __fsub_rn(__fmul_rn(fxx, fyy), __fmul_rn(fxy, fxy));
      if (d < 0.0f) {
        // math_util::find_xy(2a1, a2, a4, a2, 2a3, a5): 2x2 LU with row pivoting, f32.
        float m00 = fxx, m01 = a2, m10 = a2, m11 = fyy, r0 = -a4, r1 = -a5;
        if (fabsf(m10) > fabsf(m00)) {
          float t;
          t = m00; m00 = m10; m10 = t;
          t = m01; m01 = m11; m11 = t;
          t = r0; r0 = r1; r1 = t;
        }
        const float l = __fdiv_rn(m10, m00);
        const float u11 = __fsub_rn(m11, __fmul_rn(l, m01));
        const float z1 = __fsub_rn(r1, __fmul_rn(l, r0));
        const float y0 = __fdiv_rn(z1, u11);
        const float x0 = __fdiv_rn(__fsub_rn(r0, __fmul_rn(m01, y0)), m00);
        if (fabsf(x0) <= 1.0f && fabsf(y0) <= 1.0f) {
          const float c5 = __fdiv_rn(__fadd_rn(a1, a3), 2.0f);
          const float c4 = __fdiv_rn(__fsub_rn(a1, a3), 2.0f);
          const float c3 = __fdiv_rn(a2, 2.0f);
          const float k = __fsqrt_rn(__fadd_rn(__fmul_rn(c4, c4), __fmul_rn(c3, c3)));
          if (fabsf(c5) < k) {
            const float kPi = 3.14159274101257324f;
            float phi = __fmul_rn(__fdiv_rn(__fdiv_rn(acosf_cr(__fdiv_rn(-c5, k)), 2.0f), kPi), 180.0f);
            float theta = __fmul_rn(__fdiv_rn(__fdiv_rn(atan2f_cr(c3, c4), 2.0f), kPi), 180.0f);
            out.x = __fadd_rn(rxf, x0);
            out.y = __fadd_rn(ryf, y0);
            out.k = k;
            out.theta = theta;
            out.phi = phi;
            valid = true;
          }
        }
      }
      __syncwarp();
    }
    if (lane == 0) {
      V[c] = valid ? 1 : 0;
      if (valid) {
        R[c] = out;
        kmax = fmaxf(kmax, out.k);
      }
    }
  }
  // block max of k
  if (lane == 0) s_redf[warp] = kmax;
  __syncthreads();
  if (tid == 0) {
    float m = s_redf[0];
    for (int i = 1; i < kRefineWarps; ++i) m = fmaxf(m, s_redf[i]);
    s_kmax = __fdiv_rn(m, 10.0f);  // detector.rs:436
  }
  __syncthreads();
  const float kthr = s_kmax;
  // order-preserving compaction of the survivors (detector.rs:437-444)
  const int per = (n + kRefineThreads - 1) / kRefineThreads;
  const int c_begin = min(tid * per, n), c_end = min(c_begin + per, n);
  int mine = 0;
  for (int c = c_begin; c < c_end; ++c) {
    if (V[c]) {
      const ag_saddle s = R[c];
      if (s.k >= kthr && s.phi >= min_angle && s.phi <= max_angle) ++mine;
    }
  }
  int offset = block_exclusive_scan(mine, s_warp, &s_total);
  ag_saddle* O = refined + (size_t)f * max_saddles;
  for (int c = c_begin; c < c_end; ++c) {
    if (V[c]) {
      const ag_saddle s = R[c];
      if (s.k >= kthr && s.phi >= min_angle && s.phi <= max_angle) {
        if (offset < max_saddles) O[offset] = s;
        ++offset;
      }
    }
  }
  if (tid == 0) {
    n_refined[f] = min(s_total, max_saddles);
    if (s_total > max_saddles) atomicOr(frame_status + f, (uint32_t)AG_FRAME_SADDLE_OVERFLOW);
  }
}

// Result of the saddle entry points: each frame's refined saddles (K4's list, `in_stride` records per
// frame) in the caller's layout (`out_stride` records per frame).  One block per frame.  The count
// is exact, or 0 for a frame whose list K3 / K4 truncated (cluster or saddle overflow); the first
// min(n, cap) records are copied as 32-bit words, so consecutive lanes touch consecutive words
// whatever the 20-byte record boundaries; n > cap sets AG_FRAME_TAG_OVERFLOW.  The callers give
// out_stride >= min(n, cap): an unflagged frame has at most in_stride saddles.
// Frame lists: frame f of the chunk is the caller's frame idx[f] (out, n_out and status_out are
// indexed by it; status_out, if set, receives the frame's final status bits).
constexpr int kSaddlesOutThreads = 256;
constexpr int kSaddleWords = (int)(sizeof(ag_saddle) / sizeof(uint32_t));
static_assert(sizeof(ag_saddle) == 5 * sizeof(uint32_t), "ag_saddle is five 32-bit words");

__global__ void __launch_bounds__(kSaddlesOutThreads)
k_saddles_out(const ag_saddle* __restrict__ refined, int in_stride, const int* __restrict__ n_refined,
              uint32_t* __restrict__ frame_status, ag_saddle* __restrict__ out, int out_stride, int cap,
              int* __restrict__ n_out, const int* __restrict__ idx, uint32_t* __restrict__ status_out) {
  const int f = blockIdx.x;
  const int o = idx ? idx[f] : f;
  const uint32_t st = frame_status[f];
  const int n = (st & (AG_FRAME_CLUSTER_OVERFLOW | AG_FRAME_SADDLE_OVERFLOW)) ? 0 : n_refined[f];
  const int words = min(n, cap) * kSaddleWords;
  const uint32_t* src = reinterpret_cast<const uint32_t*>(refined + (size_t)f * in_stride);
  uint32_t* dst = reinterpret_cast<uint32_t*>(out + (size_t)o * out_stride);
  for (int i = threadIdx.x; i < words; i += kSaddlesOutThreads) dst[i] = src[i];
  if (threadIdx.x == 0) {
    n_out[o] = n;
    const uint32_t st_out = n > cap ? st | AG_FRAME_TAG_OVERFLOW : st;
    if (n > cap) frame_status[f] = st_out;
    if (status_out) status_out[o] = st_out;
  }
}

int launch_saddles_out(const ag_saddle* refined, int in_stride, const int* n_refined, uint32_t* frame_status,
                       int n_frames, ag_saddle* out, int out_stride, int cap, int* n_out, cudaStream_t s,
                       const int* idx, uint32_t* status_out) {
  if (n_frames <= 0) return 0;
  k_saddles_out<<<n_frames, kSaddlesOutThreads, 0, s>>>(refined, in_stride, n_refined, frame_status, out, out_stride,
                                                         cap, n_out, idx, status_out);
  return 1;
}

// The tag twin of k_saddles_out for frame lists: the board search of a chunk writes its tags, counts
// and status bits chunk-locally (`in_stride` records per frame); this copies the count, the status
// bits and the first min(n, cap) records of frame f to the caller's frame idx[f].  One block per frame,
// records copied as 32-bit words.
constexpr int kTagsOutThreads = 128;
constexpr int kTagWords = (int)(sizeof(ag_tag) / sizeof(uint32_t));
static_assert(sizeof(ag_tag) == 9 * sizeof(uint32_t), "ag_tag is nine 32-bit words");

__global__ void __launch_bounds__(kTagsOutThreads)
k_tags_out(const ag_tag* __restrict__ tags, int in_stride, const int* __restrict__ n_tags,
           const uint32_t* __restrict__ frame_status, const int* __restrict__ idx, ag_tag* __restrict__ out, int cap,
           int* __restrict__ n_out, uint32_t* __restrict__ status_out) {
  const int f = blockIdx.x;
  const int o = idx[f];
  const int n = n_tags[f];
  const int words = min(min(n, cap), in_stride) * kTagWords;
  const uint32_t* src = reinterpret_cast<const uint32_t*>(tags + (size_t)f * in_stride);
  uint32_t* dst = reinterpret_cast<uint32_t*>(out + (size_t)o * cap);
  for (int i = threadIdx.x; i < words; i += kTagsOutThreads) dst[i] = src[i];
  if (threadIdx.x == 0) {
    n_out[o] = n;
    if (status_out) status_out[o] = frame_status[f];
  }
}

int launch_tags_out(const ag_tag* tags, int in_stride, const int* n_tags, const uint32_t* frame_status, int n_frames,
                    const int* idx, ag_tag* out, int cap, int* n_out, uint32_t* status_out, cudaStream_t s) {
  if (n_frames <= 0) return 0;
  k_tags_out<<<n_frames, kTagsOutThreads, 0, s>>>(tags, in_stride, n_tags, frame_status, idx, out, cap, n_out,
                                                   status_out);
  return 1;
}

int launch_label_clusters(const uint32_t* mask, const FrameGeom& g, int n_frames, int* parent,
                          int max_clusters, int* acc, float2* centers, int* n_clusters,
                          uint32_t* frame_status, uint32_t* pixlist, int list_cap, int variant,
                          int* fallback, cudaStream_t s) {
  // variant 0: run-based kernel (shared-memory union-find; no per-pixel parents), followed by the
  // pixel-list kernel for the frames it declined; 1: pixel-list kernel for every frame (writes the
  // per-pixel parent array the labels tap reads)
  if (variant == 0 && pixlist && fallback && list_cap >= 2 * kRunCap) {
    const size_t smem = sizeof(int) * (kRunCap + kRowCap + 1);
    if (cudaFuncSetAttribute(k_label_runs, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
      return 0;
    k_label_runs<<<n_frames, kCclThreads, smem, s>>>(mask, g, max_clusters, acc, centers, n_clusters,
                                                     frame_status, pixlist, fallback);
    k_label_clusters<<<n_frames, kCclThreads, 0, s>>>(mask, g, parent, max_clusters, acc, centers,
                                                      n_clusters, frame_status, pixlist, list_cap, fallback);
    return 2;
  }
  k_label_clusters<<<n_frames, kCclThreads, 0, s>>>(mask, g, parent, max_clusters, acc, centers,
                                                    n_clusters, frame_status, pixlist, list_cap, nullptr);
  return 1;
}

int launch_labels_tap(const uint32_t* mask, const FrameGeom& g, const int* parent, int32_t* labels,
                      uint8_t* mask_u8, cudaStream_t s) {
  k_labels_tap<<<(g.n_px + 255) / 256, 256, 0, s>>>(mask, g, parent, labels, mask_u8);
  return 1;
}

int launch_refine_filter(const float* blur, const FrameGeom& g, int n_frames, const float2* centers,
                         const int* n_clusters, int max_clusters, ag_saddle* raw, uint8_t* raw_valid,
                         float min_angle, float max_angle, int max_saddles, ag_saddle* refined,
                         int* n_refined, uint32_t* frame_status, cudaStream_t s) {
  k_refine_filter<<<n_frames, kRefineThreads, 0, s>>>(blur, g, centers, n_clusters, max_clusters, raw,
                                                      raw_valid, min_angle, max_angle, max_saddles,
                                                      refined, n_refined, frame_status);
  return 1;
}

}  // namespace ag
