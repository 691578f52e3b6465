// Connected components of a mask (ug_lesions_desc): per image, the components of F = {mask != 0} under 4- or
// 8-connectivity, numbered 1..n in raster order of each component's first pixel (scipy.ndimage.label's numbering), a
// table of the K largest (area descending, ties by label ascending) with exact integer statistics, and the mask of the
// largest one.
//
// The labels buffer is the union-find array: while the op runs it holds image-local raster indices (-1 = background),
// and every root is the smallest index of its tree, so each component's final root is its first pixel whatever order
// the atomics land in.  Nine launches, each over (CTAs, image), none of whose geometry depends on the table:
//   lz_init     validates the table entry, resets the image's header and per-row root counts;
//   lz_local    per 32x32 tile, union-find in shared memory: each pixel starts linked to the first pixel of its row
//               run, then only the upward links a run does not already have through its left part; writes each
//               pixel's tile-local root as an image index and zeroes the pixel's area word;
//   lz_border   the neighbour pairs that cross a tile border (the same reduced link set), lock-free union on the labels
//               buffer (atomicMin links the larger root to the smaller; path halving keeps the chains short);
//   lz_flatten  one warp per row: labels[p] = root(p), component areas at the roots (lanes with one root add once),
//               the number of roots per row;
//   lz_topk     one warp per row: the K largest (area, first pixel) keys of each CTA (warp lists in registers, merged
//               in shared memory);
//   lz_select   per image: merges the CTA lists, marks the K roots with their rank, scans the row counts;
//   lz_rank     one warp per row: label = roots before it in raster order + 1 (row offset + ballot scan), kept at the
//               root with its rank;
//   lz_relabel  one warp per row: labels[p] = label of root(p), the main-lesion mask, and the box, boundary and
//               moment sums of the K ranked components (per-thread runs, shared-memory atomics, then global atomics);
//   lz_final    per image: the K table rows and the count.
// Every accumulation is an integer (atomics included): the outputs are bit-identical run to run.
#include <cstdint>
#include "common.cuh"
#include "engine.h"

namespace ug {

static constexpr int kLzMaxSide = 8 * 224;  // source sides up to 8*224, as the ragged front-end
static constexpr int kLzMaxK = 32;
static constexpr int kLzThreads = 256;
static constexpr int kLzWarps = kLzThreads / 32;
static constexpr int kLzTile = 32;           // lz_local / lz_border tiles of 32 x 32 pixels
static constexpr int kLzTargetCtas = 4096;
static constexpr int kLzLabelBits = 21;      // n <= ceil(1792^2 / 2) < 2^21
static constexpr int kLzAreaBits = 22;       // area <= 1792^2 < 2^22

// Per-image header in the workspace.
struct LzHdr {
  long long off;
  int H, W, ok, n;
  int root[kLzMaxK], area[kLzMaxK];              // the selected components (root = first pixel), rank order
  int x0[kLzMaxK], y0[kLzMaxK], x1[kLzMaxK], y1[kLzMaxK], bnd[kLzMaxK];
  unsigned long long sx[kLzMaxK], sy[kLzMaxK], sxx[kLzMaxK], sxy[kLzMaxK], syy[kLzMaxK];
};

struct LzWs {
  LzHdr* hdr;
  int* rows;                  // [B][kLzMaxSide]: roots per row, then their exclusive prefix
  unsigned long long* cand;   // [B][n_lists][K]: the CTA lists of lz_topk
  int* word;                  // [P]: area at a root, then label | (rank + 1) << kLzLabelBits
  int n_lists;
};

static size_t align256(size_t v) { return (v + 255) & ~size_t(255); }

static int lz_per_img(int B) { return std::max(1, ceil_div(kLzTargetCtas, B)); }

static LzWs ws_layout(void* base, int B, long long px, int K) {
  char* p = static_cast<char*>(base);
  LzWs w;
  w.hdr = reinterpret_cast<LzHdr*>(p);
  p += align256(sizeof(LzHdr) * (size_t)B);
  w.rows = reinterpret_cast<int*>(p);
  p += align256(sizeof(int) * (size_t)kLzMaxSide * B);
  w.cand = reinterpret_cast<unsigned long long*>(p);
  p += align256(sizeof(unsigned long long) * (size_t)lz_per_img(B) * K * B);
  w.word = reinterpret_cast<int*>(p);
  w.n_lists = 0;
  return w;
}

__global__ void __launch_bounds__(kLzThreads) lz_init(ug_lesions_desc d, LzWs w) {
  pdl_wait();
  pdl_launch_dependents();
  const int i = blockIdx.x, tid = threadIdx.x;
  __shared__ int s_ok;
  if (tid == 0) {
    long long off;
    int H, W;
    bool ok = true;
    if (d.index) {
      const ug_ragged_image e = d.index[i];
      off = e.px_offset;
      H = e.H;
      W = e.W;
      ok = off >= 0 && H >= 1 && W >= 1 && H <= kLzMaxSide && W <= kLzMaxSide && off <= d.capacity_px &&
           (long long)H * W <= d.capacity_px - off;
    } else {
      H = d.Hs;
      W = d.Ws;
      off = (long long)i * d.Hs * d.Ws;
    }
    LzHdr* h = w.hdr + i;
    h->off = off;
    h->H = H;
    h->W = W;
    h->ok = ok;
    h->n = 0;
    if (d.status) d.status[i] = ok ? 0 : 1;
    s_ok = ok;
  }
  __syncthreads();
  LzHdr* h = w.hdr + i;
  if (tid < kLzMaxK) {
    h->root[tid] = -1;
    h->area[tid] = 0;
    h->x0[tid] = h->y0[tid] = kLzMaxSide;
    h->x1[tid] = h->y1[tid] = -1;
    h->bnd[tid] = 0;
    h->sx[tid] = h->sy[tid] = h->sxx[tid] = h->sxy[tid] = h->syy[tid] = 0;
  }
  if (s_ok)
    for (int k = tid; k < kLzMaxSide; k += kLzThreads) w.rows[(size_t)i * kLzMaxSide + k] = 0;
}

// Union-find on an int array whose roots are their own index; every link goes from the larger root to the smaller.
__device__ __forceinline__ int lz_find_shared(const volatile int* L, int x) {
  int p = L[x];
  while (p != x) {
    x = p;
    p = L[x];
  }
  return x;
}

// As lz_find_shared, halving the path (see lz_find_halve for why the plain stores are safe).
__device__ __forceinline__ int lz_find_shared_halve(volatile int* L, int x) {
  while (true) {
    const int p = L[x];
    if (p == x) return x;
    const int g = L[p];
    if (g == p) return p;
    L[x] = g;
    x = g;
  }
}

__device__ void lz_union_shared(int* L, int a, int b) {
  volatile int* V = L;
  while (true) {
    a = lz_find_shared_halve(V, a);
    b = lz_find_shared_halve(V, b);
    if (a == b) return;
    if (a < b) {
      const int old = atomicMin(&L[b], a);
      if (old == b) return;
      b = old;
    } else {
      const int old = atomicMin(&L[a], b);
      if (old == a) return;
      a = old;
    }
  }
}

// Root of x in the labels buffer, halving the path on the way: a stored value is always an ancestor of the node, so a
// halving store that races a link only loses a link whose union is then retried (the atomicMin saw a non-root).
__device__ __forceinline__ int lz_find_halve(int* L, int x) {
  while (true) {
    const int p = __ldcg(L + x);
    if (p == x) return x;
    const int g = __ldcg(L + p);
    if (g == p) return p;
    __stcg(L + x, g);
    x = g;
  }
}

__device__ void lz_union_global(int* L, int a, int b) {
  while (true) {
    a = lz_find_halve(L, a);
    b = lz_find_halve(L, b);
    if (a == b) return;
    if (a < b) {
      const int old = atomicMin(&L[b], a);
      if (old == b) return;
      b = old;
    } else {
      const int old = atomicMin(&L[a], b);
      if (old == a) return;
      a = old;
    }
  }
}

__global__ void __launch_bounds__(kLzThreads) lz_local(ug_lesions_desc d, LzWs w) {
  __shared__ int s_L[kLzTile * kLzTile];
  pdl_wait();
  pdl_launch_dependents();
  const int i = blockIdx.y, tid = threadIdx.x, lx = tid & (kLzTile - 1), ly0 = tid / kLzTile;
  const LzHdr* hp = w.hdr + i;
  if (!hp->ok) return;
  const long long off = hp->off;
  const int H = hp->H, W = hp->W;
  const unsigned char* m = d.mask + off;
  int* L = d.labels + off;
  int* A = w.word + off;
  const int tx = (W + kLzTile - 1) / kLzTile, n_tiles = tx * ((H + kLzTile - 1) / kLzTile);
  constexpr int kPer = kLzTile * kLzTile / kLzThreads;
  for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const int x0 = (t % tx) * kLzTile, y0 = (t / tx) * kLzTile;
    const int tw = min(kLzTile, W - x0), th = min(kLzTile, H - y0);
    // a warp holds one tile row: each pixel starts linked to the first pixel of its horizontal run
    bool fg[kPer];
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      const int ly = ly0 + k * (kLzThreads / kLzTile), li = ly * kLzTile + lx;
      fg[k] = lx < tw && ly < th && m[(long long)(y0 + ly) * W + x0 + lx] != 0;
      const unsigned z = ~__ballot_sync(0xffffffffu, fg[k]) & ((1u << lx) - 1);
      s_L[li] = fg[k] ? ly * kLzTile + (z ? 32 - __clz(z) : 0) : -1;
    }
    __syncthreads();
    // only the links a run does not already have through its left part: a pixel whose left neighbour is in F reaches
    // that neighbour's upper neighbours through it
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      const int ly = ly0 + k * (kLzThreads / kLzTile), li = ly * kLzTile + lx;
      if (!fg[k] || ly == 0) continue;
      const bool left = lx > 0 && s_L[li - 1] >= 0, up = s_L[li - kLzTile] >= 0;
      const bool ul = lx > 0 && s_L[li - kLzTile - 1] >= 0, ur = lx + 1 < tw && s_L[li - kLzTile + 1] >= 0;
      if (d.connectivity == 8) {
        if (!left && up) lz_union_shared(s_L, li, li - kLzTile);
        if (!left && !up && ul) lz_union_shared(s_L, li, li - kLzTile - 1);
        if (!up && ur) lz_union_shared(s_L, li, li - kLzTile + 1);
      } else if (up && !(left && ul)) {
        lz_union_shared(s_L, li, li - kLzTile);
      }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
      const int ly = ly0 + k * (kLzThreads / kLzTile), li = ly * kLzTile + lx;
      if (lx < tw && ly < th) {
        const long long p = (long long)(y0 + ly) * W + x0 + lx;
        int v = -1;
        if (fg[k]) {
          const int r = lz_find_shared(s_L, li);
          v = (y0 + r / kLzTile) * W + x0 + (r % kLzTile);
        }
        L[p] = v;
        A[p] = 0;
      }
    }
    __syncthreads();  // the next tile overwrites s_L
  }
}

__global__ void __launch_bounds__(kLzThreads) lz_border(ug_lesions_desc d, LzWs w) {
  pdl_wait();
  pdl_launch_dependents();
  const int i = blockIdx.y, tid = threadIdx.x;
  const LzHdr* hp = w.hdr + i;
  if (!hp->ok) return;
  const int H = hp->H, W = hp->W;
  int* L = d.labels + hp->off;
  const bool c8 = d.connectivity == 8;
  const int tx = (W + kLzTile - 1) / kLzTile, n_tiles = tx * ((H + kLzTile - 1) / kLzTile);
  // per tile: threads 0..31 the first row, 32..63 the first column, 64..95 the last column; each pixel unions with
  // its backward neighbours (left, up, up-left, up-right) that lie in another tile
  for (int t = blockIdx.x * (kLzThreads / 96) + tid / 96; t < n_tiles; t += gridDim.x * (kLzThreads / 96)) {
    if (tid >= (kLzThreads / 96) * 96) break;
    const int x0 = (t % tx) * kLzTile, y0 = (t / tx) * kLzTile;
    const int tw = min(kLzTile, W - x0), th = min(kLzTile, H - y0);
    const int role = (tid % 96) / 32, j = tid & 31;
    int x, y;
    if (role == 0) {
      if (j >= tw) continue;
      x = x0 + j;
      y = y0;
    } else {
      if (j >= th) continue;
      x = role == 1 ? x0 : x0 + tw - 1;
      y = y0 + j;
    }
    const int p = y * W + x;
    if (L[p] < 0) continue;
    const int tileL = x0, tileR = x0 + tw - 1;
    // a pixel whose left neighbour is in F reaches that neighbour's upper neighbours through it (the left neighbour
    // is in this tile's top row or is a last-column pixel of the tile to the left, whose crossing links are made
    // here); a last-column pixel reaches its upper-right neighbour through its upper or right neighbour when either
    // is in F (their links to the right tile are that tile's first-column links)
    const bool left = x > 0 && L[p - 1] >= 0;
    if (left && x == tileL) lz_union_global(L, p, p - 1);
    if (y > 0) {
      const bool up = L[p - W] >= 0, ul = x > 0 && L[p - W - 1] >= 0, ur = x + 1 < W && L[p - W + 1] >= 0;
      if (y == y0) {
        if (c8) {
          if (!left && up) lz_union_global(L, p, p - W);
          if (!left && !up && ul) lz_union_global(L, p, p - W - 1);
          if (!up && ur) lz_union_global(L, p, p - W + 1);
        } else if (up && !(left && ul)) {
          lz_union_global(L, p, p - W);
        }
      } else if (c8) {
        if (x == tileL && !left && ul) lz_union_global(L, p, p - W - 1);
        if (x == tileR && ur && !up && !(x + 1 < W && L[p + 1] >= 0)) lz_union_global(L, p, p - W + 1);
      }
    }
  }
}

__global__ void __launch_bounds__(kLzThreads) lz_flatten(ug_lesions_desc d, LzWs w) {
  pdl_wait();
  pdl_launch_dependents();
  const int i = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const LzHdr* hp = w.hdr + i;
  if (!hp->ok) return;
  const int H = hp->H, W = hp->W;
  int* L = d.labels + hp->off;
  int* A = w.word + hp->off;
  for (int y = blockIdx.x * kLzWarps + warp; y < H; y += gridDim.x * kLzWarps) {
    int roots = 0;
    for (int x0 = 0; x0 < W; x0 += 32) {
      const int x = x0 + lane, p = y * W + x;
      int r = -1;
      if (x < W && L[p] >= 0) {
        // read-only find: the stores of this pass are roots, so a racing read sees an ancestor either way
        r = p;
        int q = L[r];
        while (q != r) {
          r = q;
          q = L[r];
        }
        L[p] = r;
      }
      const unsigned act = __ballot_sync(0xffffffffu, r >= 0);
      roots += __popc(__ballot_sync(0xffffffffu, r >= 0 && r == p));
      if (r >= 0) {
        const unsigned grp = __match_any_sync(act, r);
        if (lane == __ffs(grp) - 1) atomicAdd(&A[r], __popc(grp));
      }
    }
    if (lane == 0) w.rows[(size_t)i * kLzMaxSide + y] = roots;
  }
}

// Warp-wide sorted list of the K largest keys (lane j holds the j-th, 0 = empty): inserts the candidates of the lanes
// whose key beats the K-th.  Keys are unique (they carry the root), so the order is total.
__device__ __forceinline__ unsigned long long lz_insert(unsigned long long list, unsigned long long cand, int K,
                                                        int lane) {
  unsigned long long thr = __shfl_sync(0xffffffffu, list, K - 1);
  unsigned m = __ballot_sync(0xffffffffu, cand > thr);
  while (m) {
    const int src = __ffs(m) - 1;
    const unsigned long long c = __shfl_sync(0xffffffffu, cand, src);
    const int pos = __popc(__ballot_sync(0xffffffffu, list > c));
    const unsigned long long up = __shfl_up_sync(0xffffffffu, list, 1);
    if (lane == pos) list = c;
    else if (lane > pos) list = up;
    if (lane >= K) list = 0;
    thr = __shfl_sync(0xffffffffu, list, K - 1);
    m &= ~(1u << src);
    m &= __ballot_sync(0xffffffffu, cand > thr);
  }
  return list;
}

__device__ __forceinline__ unsigned long long lz_key(int area, int root) {
  return (unsigned long long)area << 32 | (0xFFFFFFFFu - (unsigned)root);
}

__global__ void __launch_bounds__(kLzThreads) lz_topk(ug_lesions_desc d, LzWs w) {
  __shared__ unsigned long long s_list[kLzWarps][32];
  pdl_wait();
  pdl_launch_dependents();
  const int i = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, K = d.K;
  const LzHdr* hp = w.hdr + i;
  if (!hp->ok) return;
  const int H = hp->H, W = hp->W;
  const int* L = d.labels + hp->off;
  const int* A = w.word + hp->off;
  unsigned long long list = 0;
  for (int y = blockIdx.x * kLzWarps + warp; y < H; y += gridDim.x * kLzWarps)
    for (int x0 = 0; x0 < W; x0 += 32) {
      const int x = x0 + lane, p = y * W + x;
      const unsigned long long c = x < W && L[p] == p ? lz_key(A[p], p) : 0;
      list = lz_insert(list, c, K, lane);
    }
  s_list[warp][lane] = list;
  __syncthreads();
  if (warp != 0) return;
  for (int k = 1; k < kLzWarps; ++k) list = lz_insert(list, s_list[k][lane], K, lane);
  if (lane < K) w.cand[((size_t)i * w.n_lists + blockIdx.x) * K + lane] = list;
}

__global__ void __launch_bounds__(kLzThreads) lz_select(ug_lesions_desc d, LzWs w) {
  __shared__ int s_sum[kLzThreads];
  pdl_wait();
  pdl_launch_dependents();
  const int i = blockIdx.x, tid = threadIdx.x, K = d.K;
  LzHdr* hp = w.hdr + i;
  if (!hp->ok) return;
  const int H = hp->H;
  if (tid < 32) {
    unsigned long long list = 0;
    for (int l = 0; l < w.n_lists; ++l) {
      const unsigned long long c = tid < K ? w.cand[((size_t)i * w.n_lists + l) * K + tid] : 0;
      list = lz_insert(list, c, K, tid);
    }
    if (tid < K && list) {
      const int root = (int)(0xFFFFFFFFu - (unsigned)list), area = (int)(list >> 32);
      hp->root[tid] = root;
      hp->area[tid] = area;
      w.word[hp->off + root] = area | (tid + 1) << kLzAreaBits;
    }
  }
  // exclusive prefix of the roots per row: each thread a run of consecutive rows
  int* rows = w.rows + (size_t)i * kLzMaxSide;
  constexpr int kRun = (kLzMaxSide + kLzThreads - 1) / kLzThreads;
  const int r0 = tid * kRun;
  int v[kRun], sum = 0;
#pragma unroll
  for (int k = 0; k < kRun; ++k) {
    v[k] = r0 + k < H ? rows[r0 + k] : 0;
    sum += v[k];
  }
  s_sum[tid] = sum;
  __syncthreads();
  for (int o = 1; o < kLzThreads; o <<= 1) {
    const int t = tid >= o ? s_sum[tid - o] : 0;
    __syncthreads();
    s_sum[tid] += t;
    __syncthreads();
  }
  int run = s_sum[tid] - sum;
#pragma unroll
  for (int k = 0; k < kRun; ++k) {
    if (r0 + k < H) rows[r0 + k] = run;
    run += v[k];
  }
  if (tid == kLzThreads - 1) hp->n = s_sum[tid];
}

__global__ void __launch_bounds__(kLzThreads) lz_rank(ug_lesions_desc d, LzWs w) {
  pdl_wait();
  pdl_launch_dependents();
  const int i = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const LzHdr* hp = w.hdr + i;
  if (!hp->ok) return;
  const int H = hp->H, W = hp->W;
  const int* L = d.labels + hp->off;
  int* A = w.word + hp->off;
  for (int y = blockIdx.x * kLzWarps + warp; y < H; y += gridDim.x * kLzWarps) {
    int base = w.rows[(size_t)i * kLzMaxSide + y];
    for (int x0 = 0; x0 < W; x0 += 32) {
      const int x = x0 + lane, p = y * W + x;
      const bool root = x < W && L[p] == p;
      const unsigned b = __ballot_sync(0xffffffffu, root);
      if (root) {
        const int label = base + __popc(b & ((1u << lane) - 1)) + 1;
        A[p] = label | (A[p] >> kLzAreaBits) << kLzLabelBits;
      }
      base += __popc(b);
    }
  }
}

// One thread's running sums for one ranked component, flushed to shared memory when the component changes.
struct LzRun {
  int slot, x0, y0, x1, y1, bnd;
  unsigned long long sx, sy, sxx, sxy, syy;
};

__global__ void __launch_bounds__(kLzThreads) lz_relabel(ug_lesions_desc d, LzWs w) {
  __shared__ int s_box[5][kLzMaxK];  // x0, y0, x1, y1, boundary
  __shared__ unsigned long long s_sum[5][kLzMaxK];
  __shared__ int s_any;
  pdl_wait();
  pdl_launch_dependents();
  const int i = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  LzHdr* hp = w.hdr + i;
  if (!hp->ok) return;
  const int H = hp->H, W = hp->W;
  const unsigned char* m = d.mask + hp->off;
  int* L = d.labels + hp->off;
  const int* A = w.word + hp->off;
  unsigned char* mm = d.main_mask ? d.main_mask + hp->off : nullptr;
  if (tid < kLzMaxK) {
    s_box[0][tid] = s_box[1][tid] = kLzMaxSide;
    s_box[2][tid] = s_box[3][tid] = -1;
    s_box[4][tid] = 0;
    for (int k = 0; k < 5; ++k) s_sum[k][tid] = 0;
  }
  if (tid == 0) s_any = 0;
  __syncthreads();
  LzRun run;
  run.slot = -1;
  auto flush = [&]() {
    if (run.slot < 0) return;
    const int s = run.slot;
    atomicMin(&s_box[0][s], run.x0);
    atomicMin(&s_box[1][s], run.y0);
    atomicMax(&s_box[2][s], run.x1);
    atomicMax(&s_box[3][s], run.y1);
    atomicAdd(&s_box[4][s], run.bnd);
    atomicAdd(&s_sum[0][s], run.sx);
    atomicAdd(&s_sum[1][s], run.sy);
    atomicAdd(&s_sum[2][s], run.sxx);
    atomicAdd(&s_sum[3][s], run.sxy);
    atomicAdd(&s_sum[4][s], run.syy);
    s_any = 1;
  };
  for (int y = blockIdx.x * kLzWarps + warp; y < H; y += gridDim.x * kLzWarps) {
    for (int x = lane; x < W; x += 32) {
      const int p = y * W + x;
      const int r = L[p];
      int slot = -1;
      if (r >= 0) {
        const int v = A[r];
        L[p] = v & ((1 << kLzLabelBits) - 1);
        slot = (v >> kLzLabelBits) - 1;
      } else {
        L[p] = 0;
      }
      if (mm) mm[p] = slot == 0;
      if (slot < 0) continue;
      const bool edge = x == 0 || x + 1 == W || y == 0 || y + 1 == H || !m[p - 1] || !m[p + 1] || !m[p - W] ||
                        !m[p + W];
      if (slot != run.slot) {
        flush();
        run.slot = slot;
        run.x0 = run.x1 = x;
        run.y0 = run.y1 = y;
        run.bnd = 0;
        run.sx = run.sy = run.sxx = run.sxy = run.syy = 0;
      }
      run.x0 = min(run.x0, x);
      run.x1 = max(run.x1, x);
      run.y0 = min(run.y0, y);
      run.y1 = max(run.y1, y);
      run.bnd += edge;
      run.sx += (unsigned)x;
      run.sy += (unsigned)y;
      run.sxx += (unsigned long long)x * x;
      run.sxy += (unsigned long long)x * y;
      run.syy += (unsigned long long)y * y;
    }
  }
  flush();
  __syncthreads();
  if (!s_any || tid >= d.K || s_box[2][tid] < 0) return;
  atomicMin(&hp->x0[tid], s_box[0][tid]);
  atomicMin(&hp->y0[tid], s_box[1][tid]);
  atomicMax(&hp->x1[tid], s_box[2][tid]);
  atomicMax(&hp->y1[tid], s_box[3][tid]);
  atomicAdd(&hp->bnd[tid], s_box[4][tid]);
  atomicAdd(&hp->sx[tid], s_sum[0][tid]);
  atomicAdd(&hp->sy[tid], s_sum[1][tid]);
  atomicAdd(&hp->sxx[tid], s_sum[2][tid]);
  atomicAdd(&hp->sxy[tid], s_sum[3][tid]);
  atomicAdd(&hp->syy[tid], s_sum[4][tid]);
}

__global__ void __launch_bounds__(32) lz_final(ug_lesions_desc d, LzWs w) {
  pdl_wait();
  pdl_launch_dependents();
  const int i = blockIdx.x, s = threadIdx.x;
  const LzHdr* hp = w.hdr + i;
  const bool ok = hp->ok;
  if (s == 0) d.count[i] = ok ? hp->n : 0;
  if (s >= d.K) return;
  ug_lesion e = {};
  if (ok && hp->root[s] >= 0) {
    e.label = w.word[hp->off + hp->root[s]] & ((1 << kLzLabelBits) - 1);
    e.area = hp->area[s];
    e.x0 = hp->x0[s];
    e.y0 = hp->y0[s];
    e.x1 = hp->x1[s] + 1;
    e.y1 = hp->y1[s] + 1;
    e.boundary = hp->bnd[s];
    e.sx = (long long)hp->sx[s];
    e.sy = (long long)hp->sy[s];
    e.sxx = (long long)hp->sxx[s];
    e.sxy = (long long)hp->sxy[s];
    e.syy = (long long)hp->syy[s];
  }
  d.lesions[(size_t)i * d.K + s] = e;
}

int launch_lesions(ug_engine* h, const ug_lesions_desc* d, cudaStream_t s) {
  if (!d->mask || !d->labels || !d->lesions || !d->count || !d->workspace || d->B <= 0 || d->B > 65535 ||
      (d->connectivity != 4 && d->connectivity != 8) || d->K < 1 || d->K > kLzMaxK ||
      (d->index ? d->capacity_px <= 0
                : (d->Hs < 1 || d->Ws < 1 || d->Hs > kLzMaxSide || d->Ws > kLzMaxSide)))
    return set_error(h, UG_EINVAL,
                     "lesions: bad args (mask, labels, lesions, count, workspace set, 1 <= B <= 65535, connectivity 4 "
                     "or 8, 1 <= K <= %d, Hs, Ws in [1, %d] or a table with capacity_px > 0)",
                     kLzMaxK, kLzMaxSide);
  const long long px = d->index ? d->capacity_px : (long long)d->B * d->Hs * d->Ws;
  const size_t need = ug_lesions_workspace_bytes(d->B, px, d->K);
  if (d->workspace_bytes < need)
    return set_error(h, UG_EINVAL, "lesions: workspace too small (%zu < %zu)", d->workspace_bytes, need);
  LzWs w = ws_layout(d->workspace, d->B, px, d->K);
  // the table is not read here: size the grids for the largest image allowed
  const int hmax = d->index ? kLzMaxSide : d->Hs, wmax = d->index ? kLzMaxSide : d->Ws;
  const int per_img = lz_per_img(d->B);
  const int tiles = ceil_div(hmax, kLzTile) * ceil_div(wmax, kLzTile);
  const dim3 g_tiles(std::min(tiles, per_img), d->B);
  const dim3 g_border(std::min(ceil_div(tiles, kLzThreads / 96), per_img), d->B);
  const dim3 g_rows(std::min(ceil_div(hmax, kLzWarps), per_img), d->B);
  w.n_lists = (int)g_rows.x;
  h->launches += 9;
  int rc = check_cuda(h, launch_pdl(lz_init, dim3(d->B), kLzThreads, 0, s, *d, w), "lesions init");
  if (rc == UG_OK) rc = check_cuda(h, launch_pdl(lz_local, g_tiles, kLzThreads, 0, s, *d, w), "lesions local");
  if (rc == UG_OK) rc = check_cuda(h, launch_pdl(lz_border, g_border, kLzThreads, 0, s, *d, w), "lesions border");
  if (rc == UG_OK) rc = check_cuda(h, launch_pdl(lz_flatten, g_rows, kLzThreads, 0, s, *d, w), "lesions flatten");
  if (rc == UG_OK) rc = check_cuda(h, launch_pdl(lz_topk, g_rows, kLzThreads, 0, s, *d, w), "lesions topk");
  if (rc == UG_OK) rc = check_cuda(h, launch_pdl(lz_select, dim3(d->B), kLzThreads, 0, s, *d, w), "lesions select");
  if (rc == UG_OK) rc = check_cuda(h, launch_pdl(lz_rank, g_rows, kLzThreads, 0, s, *d, w), "lesions rank");
  if (rc == UG_OK) rc = check_cuda(h, launch_pdl(lz_relabel, g_rows, kLzThreads, 0, s, *d, w), "lesions relabel");
  if (rc == UG_OK) rc = check_cuda(h, launch_pdl(lz_final, dim3(d->B), 32, 0, s, *d, w), "lesions final");
  return rc;
}

}  // namespace ug

extern "C" size_t ug_lesions_workspace_bytes(int B, long long capacity_px, int K) {
  using namespace ug;
  if (B <= 0 || capacity_px <= 0 || K < 1 || K > kLzMaxK) return 0;
  return align256(sizeof(LzHdr) * (size_t)B) + align256(sizeof(int) * (size_t)kLzMaxSide * B) +
         align256(sizeof(unsigned long long) * (size_t)lz_per_img(B) * K * B) + sizeof(int) * (size_t)capacity_px;
}
