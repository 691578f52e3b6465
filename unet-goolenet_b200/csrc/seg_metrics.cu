// Segmentation metrics against ground truth (ug_seg_metrics_desc): per image, the confusion counts of the foreground
// sets P = {pred != 0} and G = {gt != 0}, and the Hausdorff distance and its 95th percentile between their surfaces
// (the pixels of a set with a 4-neighbour outside it; outside the image counts as outside), in pixel units.
//
// Seven launches, each over (CTAs, image), none of whose geometry depends on the table (a plan image's host fills it
// after the program is built):
//   sm_init    validates the table entry, resets the image's header and histograms;
//   sm_edges   one pass over pred and gt in bands of rows (one-row halo staged in shared memory): tp / fp / fn, the
//              surface flags of every pixel (workspace byte), |dP|, |dG| and the bounding box of P u G;
//   sm_columns one thread per bounding-box column: the distance to the nearest dG and dP pixel in the column (exact
//              separable EDT, phase 1), packed with the surface flags into one 32-bit word per pixel;
//   sm_rows    one warp per bounding-box row: the lower envelope of the parabolas f(x') + (x - x')^2
//              (Felzenszwalb-Huttenlocher, integer intersection tests) of each direction, built by lane 0 in shared
//              memory and evaluated by all lanes at the row's query pixels only; the squared distance replaces the
//              column distances in the pixel's word.  Linear in the row's width whatever the masks look like;
//   sm_hist1 / sm_hist2 / sm_final  an integer radix select (12 + 11 bits of the 23-bit squared distances) of the
//              order statistics lo = floor(0.95 (n-1)) and hi = min(lo + 1, n - 1) of each direction, then HD and HD95
//              in fp64 with np.percentile's linear method restated operation by operation.
// Every accumulation is an integer (atomics included): the outputs are bit-identical run to run.
#include <cstdint>
#include "common.cuh"
#include "engine.h"

namespace ug {

static constexpr int kSmMaxSide = 8 * 224;  // source sides up to 8*224, as the ragged front-end
static constexpr int kSmThreads = 256;
static constexpr int kSmRows = 8;            // rows per band of sm_edges
static constexpr int kSmColThreads = 128;
static constexpr int kSmRowWarps = 2;
static constexpr int kSmTargetCtas = 4096;
static constexpr int kSmBins1 = 4096;        // key >> 11
static constexpr int kSmBins2 = 2048;        // key & 2047
static constexpr unsigned kSmInf = 0xFFFu;   // "no surface pixel in this column" (sides <= 1792 < 4095)
static constexpr unsigned kSmP = 1u << 30, kSmG = 1u << 31, kSmKey = (1u << 23) - 1;

// Per-image header in the workspace.
struct SmHdr {
  long long off;
  int H, W, ok;
  int x0, y0, x1, y1;        // bounding box of P u G, inclusive (x1 < x0: both sets empty)
  int tp, fp, fn, nP, nG;    // counts, |dP|, |dG|
  unsigned maxk[2];          // largest squared distance of d_PG, d_GP
  int bin[4], rem[4];        // radix select: (direction, lo / hi) -> first-level bin and the rank inside it
};

struct SmWs {
  SmHdr* hdr;
  unsigned* hist1;           // [B][2][kSmBins1]
  unsigned* hist2;           // [B][4][kSmBins2]
  unsigned* word;            // [P]: per pixel, column distances and then the squared distance, with the flag bits
  unsigned char* flags;      // [P]: bit 0 = in dP, bit 1 = in dG
};

static size_t align256(size_t v) { return (v + 255) & ~size_t(255); }

static SmWs ws_layout(void* base, int B, long long px) {
  char* p = static_cast<char*>(base);
  SmWs w;
  w.hdr = reinterpret_cast<SmHdr*>(p);
  p += align256(sizeof(SmHdr) * (size_t)B);
  w.hist1 = reinterpret_cast<unsigned*>(p);
  p += align256(sizeof(unsigned) * 2 * kSmBins1 * (size_t)B);
  w.hist2 = reinterpret_cast<unsigned*>(p);
  p += align256(sizeof(unsigned) * 4 * kSmBins2 * (size_t)B);
  w.word = reinterpret_cast<unsigned*>(p);
  p += align256(sizeof(unsigned) * (size_t)px);
  w.flags = reinterpret_cast<unsigned char*>(p);
  return w;
}

__global__ void __launch_bounds__(kSmThreads) sm_init(ug_seg_metrics_desc d, SmWs w) {
  pdl_wait();
  pdl_launch_dependents();
  const int i = blockIdx.x, tid = threadIdx.x;
  if (tid == 0) {
    SmHdr h = {};
    bool ok = true;
    if (d.index) {
      const ug_ragged_image e = d.index[i];
      h.off = e.px_offset;
      h.H = e.H;
      h.W = e.W;
      ok = h.off >= 0 && h.H >= 1 && h.W >= 1 && h.H <= kSmMaxSide && h.W <= kSmMaxSide && h.off <= d.capacity_px &&
           (long long)h.H * h.W <= d.capacity_px - h.off;
    } else {
      h.H = d.Hs;
      h.W = d.Ws;
      h.off = (long long)i * d.Hs * d.Ws;
    }
    h.ok = ok;
    h.x0 = h.W;
    h.y0 = h.H;
    h.x1 = h.y1 = -1;
    w.hdr[i] = h;
    if (d.status) d.status[i] = ok ? 0 : 1;
  }
  for (int k = tid; k < 2 * kSmBins1; k += kSmThreads) w.hist1[(size_t)i * 2 * kSmBins1 + k] = 0;
  for (int k = tid; k < 4 * kSmBins2; k += kSmThreads) w.hist2[(size_t)i * 4 * kSmBins2 + k] = 0;
}

__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ int warp_min(int v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ int warp_max(int v) {
#pragma unroll
  for (int o = 16; o; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

__global__ void __launch_bounds__(kSmThreads) sm_edges(ug_seg_metrics_desc d, SmWs w) {
  // rows r0-1 .. r0+kSmRows of the band: bit 0 = in P, bit 1 = in G (0 outside the image)
  __shared__ unsigned char stage[(kSmRows + 2) * kSmMaxSide];
  pdl_wait();
  pdl_launch_dependents();
  const int i = blockIdx.y, tid = threadIdx.x, lane = tid & 31;
  const SmHdr h = w.hdr[i];
  if (!h.ok) return;
  const int H = h.H, W = h.W;
  const unsigned char* pred = d.pred + h.off;
  const unsigned char* gt = d.gt + h.off;
  unsigned char* fl = w.flags + h.off;
  int tp = 0, fp = 0, fn = 0, nP = 0, nG = 0, x0 = W, y0 = H, x1 = -1, y1 = -1;
  const int n_bands = (H + kSmRows - 1) / kSmRows;
  for (int band = blockIdx.x; band < n_bands; band += gridDim.x) {
    const int r0 = band * kSmRows, nr = min(kSmRows, H - r0), ns = (nr + 2) * W;
    {
      int r = tid / W, x = tid - r * W;
      for (int k = tid; k < ns; k += kSmThreads) {
        const int y = r0 - 1 + r;
        unsigned char v = 0;
        if (y >= 0 && y < H) {
          const long long p = (long long)y * W + x;
          v = (pred[p] != 0) | (gt[p] != 0) << 1;
        }
        stage[k] = v;
        x += kSmThreads;
        if (x >= W) {
          const int t = x / W;
          r += t;
          x -= t * W;
        }
      }
    }
    __syncthreads();
    const int n = nr * W;
    int r = tid / W, x = tid - r * W;
    for (int k = tid; k < n; k += kSmThreads) {
      const unsigned char* row = stage + (r + 1) * W;
      const unsigned c = row[x];
      const unsigned in = c & row[x - W] & row[x + W] & (x > 0 ? row[x - 1] : 0u) & (x + 1 < W ? row[x + 1] : 0u);
      const unsigned s = c & ~in;  // bit 0: on dP, bit 1: on dG
      fl[(long long)(r0 + r) * W + x] = (unsigned char)s;
      tp += c == 3;
      fp += c == 1;
      fn += c == 2;
      nP += s & 1;
      nG += s >> 1;
      if (c) {
        x0 = min(x0, x);
        x1 = max(x1, x);
        y0 = min(y0, r0 + r);
        y1 = max(y1, r0 + r);
      }
      x += kSmThreads;
      if (x >= W) {
        const int t = x / W;
        r += t;
        x -= t * W;
      }
    }
    __syncthreads();  // the next band overwrites the stage
  }
  tp = warp_sum(tp);
  fp = warp_sum(fp);
  fn = warp_sum(fn);
  nP = warp_sum(nP);
  nG = warp_sum(nG);
  x0 = warp_min(x0);
  y0 = warp_min(y0);
  x1 = warp_max(x1);
  y1 = warp_max(y1);
  if (lane == 0) {
    SmHdr* g = w.hdr + i;
    if (tp) atomicAdd(&g->tp, tp);
    if (fp) atomicAdd(&g->fp, fp);
    if (fn) atomicAdd(&g->fn, fn);
    if (nP) atomicAdd(&g->nP, nP);
    if (nG) atomicAdd(&g->nG, nG);
    if (x1 >= 0) {
      atomicMin(&g->x0, x0);
      atomicMin(&g->y0, y0);
      atomicMax(&g->x1, x1);
      atomicMax(&g->y1, y1);
    }
  }
}

// Phase 1 of the EDT: per bounding-box column, the vertical distance to the nearest dG (bits 0-11) and dP (bits 12-23)
// pixel of the column, kSmInf if there is none; bits 30 / 31 carry the pixel's own dP / dG flags.
__global__ void __launch_bounds__(kSmColThreads) sm_columns(ug_seg_metrics_desc d, SmWs w) {
  pdl_wait();
  pdl_launch_dependents();
  const int i = blockIdx.y;
  const SmHdr h = w.hdr[i];
  const int x = blockIdx.x * kSmColThreads + threadIdx.x;
  if (!h.ok || h.x1 < h.x0 || x > h.x1 - h.x0) return;
  const int W = h.W, bh = h.y1 - h.y0 + 1;
  const long long base = h.off + (long long)h.y0 * W + h.x0 + x;
  const unsigned char* __restrict__ fl = w.flags + base;
  unsigned* __restrict__ wd = w.word + base;
  int lastG = -(1 << 20), lastP = -(1 << 20);
  constexpr int U = 8;  // flags loaded ahead: the loads do not depend on the scan
  for (int y = 0; y < bh; y += U) {
    unsigned char f[U];
#pragma unroll
    for (int u = 0; u < U; ++u) f[u] = y + u < bh ? fl[(long long)(y + u) * W] : 0;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int yy = y + u;
      if (yy < bh) {
        if (f[u] & 2) lastG = yy;
        if (f[u] & 1) lastP = yy;
        const unsigned dg = min(yy - lastG, (int)kSmInf), dp = min(yy - lastP, (int)kSmInf);
        wd[(long long)yy * W] = dg | dp << 12 | (f[u] & 1u) << 30 | (unsigned)(f[u] >> 1) << 31;
      }
    }
  }
  int nextG = 1 << 20, nextP = 1 << 20;
  for (int y = bh - 1; y >= 0; y -= U) {
    unsigned v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) v[u] = y - u >= 0 ? wd[(long long)(y - u) * W] : 0u;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int yy = y - u;
      if (yy >= 0) {
        if (v[u] & kSmG) nextG = yy;
        if (v[u] & kSmP) nextP = yy;
        const unsigned dg = min(v[u] & kSmInf, (unsigned)min(nextG - yy, (int)kSmInf));
        const unsigned dp = min((v[u] >> 12) & kSmInf, (unsigned)min(nextP - yy, (int)kSmInf));
        wd[(long long)yy * W] = dg | dp << 12 | (v[u] & (kSmP | kSmG));
      }
    }
  }
}

// Lower envelope of the parabolas f(q) + (x - q)^2 over the sites q of one row (those with a finite column distance
// c(q) = (row[q] >> shift) & kSmInf, f = c^2), Felzenszwalb-Huttenlocher with exact integer intersection tests.  The
// stack entries are q | c << 16.  Returns the number of entries.
__device__ int sm_envelope(const unsigned* row, int n, int shift, unsigned* st) {
  int k = -1;
  for (int q = 0; q < n; ++q) {
    const int c = (row[q] >> shift) & kSmInf;
    if (c == (int)kSmInf) continue;
    const long long fq = (long long)c * c + (long long)q * q;
    while (k >= 1) {
      // pop v[k] when the intersection of q with v[k] is not right of the intersection of v[k] with v[k-1]
      const int v1 = st[k] & 0xFFFF, c1 = st[k] >> 16, v0 = st[k - 1] & 0xFFFF, c0 = st[k - 1] >> 16;
      const long long f1 = (long long)c1 * c1 + (long long)v1 * v1, f0 = (long long)c0 * c0 + (long long)v0 * v0;
      if ((fq - f1) * (v1 - v0) <= (f1 - f0) * (q - v1)) --k;
      else break;
    }
    st[++k] = (unsigned)q | (unsigned)c << 16;
  }
  return k + 1;
}

__device__ __forceinline__ int sm_par(unsigned e, int x) {
  const int v = e & 0xFFFF, c = e >> 16;
  return c * c + (x - v) * (x - v);
}

// Index of the envelope entry that is lowest at x: the first j with j == n-1 or par(j+1, x) > par(j, x).
__device__ __forceinline__ int sm_locate(const unsigned* st, int n, int x) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (sm_par(st[mid + 1], x) <= sm_par(st[mid], x)) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(32 * kSmRowWarps) sm_rows(ug_seg_metrics_desc d, SmWs w) {
  __shared__ unsigned s_row[kSmRowWarps][kSmMaxSide];
  __shared__ unsigned s_env[kSmRowWarps][2][kSmMaxSide];
  pdl_wait();
  pdl_launch_dependents();
  const int i = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const SmHdr h = w.hdr[i];
  if (!h.ok || h.x1 < h.x0) return;
  const int W = h.W, bw = h.x1 - h.x0 + 1, bh = h.y1 - h.y0 + 1;
  unsigned* row = s_row[warp];
  unsigned* envG = s_env[warp][0];  // sites on dG: queried at the dP pixels (d_PG)
  unsigned* envP = s_env[warp][1];
  const int seg = (bw + 31) / 32, xs = min(bw, lane * seg), xe = min(bw, xs + seg);
  for (int y = blockIdx.x * kSmRowWarps + warp; y < bh; y += gridDim.x * kSmRowWarps) {
    unsigned* g = w.word + h.off + (long long)(h.y0 + y) * W + h.x0;
    unsigned any = 0;
    for (int x = lane; x < bw; x += 32) {
      const unsigned v = g[x];
      row[x] = v;
      any |= v;
    }
    any = __reduce_or_sync(0xffffffffu, any);
    __syncwarp();
    if (!(any & (kSmP | kSmG))) continue;  // no query pixel: the row's words are never read again
    int nG = 0, nP = 0;
    if (lane == 0) {
      if ((any & kSmP) && h.nG) nG = sm_envelope(row, bw, 0, envG);
      if ((any & kSmG) && h.nP) nP = sm_envelope(row, bw, 12, envP);
    }
    nG = __shfl_sync(0xffffffffu, nG, 0);
    nP = __shfl_sync(0xffffffffu, nP, 0);
    __syncwarp();
    // lane l: the columns [xs, xe), read and rewritten in place (the envelopes carry their own column distances); the
    // pointers into the envelopes only move right
    int jG = -1, jP = -1;
    for (int x = xs; x < xe; ++x) {
      const unsigned v = row[x], fl = v & (kSmP | kSmG);
      unsigned key = 0;
      if (fl == kSmP && nG) {
        if (jG < 0) jG = sm_locate(envG, nG, x);
        while (jG + 1 < nG && sm_par(envG[jG + 1], x) <= sm_par(envG[jG], x)) ++jG;
        key = sm_par(envG[jG], x);
      } else if (fl == kSmG && nP) {
        if (jP < 0) jP = sm_locate(envP, nP, x);
        while (jP + 1 < nP && sm_par(envP[jP + 1], x) <= sm_par(envP[jP], x)) ++jP;
        key = sm_par(envP[jP], x);
      }
      row[x] = key | fl;  // a pixel on both surfaces is at distance 0 in both directions
    }
    __syncwarp();
    for (int x = lane; x < bw; x += 32) g[x] = row[x];
    __syncwarp();
  }
}

// Histogram of the first 12 key bits of each direction (query pixels only), and the largest key of each.
__global__ void __launch_bounds__(kSmThreads) sm_hist1(ug_seg_metrics_desc d, SmWs w) {
  __shared__ unsigned hist[2 * kSmBins1];
  pdl_wait();
  pdl_launch_dependents();
  const int i = blockIdx.y, tid = threadIdx.x;
  const SmHdr h = w.hdr[i];
  if (!h.ok || h.x1 < h.x0) return;
  for (int k = tid; k < 2 * kSmBins1; k += kSmThreads) hist[k] = 0;
  __syncthreads();
  const int W = h.W, bw = h.x1 - h.x0 + 1, bh = h.y1 - h.y0 + 1;
  unsigned m0 = 0, m1 = 0;
  for (int y = blockIdx.x; y < bh; y += gridDim.x) {
    const unsigned* g = w.word + h.off + (long long)(h.y0 + y) * W + h.x0;
    for (int x = tid; x < bw; x += kSmThreads) {
      const unsigned v = g[x], key = v & kSmKey;
      if (v & kSmP) {
        atomicAdd(&hist[key >> 11], 1u);
        m0 = max(m0, key);
      }
      if (v & kSmG) {
        atomicAdd(&hist[kSmBins1 + (key >> 11)], 1u);
        m1 = max(m1, key);
      }
    }
  }
  m0 = (unsigned)warp_max((int)m0);
  m1 = (unsigned)warp_max((int)m1);
  if ((tid & 31) == 0) {
    if (m0) atomicMax(&w.hdr[i].maxk[0], m0);
    if (m1) atomicMax(&w.hdr[i].maxk[1], m1);
  }
  __syncthreads();
  unsigned* gh = w.hist1 + (size_t)i * 2 * kSmBins1;
  for (int k = tid; k < 2 * kSmBins1; k += kSmThreads)
    if (hist[k]) atomicAdd(&gh[k], hist[k]);
}

// One warp: the bin of `hist` (nb bins) holding the element of rank `rank` (0-based) and the rank inside that bin.
__device__ void sm_find(const unsigned* hist, int nb, long long rank, int lane, int* bin, int* rem) {
  const int per = nb / 32;
  long long mine = 0;
  for (int k = 0; k < per; ++k) mine += hist[lane * per + k];
  long long incl = mine;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  const long long excl = incl - mine;
  const unsigned hit = __ballot_sync(0xffffffffu, excl <= rank && rank < incl);
  const int src = hit ? __ffs(hit) - 1 : 31;
  if (lane == src) {
    long long c = excl;
    int b = lane * per;
    for (int k = 0; k < per; ++k, ++b) {
      const unsigned n = hist[b];
      if (rank < c + n) break;
      c += n;
    }
    *bin = min(b, lane * per + per - 1);
    *rem = (int)(rank - c);
  }
}

__device__ __forceinline__ void sm_ranks(long long n, long long* lo, long long* hi) {
  const double v = __dmul_rn((double)(n - 1), 0.95);
  *lo = (long long)floor(v);
  *hi = min(*lo + 1, n - 1);
}

// Select the first-level bins of the lo / hi order statistics, then histogram the last 11 bits of the keys in them.
__global__ void __launch_bounds__(kSmThreads) sm_hist2(ug_seg_metrics_desc d, SmWs w) {
  __shared__ unsigned hist[4 * kSmBins2];
  __shared__ int s_bin[4];
  pdl_wait();
  pdl_launch_dependents();
  const int i = blockIdx.y, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const SmHdr h = w.hdr[i];
  if (!h.ok || h.x1 < h.x0) return;
  for (int k = tid; k < 4 * kSmBins2; k += kSmThreads) hist[k] = 0;
  if (warp < 4) {
    const int dir = warp >> 1, n = dir ? h.nG : h.nP;
    int bin = -1, rem = 0;
    if (n > 0) {
      long long lo, hi;
      sm_ranks(n, &lo, &hi);
      sm_find(w.hist1 + ((size_t)i * 2 + dir) * kSmBins1, kSmBins1, (warp & 1) ? hi : lo, lane, &bin, &rem);
    }
    bin = __reduce_max_sync(0xffffffffu, bin);
    rem = __reduce_max_sync(0xffffffffu, rem);
    if (lane == 0) {
      s_bin[warp] = bin;
      if (blockIdx.x == 0) {
        w.hdr[i].bin[warp] = bin;
        w.hdr[i].rem[warp] = rem;
      }
    }
  }
  __syncthreads();
  const int b0 = s_bin[0], b1 = s_bin[1], b2 = s_bin[2], b3 = s_bin[3];
  const int W = h.W, bw = h.x1 - h.x0 + 1, bh = h.y1 - h.y0 + 1;
  for (int y = blockIdx.x; y < bh; y += gridDim.x) {
    const unsigned* g = w.word + h.off + (long long)(h.y0 + y) * W + h.x0;
    for (int x = tid; x < bw; x += kSmThreads) {
      const unsigned v = g[x], key = v & kSmKey;
      const int b = key >> 11, low = key & 2047;
      if (v & kSmP) {
        if (b == b0) atomicAdd(&hist[low], 1u);
        if (b == b1) atomicAdd(&hist[kSmBins2 + low], 1u);
      }
      if (v & kSmG) {
        if (b == b2) atomicAdd(&hist[2 * kSmBins2 + low], 1u);
        if (b == b3) atomicAdd(&hist[3 * kSmBins2 + low], 1u);
      }
    }
  }
  __syncthreads();
  unsigned* gh = w.hist2 + (size_t)i * 4 * kSmBins2;
  for (int k = tid; k < 4 * kSmBins2; k += kSmThreads)
    if (hist[k]) atomicAdd(&gh[k], hist[k]);
}

// np.percentile(sqrt(keys), 95) with numpy's linear method, from the lo / hi order statistics: _lerp(a, b, g) =
// a + (b - a) * g, or b - (b - a) * (1 - g) where g >= 0.5, each operation rounded on its own (no contraction).
__device__ double sm_pct95(long long n, unsigned klo, unsigned khi) {
  long long lo, hi;
  sm_ranks(n, &lo, &hi);
  const double v = __dmul_rn((double)(n - 1), 0.95), g = __dsub_rn(v, (double)lo);
  const double a = __dsqrt_rn((double)klo), b = __dsqrt_rn((double)khi), diff = __dsub_rn(b, a);
  return g >= 0.5 ? __dsub_rn(b, __dmul_rn(diff, __dsub_rn(1.0, g))) : __dadd_rn(a, __dmul_rn(diff, g));
}

__global__ void __launch_bounds__(128) sm_final(ug_seg_metrics_desc d, SmWs w) {
  __shared__ unsigned s_key[4];
  pdl_wait();
  pdl_launch_dependents();
  const int i = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const SmHdr h = w.hdr[i];
  const bool any = h.ok && h.nP > 0 && h.nG > 0;
  if (any) {
    int low = 0, rem = 0;
    sm_find(w.hist2 + ((size_t)i * 4 + warp) * kSmBins2, kSmBins2, w.hdr[i].rem[warp], lane, &low, &rem);
    low = __reduce_max_sync(0xffffffffu, low);
    if (lane == 0) s_key[warp] = (unsigned)w.hdr[i].bin[warp] << 11 | (unsigned)low;
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  const double nan = __longlong_as_double(0x7ff8000000000000LL), inf = __longlong_as_double(0x7ff0000000000000LL);
  double hd = nan, hd95 = nan;
  if (any) {
    hd = __dsqrt_rn((double)max(h.maxk[0], h.maxk[1]));
    hd95 = fmax(sm_pct95(h.nP, s_key[0], s_key[1]), sm_pct95(h.nG, s_key[2], s_key[3]));
  } else if (h.ok && (h.nP > 0 || h.nG > 0)) {
    hd = hd95 = inf;
  }
  d.counts[3LL * i] = h.ok ? h.tp : 0;
  d.counts[3LL * i + 1] = h.ok ? h.fp : 0;
  d.counts[3LL * i + 2] = h.ok ? h.fn : 0;
  d.hd[2LL * i] = hd;
  d.hd[2LL * i + 1] = hd95;
}

int launch_seg_metrics(ug_engine* h, const ug_seg_metrics_desc* d, cudaStream_t s) {
  if (!d->pred || !d->gt || !d->counts || !d->hd || !d->workspace || d->B <= 0 || d->B > 65535 ||
      (d->index ? d->capacity_px <= 0
                : (d->Hs < 1 || d->Ws < 1 || d->Hs > kSmMaxSide || d->Ws > kSmMaxSide)))
    return set_error(h, UG_EINVAL,
                     "seg_metrics: bad args (pred, gt, counts, hd, workspace set, 1 <= B <= 65535, Hs, Ws in [1, %d] "
                     "or a table with capacity_px > 0)",
                     kSmMaxSide);
  const long long px = d->index ? d->capacity_px : (long long)d->B * d->Hs * d->Ws;
  const size_t need = ug_seg_metrics_workspace_bytes(d->B, px);
  if (d->workspace_bytes < need)
    return set_error(h, UG_EINVAL, "seg_metrics: workspace too small (%zu < %zu)", d->workspace_bytes, need);
  const SmWs w = ws_layout(d->workspace, d->B, px);
  // the table is not read here: size the grids for the largest image allowed
  const int hmax = d->index ? kSmMaxSide : d->Hs, wmax = d->index ? kSmMaxSide : d->Ws;
  const int per_img = std::max(1, ceil_div(kSmTargetCtas, d->B));
  const dim3 g_band(std::min(ceil_div(hmax, kSmRows), per_img), d->B);
  const dim3 g_cols(ceil_div(wmax, kSmColThreads), d->B);
  const dim3 g_rows(std::min(ceil_div(hmax, kSmRowWarps), per_img), d->B);
  const dim3 g_hist(std::min(hmax, per_img), d->B);
  h->launches += 7;
  int rc = check_cuda(h, launch_pdl(sm_init, dim3(d->B), kSmThreads, 0, s, *d, w), "seg_metrics init");
  if (rc == UG_OK) rc = check_cuda(h, launch_pdl(sm_edges, g_band, kSmThreads, 0, s, *d, w), "seg_metrics edges");
  if (rc == UG_OK) rc = check_cuda(h, launch_pdl(sm_columns, g_cols, kSmColThreads, 0, s, *d, w), "seg_metrics columns");
  if (rc == UG_OK) rc = check_cuda(h, launch_pdl(sm_rows, g_rows, 32 * kSmRowWarps, 0, s, *d, w), "seg_metrics rows");
  if (rc == UG_OK) rc = check_cuda(h, launch_pdl(sm_hist1, g_hist, kSmThreads, 0, s, *d, w), "seg_metrics hist1");
  if (rc == UG_OK) rc = check_cuda(h, launch_pdl(sm_hist2, g_hist, kSmThreads, 0, s, *d, w), "seg_metrics hist2");
  if (rc == UG_OK) rc = check_cuda(h, launch_pdl(sm_final, dim3(d->B), 128, 0, s, *d, w), "seg_metrics final");
  return rc;
}

}  // namespace ug

extern "C" size_t ug_seg_metrics_workspace_bytes(int B, long long capacity_px) {
  if (B <= 0 || capacity_px <= 0) return 0;
  using namespace ug;
  return align256(sizeof(SmHdr) * (size_t)B) + align256(sizeof(unsigned) * 2 * kSmBins1 * (size_t)B) +
         align256(sizeof(unsigned) * 4 * kSmBins2 * (size_t)B) + align256(sizeof(unsigned) * (size_t)capacity_px) +
         (size_t)capacity_px;
}
