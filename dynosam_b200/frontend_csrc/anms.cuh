// anms.cuh -- AdaptiveNonMaximumSuppression(RangeTree) on the device (included by frontend.cu).
//
// The reference (NonMaximumSupression.cc:45-93 -> anms::RangeTree, anms.cc:278-362) ranks the key-points with
// cv::sortIdx(responses, SORT_DESCENDING) and walks them greedily for each width of a binary search.  At both call sites
// every response is equal, so the rank is a permutation that depends only on n (anms_tie_source), and the walk is a
// sequential greedy pass: a point that is not yet suppressed is selected and suppresses every point whose truncated cell
// lies in the inclusive box [max(0, (int)(x - w)), (int)(x + w)] x [max(0, (int)(y - w)), (int)(y + w)] (float bounds).
//
// One CTA per list: the list is gathered in walk order, warp 0 runs the greedy pass in 32-point chunks over a
// suppression bitmap of the list's bounding box of cells, and the whole binary search runs in the CTA.  Points and
// bitmap live in shared memory when they fit, in global scratch otherwise.
#pragma once
#include <climits>
#include <cmath>
#include <cstdint>

// cv::sortIdx over n equal keys, descending: libstdc++'s introsort on an all-equal range (each level swaps `first` with
// `mid`, reverses [first + 1, last), recurses on [cut, last) and loops on [first, cut) while more than 16 remain; the
// insertion-sort tail moves nothing), then OpenCV reverses the index row.  Returns the input index at walk position k,
// in O(log n): the ranges containing the position are found top-down, the level maps are undone bottom-up.
__host__ __device__ inline int anms_tie_source(int n, int k) {
  int fs[40], ls[40], depth = 0;
  const int p = n - 1 - k;
  int first = 0, last = n;
  while (last - first > 16) {
    const int cut = first + 1 + (last - first - 1)/2;
    fs[depth] = first; ls[depth] = last; depth++;
    if (p >= cut) first = cut; else last = cut;
  }
  int q = p;
  while (depth > 0) {
    depth--;
    const int f = fs[depth], l = ls[depth], mid = f + (l - f)/2;
    if (q > f) q = f + l - q;                 // undo the reversal of [f + 1, l)
    if (q == f) q = mid; else if (q == mid) q = f;   // undo swap(first, mid)
  }
  return q;
}

// double -> int as x86-64 cvttsd2si (what the reference's implicit conversions compile to): NaN / out of range -> INT_MIN
__host__ __device__ inline int anms_c_int(double v) { return (v != v || v >= 2147483648.0 || v < -2147483648.0) ? INT_MIN : (int)v; }

// anms.cc:281-310 with C semantics (K >= 1; K = 1 gives high = INT_MIN and therefore an empty result)
struct AnmsSearch { int high, low; unsigned kmin, kmax; };
__host__ __device__ inline AnmsSearch anms_search_init(int n, int K, float tolerance, int cols, int rows) {
  AnmsSearch s;
  const int exp1 = rows + cols + 2*K;
  const long long exp2 = (long long)4*cols + (long long)4*K + (long long)4*rows*K + (long long)rows*rows + (long long)cols*cols -
                         (long long)2*rows*cols + (long long)4*rows*cols*K;
  const double exp3 = sqrt((double)exp2), exp4 = (double)(K - 1);
  const double sol1 = -round((exp1 + exp3)/exp4), sol2 = -round((exp1 - exp3)/exp4);
  s.high = anms_c_int(sol1 > sol2 ? sol1 : sol2);
  s.low = anms_c_int(floor(sqrt((double)n/K)));
  const float kf = (float)K, kt = kf*tolerance;              // tolerance is float: Kmin / Kmax are rounded in fp32
  s.kmin = (unsigned)roundf(kf - kt); s.kmax = (unsigned)roundf(kf + kt);
  return s;
}

constexpr int ANMS_THREADS = 256;
struct AnmsArgs {
  const int* off; const int* cnt; const int* K;    // per list: first element, length, number of points wanted
  const float* xy;                                 // float coordinates xy[off + i][2], or (xy == nullptr)
  const int* pix; int W;                           // linear pixel indices pix[off + i] of a W-wide image
  float tolerance; int cols, rows;
  float2* g_pts;                                   // global fallbacks: points at off, bitmap at bm_off[list]
  uint32_t* g_bm; const long long* bm_off;
  int* g_sel; long long sel_stride;                // two selection buffers (this width, previous width) at off
  int* out; int* out_n;                            // selected input indices (local to the list), in selection order
  int smem_bytes;
};

__device__ __forceinline__ float2 anms_point(const AnmsArgs& a, int off, int i) {
  if (a.xy) return make_float2(a.xy[2*(size_t)(off + i)], a.xy[2*(size_t)(off + i) + 1]);
  const int p = a.pix[off + i];
  return make_float2((float)(p % a.W), (float)(p / a.W));
}

__global__ void __launch_bounds__(ANMS_THREADS) anms_range_tree_kernel(AnmsArgs a) {
  extern __shared__ __align__(16) unsigned char anms_smem[];
  __shared__ int s_bx0, s_bx1, s_by0, s_by1, s_cnt;
  const int l = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = a.cnt[l], off = a.off[l], K = a.K[l];
  if (n == 0 || K <= 0) { if (tid == 0) a.out_n[l] = 0; return; }     // K = 0: no features (the reference is undefined there)
  // bounding box of the truncated cells
  int bx0 = INT_MAX, bx1 = -1, by0 = INT_MAX, by1 = -1;
  for (int i = tid; i < n; i += ANMS_THREADS) {
    const float2 p = anms_point(a, off, i);
    const int cx = (int)p.x, cy = (int)p.y;
    bx0 = min(bx0, cx); bx1 = max(bx1, cx); by0 = min(by0, cy); by1 = max(by1, cy);
  }
  for (int o = 16; o > 0; o >>= 1) {
    bx0 = min(bx0, __shfl_xor_sync(0xffffffffu, bx0, o)); bx1 = max(bx1, __shfl_xor_sync(0xffffffffu, bx1, o));
    by0 = min(by0, __shfl_xor_sync(0xffffffffu, by0, o)); by1 = max(by1, __shfl_xor_sync(0xffffffffu, by1, o));
  }
  if (tid == 0) { s_bx0 = INT_MAX; s_bx1 = -1; s_by0 = INT_MAX; s_by1 = -1; }
  __syncthreads();
  if (lane == 0) { atomicMin(&s_bx0, bx0); atomicMax(&s_bx1, bx1); atomicMin(&s_by0, by0); atomicMax(&s_by1, by1); }
  __syncthreads();
  bx0 = s_bx0; bx1 = s_bx1; by0 = s_by0; by1 = s_by1;
  const int bwords = ((bx1 - bx0) >> 5) + 1, bh = by1 - by0 + 1;
  const long long words = (long long)bwords*bh, bm_bytes = 4*words, pt_bytes = 8LL*n;
  float2* pts; uint32_t* bm;
  if (bm_bytes + pt_bytes <= a.smem_bytes) { pts = (float2*)anms_smem; bm = (uint32_t*)(anms_smem + pt_bytes); }
  else if (bm_bytes <= a.smem_bytes) { bm = (uint32_t*)anms_smem; pts = a.g_pts + off; }
  else if (pt_bytes <= a.smem_bytes) { pts = (float2*)anms_smem; bm = a.g_bm + a.bm_off[l]; }
  else { pts = a.g_pts + off; bm = a.g_bm + a.bm_off[l]; }
  for (int k = tid; k < n; k += ANMS_THREADS) pts[k] = anms_point(a, off, anms_tie_source(n, k));   // walk order

  const AnmsSearch S = anms_search_init(n, K, a.tolerance, a.cols, a.rows);
  int high = S.high, low = S.low, prevwidth = -1, prev_cnt = 0, final_cnt = 0;
  int* cur = a.g_sel + off; int* prev = a.g_sel + a.sel_stride + off; const int* fin = prev;
  for (;;) {
    const int width = low + (int)((unsigned)high - (unsigned)low)/2;
    if (width == prevwidth || low > high) { fin = prev; final_cnt = prev_cnt; break; }   // the previous iteration's selection
    for (long long i = tid; i < words; i += ANMS_THREADS) bm[i] = 0u;
    __syncthreads();
    if (warp == 0) {
      const float wf = (float)width;
      int cnt = 0;
      for (int base = 0; base < n; base += 32) {
        const int k = base + lane;
        float x = 0.f, y = 0.f; int cx = 0, cy = 0; bool alive = false;
        if (k < n) {
          const float2 p = pts[k]; x = p.x; y = p.y; cx = (int)x; cy = (int)y;
          const int rx = cx - bx0, ry = cy - by0;
          alive = ((bm[(size_t)ry*bwords + (rx >> 5)] >> (rx & 31)) & 1u) == 0u;
        }
        unsigned m = __ballot_sync(0xffffffffu, alive);
        while (m) {
          const int src = __ffs(m) - 1;
          const float sx = __shfl_sync(0xffffffffu, x, src), sy = __shfl_sync(0xffffffffu, y, src);
          const int minx = max((int)(sx - wf), 0), maxx = (int)(sx + wf), miny = max((int)(sy - wf), 0), maxy = (int)(sy + wf);
          if (lane == 0) cur[cnt] = base + src;
          cnt++;
          if (lane <= src || (cx >= minx && cx <= maxx && cy >= miny && cy <= maxy)) alive = false;
          // mark the box (clipped to the bounding box) for the later chunks: lanes take (row, word) pairs
          const int c0 = max(minx, bx0) - bx0, c1 = min(maxx, bx1) - bx0, r0 = max(miny, by0) - by0, r1 = min(maxy, by1) - by0;
          const int w0 = c0 >> 5, nw = (c1 >> 5) - w0 + 1, nr = r1 - r0 + 1;
          for (int t = lane; t < nw*nr; t += 32) {
            const int r = r0 + t/nw, w = w0 + t%nw;
            const int lo = max(c0 - 32*w, 0), hi = min(c1 - 32*w, 31);
            const uint32_t bits = (hi == 31 ? 0xffffffffu : ((1u << (hi + 1)) - 1u)) & ~((1u << lo) - 1u);
            bm[(size_t)r*bwords + w] |= bits;
          }
          __syncwarp();
          m = __ballot_sync(0xffffffffu, alive);
        }
      }
      if (lane == 0) s_cnt = cnt;
    }
    __syncthreads();
    const int c = s_cnt;
    __syncthreads();
    if ((unsigned)c >= S.kmin && (unsigned)c <= S.kmax) { fin = cur; final_cnt = c; break; }
    if ((unsigned)c < S.kmin) high = width - 1; else low = width + 1;
    prevwidth = width; prev_cnt = c;
    int* t = cur; cur = prev; prev = t;
  }
  for (int t = tid; t < final_cnt; t += ANMS_THREADS) a.out[off + t] = anms_tie_source(n, fin[t]);
  if (tid == 0) a.out_n[l] = final_cnt;
}
