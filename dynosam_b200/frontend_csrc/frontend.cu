// frontend.cu -- libdynofront: front-end rows a13 / a14 of SURVEY.md section 8 as sm_100a kernels (include/dynofront.h).
// Compiled with -fmad=false: the KLT arithmetic follows OpenCV's scalar float code, which is not FMA-contracted.
//
// Ordering semantics that make the reference sequential are kept exactly:
//  * trackDynamic's cv::circle side effect on the detection mask makes acceptance of feature i depend on the
//    earlier accepted features (FeatureTracker.cc:385-392,472-482): resolved in parallel as a greedy independent
//    set over the "covers" relation, in rounds, inside one CTA;
//  * the tracking mask takes the label of the LAST accepted feature that covers a pixel: max-index-wins scatter;
//  * new tracklet ids are handed out in iteration order: prefix count over the accepted features;
//  * propogateMask processes objects one after the other, each vote seeing the previous object's writes.
#include <cuda_runtime.h>
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/dynofront.h"
#include "anms.cuh"

#define FCK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { h->err = std::string(#call) + ": " + cudaGetErrorString(e_); return -3; } } while (0)

struct dynofront_ctx {
  int dev = 0, W = 0, H = 0; cudaStream_t s = nullptr; std::string err; bool have_prev = false, have_cur = false, have_pyr = false, have_pyr_cur = false;
  float* flow = nullptr; int32_t* mask = nullptr; uint8_t* det = nullptr; bool has_det = false;
  uint8_t* det_work = nullptr; uint8_t* trk = nullptr; int* trk_idx = nullptr; bool det_work_valid = false;
  // feature scratch (capacity cap)
  int cap = 0; double* f_kp = nullptr; int32_t *f_lab = nullptr, *f_age = nullptr; int64_t* f_tid = nullptr;
  int *f_x = nullptr, *f_y = nullptr, *f_state = nullptr, *f_next = nullptr; double* f_out = nullptr; int32_t* f_oage = nullptr; int64_t* f_otid = nullptr;
  int32_t* f_olab = nullptr; uint8_t* f_acc = nullptr; int* cell = nullptr; long long* nextid = nullptr;
  // sampling scratch
  int* tile_cnt = nullptr; int* obj_tot = nullptr; int* d_objs = nullptr; int* d_zero = nullptr; int* d_idx = nullptr; size_t idx_cap = 0;
  // propagate scratch
  int32_t* pmask = nullptr; float* pflow = nullptr; int32_t* cmask = nullptr; int* pflag = nullptr;
  // KLT
  std::vector<uint8_t*> pyr[2]; std::vector<short*> der; std::vector<int> lw, lh;
  float *k_prev = nullptr, *k_next = nullptr, *k_err = nullptr; uint8_t* k_st = nullptr; int k_cap = 0;
  float *k_back = nullptr, *k_eig = nullptr; uint8_t *k_st2 = nullptr, *k_keep = nullptr; int32_t* k_age = nullptr; int* k_count = nullptr;   // forward-backward tracker
  double* st_depth = nullptr; int st_cap = 0;     // stereoTrack
  std::vector<short*> der2;                       // Scharr derivatives of the CURRENT image (backward pass)
  // external-flow static tracker scratch
  int sf_cap = 0, sf_cells = 0; double* sf_kp = nullptr; int32_t* sf_age = nullptr; uint8_t* sf_use = nullptr; int32_t* sf_det = nullptr;
  int *sf_cell = nullptr, *sf_win = nullptr, *sf_win2 = nullptr, *sf_cnt = nullptr; uint8_t* sf_pass = nullptr; uint8_t* sf_acc = nullptr; double* sf_out = nullptr;
  int32_t* sf_oage = nullptr; long long* sf_otid = nullptr;
  // sampleDynamic on the device (candidate lists, ANMS scratch, per-object plan) and batched ANMS of float lists
  int *sd_idx = nullptr, *sd_off = nullptr, *sd_K = nullptr, *sd_sel = nullptr, *sd_out = nullptr, *sd_nsel = nullptr; float2* sd_pts = nullptr;
  uint32_t* sd_bm = nullptr; long long* sd_bm_off = nullptr; unsigned char *sd_host = nullptr, *sd_host_dev = nullptr; long long sd_host_cap = -1;
  int an_cap = 0, an_lists = 0; long long an_bm_cap = 0; float* an_xy = nullptr; float2* an_pts = nullptr; int *an_sel = nullptr, *an_out = nullptr;
  int *an_meta = nullptr; uint32_t* an_bm = nullptr; long long* an_bm_off = nullptr; int anms_smem = 0;
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  std::vector<void*> allocs;
};
template <class T> static int falloc(dynofront_ctx* h, T** p, size_t n) {
  *p = nullptr; if (n == 0) n = 1;
  FCK(cudaMalloc((void**)p, n*sizeof(T))); h->allocs.push_back((void*)*p); return 0;
}

// ---------------------------------------------------------------------------------------------------- trackDynamic
struct Disc { int r; int hw[16]; };   // half width of the filled cv::circle per |dy|
static Disc make_disc(int r) {       // OpenCV drawing.cpp Circle(): midpoint algorithm, filled spans
  Disc d; d.r = r; for (int i = 0; i < 16; i++) d.hw[i] = -1;
  int err = 0, dx = r, dy = 0, plus = 1, minus = (r << 1) - 1;
  while (dx >= dy) {
    d.hw[dy] = std::max(d.hw[dy], dx); d.hw[dx] = std::max(d.hw[dx], dy);
    dy++; err += plus; plus += 2;
    const int mask = (err <= 0) - 1;
    err -= minus & mask; dx += mask; minus -= mask & 2;
  }
  return d;
}
__device__ __forceinline__ bool disc_covers(const Disc& d, int dxp, int dyp) {
  const int ay = dyp < 0 ? -dyp : dyp, ax = dxp < 0 ? -dxp : dxp;
  return ay <= d.r && ax <= d.hw[ay];
}
__device__ __forceinline__ bool within_shrunken(double kx, double ky, int rows, int cols, int sr, int sc) {
  const int pc = (int)kx, pr = (int)ky;     // static_cast<int>
  return pr > sr && pr < rows - sr && pc > sc && pc < cols - sc;
}

__global__ void td_candidate_kernel(int n, const double* __restrict__ kp, const int32_t* __restrict__ plab, const int32_t* __restrict__ page,
                                    const float* __restrict__ flow, const int32_t* __restrict__ mask, const uint8_t* __restrict__ det, int W, int H,
                                    dynofront_track_params prm, int* fx, int* fy, int* state, double* out /*[n][4]*/, int32_t* oage, int32_t* olab) {
  const int i = blockIdx.x*blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double kx = kp[2*i], ky = kp[2*i + 1];
  const int x = (int)kx, y = (int)ky;
  fx[i] = x; fy[i] = y;
  int st = 2;   // 0 unknown (candidate), 1 accepted, 2 rejected
  out[4*i] = out[4*i+1] = out[4*i+2] = out[4*i+3] = 0.0; oage[i] = 0; olab[i] = 0;
  if (x >= 0 && x < W && y >= 0 && y < H) {
    const int lab = mask[(size_t)y*W + x];
    const bool det_ok = det ? det[(size_t)y*W + x] != 0 : true;
    const bool contained = kx >= 0.0 && kx < (double)W && ky >= 0.0 && ky < (double)H;
    if (det_ok && contained && lab != 0 && lab == plab[i]) {
      const double fxe = (double)flow[2*((size_t)y*W + x)], fye = (double)flow[2*((size_t)y*W + x) + 1];
      const double px = kx + fxe, py = ky + fye;
      if (within_shrunken(px, py, H, W, prm.shrink_row, prm.shrink_col) && !(fxe == 0 || fye == 0)) {
        st = 0;
        out[4*i] = px; out[4*i+1] = py; out[4*i+2] = fxe; out[4*i+3] = fye;
        oage[i] = page[i] + 1; olab[i] = lab;
      }
    }
  }
  state[i] = st;
}
__global__ void td_link_kernel(int n, const int* fx, const int* fy, const int* state, int W, int* cell, int* next) {
  const int i = blockIdx.x*blockDim.x + threadIdx.x;
  if (i >= n || state[i] != 0) return;
  next[i] = atomicExch(&cell[(size_t)fy[i]*W + fx[i]], i);
}
// greedy resolution + tracklet ids, one CTA
__global__ void __launch_bounds__(1024) td_resolve_kernel(int n, const int* fx, const int* fy, int* state, const int* cell, const int* next,
                                                          int W, int H, Disc disc, int max_age, const int64_t* ptid, int32_t* oage, int64_t* otid,
                                                          uint8_t* acc, long long* nextid) {
  __shared__ int remaining;
  for (;;) {
    if (threadIdx.x == 0) remaining = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      if (state[i] != 0) continue;
      bool any_acc = false, any_unknown = false;
      for (int dy = -disc.r; dy <= disc.r && !any_acc; dy++) {
        const int yy = fy[i] + dy; if (yy < 0 || yy >= H) continue;
        const int hw = disc.hw[dy < 0 ? -dy : dy];
        for (int dx = -hw; dx <= hw && !any_acc; dx++) {
          const int xx = fx[i] + dx; if (xx < 0 || xx >= W) continue;
          for (int j = cell[(size_t)yy*W + xx]; j >= 0; j = next[j]) {
            if (j >= i) continue;
            const int sj = ((volatile int*)state)[j];
            if (sj == 1) { any_acc = true; break; }
            if (sj == 0) any_unknown = true;
          }
        }
      }
      if (any_acc) state[i] = 2;
      else if (!any_unknown) state[i] = 1;
      else atomicAdd(&remaining, 1);
    }
    __syncthreads();
    if (remaining == 0) break;
    __syncthreads();
  }
  if (threadIdx.x == 0) {           // tracklet ids in iteration order (FeatureTracker.cc:446-450)
    long long id = *nextid;
    for (int i = 0; i < n; i++) {
      const bool a = state[i] == 1; acc[i] = a ? 1 : 0;
      if (!a) { oage[i] = 0; otid[i] = 0; continue; }
      if (oage[i] > max_age) { otid[i] = id++; oage[i] = 0; } else otid[i] = ptid[i];
    }
    *nextid = id;
  }
}
__global__ void td_clear_rejected_kernel(int n, const uint8_t* acc, double* out, int32_t* olab) {
  const int i = blockIdx.x*blockDim.x + threadIdx.x;
  if (i >= n || acc[i]) return;
  out[4*i] = out[4*i+1] = out[4*i+2] = out[4*i+3] = 0.0; olab[i] = 0;
}
__global__ void td_masks_kernel(int n, const int* fx, const int* fy, const uint8_t* acc, int W, int H, Disc disc, uint8_t* det, int* trk_idx) {
  const int i = blockIdx.x*blockDim.x + threadIdx.x;
  if (i >= n || !acc[i]) return;
  for (int dy = -disc.r; dy <= disc.r; dy++) {
    const int yy = fy[i] + dy; if (yy < 0 || yy >= H) continue;
    const int hw = disc.hw[dy < 0 ? -dy : dy];
    for (int dx = -hw; dx <= hw; dx++) {
      const int xx = fx[i] + dx; if (xx < 0 || xx >= W) continue;
      det[(size_t)yy*W + xx] = 0;
      atomicMax(&trk_idx[(size_t)yy*W + xx], i + 1);     // last writer (largest index) wins
    }
  }
}
__global__ void td_trk_final_kernel(size_t npx, const int* trk_idx, const int32_t* olab, uint8_t* trk) {
  const size_t p = (size_t)blockIdx.x*blockDim.x + threadIdx.x;
  if (p >= npx) return;
  const int t = trk_idx[p];
  const int l = t ? olab[t - 1] : 0;
  trk[p] = (uint8_t)(l > 255 ? 255 : l);
}
__global__ void fill_u8_kernel(uint8_t* p, size_t n, uint8_t v) { const size_t i = (size_t)blockIdx.x*blockDim.x + threadIdx.x; if (i < n) p[i] = v; }
__global__ void fill_i32_kernel(int* p, size_t n, int v) { const size_t i = (size_t)blockIdx.x*blockDim.x + threadIdx.x; if (i < n) p[i] = v; }

// ---------------------------------------------------------------------------------------------------- sampleDynamic scan
constexpr int ST_TILE = 1024, ST_MAXOBJ = 64;
__device__ __forceinline__ int sample_slot(size_t p, int W, int H, const uint8_t* det, const int32_t* mask, const float* flow, const int* objs, int nobj,
                                           dynofront_track_params prm, bool* zero) {
  *zero = false;
  if (det[p] == 0) return -1;
  const int lab = mask[p];
  int slot = -1;
  for (int o = 0; o < nobj; o++) if (objs[o] == lab) { slot = o; break; }
  if (slot < 0 || lab == 0) return -1;
  const double fx = (double)flow[2*p], fy = (double)flow[2*p + 1];
  if (fx == 0 || fy == 0) { *zero = true; return -(slot + 2); }
  const int i = (int)(p / W), j = (int)(p % W);
  if (!within_shrunken((double)j, (double)i, H, W, prm.shrink_row, prm.shrink_col)) return -1;
  return slot;
}
__global__ void __launch_bounds__(ST_TILE) sc_count_kernel(size_t npx, int W, int H, const uint8_t* det, const int32_t* mask, const float* flow,
                                                           const int* objs, int nobj, dynofront_track_params prm, int* tile_cnt, int* zero_cnt) {
  __shared__ int cnt[ST_MAXOBJ], zc[ST_MAXOBJ];
  if (threadIdx.x < ST_MAXOBJ) { cnt[threadIdx.x] = 0; zc[threadIdx.x] = 0; }
  __syncthreads();
  const size_t p = (size_t)blockIdx.x*ST_TILE + threadIdx.x;
  if (p < npx) {
    bool z; const int s = sample_slot(p, W, H, det, mask, flow, objs, nobj, prm, &z);
    if (s >= 0) atomicAdd(&cnt[s], 1); else if (z) atomicAdd(&zc[-s - 2], 1);
  }
  __syncthreads();
  if ((int)threadIdx.x < nobj) { tile_cnt[(size_t)blockIdx.x*ST_MAXOBJ + threadIdx.x] = cnt[threadIdx.x]; if (zc[threadIdx.x]) atomicAdd(&zero_cnt[threadIdx.x], zc[threadIdx.x]); }
}
__global__ void sc_scan_kernel(int ntiles, int nobj, int* tile_cnt, int* obj_tot) {
  const int o = threadIdx.x;
  if (o >= nobj) return;
  int run = 0;
  for (int t = 0; t < ntiles; t++) { const int c = tile_cnt[(size_t)t*ST_MAXOBJ + o]; tile_cnt[(size_t)t*ST_MAXOBJ + o] = run; run += c; }
  obj_tot[o] = run;
}
__global__ void __launch_bounds__(ST_TILE) sc_scatter_kernel(size_t npx, int W, int H, const uint8_t* det, const int32_t* mask, const float* flow,
                                                             const int* objs, int nobj, dynofront_track_params prm, const int* tile_off,
                                                             const int* obj_off, int* indices, long long capacity) {
  __shared__ int wc[32][ST_MAXOBJ];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t p = (size_t)blockIdx.x*ST_TILE + threadIdx.x;
  int s = -1;
  if (p < npx) { bool z; s = sample_slot(p, W, H, det, mask, flow, objs, nobj, prm, &z); if (s < 0) s = -1; }
  int myrank = 0;
  for (int o = 0; o < nobj; o++) {
    const unsigned b = __ballot_sync(0xffffffffu, s == o);
    if (lane == 0) wc[warp][o] = __popc(b);
    if (s == o) myrank = __popc(b & ((1u << lane) - 1));
  }
  __syncthreads();
  if (s >= 0) {
    int base = 0;
    for (int w = 0; w < warp; w++) base += wc[w][s];
    const long long dst = (long long)obj_off[s] + tile_off[(size_t)blockIdx.x*ST_MAXOBJ + s] + base + myrank;
    if (dst < capacity) indices[dst] = (int)p;
  }
}

// ---------------------------------------------------------------------------------------------------- sampleDynamic tail
// FeatureTracker.cc:955-1015 after the scan: per object K = max(max_features - num_track, 0) (:966-969), the candidate
// lists (ascending pixel index, the order of a serial run of the reference's fill) through suppressNonMax(RangeTree),
// then the new features.  Tracklet ids follow the order of objects[] (the reference's parallel for_each over a hash map
// leaves that order undefined), as dynofront_track_dynamic hands ids out in array order.
__global__ void sd_plan_kernel(int nobj, const int* obj_tot, const int* num_track, int max_features, int* off, int* K) {
  if (threadIdx.x != 0) return;
  int run = 0;
  for (int o = 0; o < nobj; o++) { off[o] = run; run += obj_tot[o]; K[o] = max(max_features - num_track[o], 0); }
}
// one CTA per object: exclusive scan of the selected counts over the objects gives the first feature / tracklet id;
// age 0, key-point (j, i), measured flow float -> double, predicted key-point = key-point + flow.  Writes straight into
// the mapped host staging buffer, so only the selected features cross PCIe.
__global__ void sd_construct_kernel(int nobj, const int* off, const int* tot, const int* zero, const int* nsel, const int* sel, const int* idx, int W,
                                    const float* __restrict__ flow, long long capacity, long long base_id, int32_t* stats, double* feat, long long* tid) {
  const int o = blockIdx.x;
  int pre = 0;
  for (int q = 0; q < o; q++) pre += nsel[q];
  const int ns = nsel[o];
  if (threadIdx.x == 0) { stats[o] = tot[o]; stats[ST_MAXOBJ + o] = zero[o]; stats[2*ST_MAXOBJ + o] = ns; stats[3*ST_MAXOBJ + o] = pre; }
  for (int t = threadIdx.x; t < ns; t += blockDim.x) {
    const long long f = (long long)pre + t;
    if (f >= capacity) break;
    const int p = idx[off[o] + sel[off[o] + t]];
    const int i = p / W, j = p % W;
    const double fx = (double)flow[2*(size_t)p], fy = (double)flow[2*(size_t)p + 1];
    double* r = feat + 6*f;
    r[0] = (double)j; r[1] = (double)i; r[2] = fx; r[3] = fy; r[4] = (double)j + fx; r[5] = (double)i + fy;
    tid[f] = base_id + f;
  }
}

// ---------------------------------------------------------------------------------------------------- propogateMask
__global__ void __launch_bounds__(256) pm_vote_kernel(int n, const double* kp, const int32_t* lab, int label, const int32_t* cur, int W, int H,
                                                     int min_votes, int* flag) {
  __shared__ int hist[256]; __shared__ int total;
  hist[threadIdx.x] = 0; if (threadIdx.x == 0) total = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    if (lab[i] != label) continue;
    const int u = (int)kp[2*i], v = (int)kp[2*i + 1];
    if (u < W && u > 0 && v < H && v > 0) {
      const int l = cur[(size_t)v*W + u];
      atomicAdd(&total, 1);
      if (l >= 0 && l < 256) atomicAdd(&hist[l], 1);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int best = -1, bc = -1;
    for (int l = 0; l < 256; l++) if (hist[l] > 0 && hist[l] > bc) { bc = hist[l]; best = l; }   // first maximum in ascending label order
    *flag = (total >= min_votes && best == 0) ? 1 : 0;
  }
}
__global__ void pm_warp_kernel(size_t npx, int W, int H, const int32_t* pmask, const float* pflow, int label, dynofront_track_params prm,
                               const int* flag, int32_t* cur) {
  if (*flag == 0) return;
  const size_t p = (size_t)blockIdx.x*blockDim.x + threadIdx.x;
  if (p >= npx || pmask[p] != label) return;
  const double fx = (double)pflow[2*p], fy = (double)pflow[2*p + 1];
  if (fx == 0 || fy == 0) return;
  const int j = (int)(p / W), k = (int)(p % W);
  const double px = k + fx, py = j + fy;
  if (!within_shrunken(px, py, H, W, prm.shrink_row, prm.shrink_col)) return;
  if (px < W && px > 0 && py < H && py > 0) cur[(size_t)((int)py)*W + (int)px] = label;
}

// ---------------------------------------------------------------------------------------------------- pyramidal KLT
__device__ __forceinline__ int reflect101(int i, int n) { if (i < 0) i = -i; if (i >= n) i = 2*n - 2 - i; return i; }
__global__ void pyr_down_kernel(const uint8_t* __restrict__ src, int sw, int sh, uint8_t* __restrict__ dst, int dw, int dh) {
  const int x = blockIdx.x*blockDim.x + threadIdx.x, y = blockIdx.y*blockDim.y + threadIdx.y;
  if (x >= dw || y >= dh) return;
  const int k[5] = { 1, 4, 6, 4, 1 };
  int sum = 0;
  for (int j = -2; j <= 2; j++) {
    const int yy = reflect101(2*y + j, sh);
    int row = 0;
    for (int i = -2; i <= 2; i++) row += k[i + 2]*src[(size_t)yy*sw + reflect101(2*x + i, sw)];
    sum += k[j + 2]*row;
  }
  dst[(size_t)y*dw + x] = (uint8_t)((sum + 128) >> 8);
}
__global__ void scharr_kernel(const uint8_t* __restrict__ src, int w, int h, short* __restrict__ dst) {
  const int x = blockIdx.x*blockDim.x + threadIdx.x, y = blockIdx.y*blockDim.y + threadIdx.y;
  if (x >= w || y >= h) return;
  const int y0 = y > 0 ? y - 1 : (h > 1 ? 1 : 0), y2 = y < h - 1 ? y + 1 : (h > 1 ? h - 2 : 0);
  const int xm = x > 0 ? x - 1 : (w > 1 ? 1 : 0), xp = x < w - 1 ? x + 1 : (w > 1 ? w - 2 : 0);
  auto t0 = [&](int xx) { return (src[(size_t)y0*w + xx] + src[(size_t)y2*w + xx])*3 + src[(size_t)y*w + xx]*10; };
  auto t1 = [&](int xx) { return (int)src[(size_t)y2*w + xx] - (int)src[(size_t)y0*w + xx]; };
  dst[2*((size_t)y*w + x)] = (short)(t0(xp) - t0(xm));
  dst[2*((size_t)y*w + x) + 1] = (short)((t1(xp) + t1(xm))*3 + t1(x)*10);
}

struct KltLevels { const uint8_t* I[8]; const uint8_t* J[8]; const short* D[8]; int w[8], h[8]; int nlev; };
constexpr int KLT_WARPS = 4, KLT_MAXWIN = 31;
#define DESCALE(x, n) (((x) + (1 << ((n) - 1))) >> (n))

__device__ __forceinline__ int img_at(const uint8_t* I, int w, int h, int x, int y) { return I[(size_t)reflect101(y, h)*w + reflect101(x, w)]; }
__device__ __forceinline__ int der_at(const short* D, int w, int h, int x, int y, int c) { return (x < 0 || x >= w || y < 0 || y >= h) ? 0 : D[2*((size_t)y*w + x) + c]; }

__global__ void __launch_bounds__(KLT_WARPS*32) klt_kernel(KltLevels L, int n, const float* __restrict__ prevPts, float* __restrict__ nextPts,
                                                           uint8_t* __restrict__ status, float* __restrict__ err, int win, int maxCount, float eps2,
                                                           int use_initial, float minEigThreshold, float* __restrict__ eig_out) {
  extern __shared__ short ksm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pt = blockIdx.x*KLT_WARPS + warp;
  if (pt >= n) return;
  const int area = win*win;
  short* Ipatch = ksm + (size_t)warp*area*3; short* dI = Ipatch + area;
  const float halfWin = (win - 1)*0.5f;
  const float px0 = prevPts[2*pt], py0 = prevPts[2*pt + 1];
  float nx = nextPts[2*pt], ny = nextPts[2*pt + 1];
  bool st = true; float e = 0.f;
  for (int level = L.nlev - 1; level >= 0; level--) {
    const int w = L.w[level], h = L.h[level];
    const float sc = (float)(1.0/(1 << level));
    float ppx = px0*sc, ppy = py0*sc;
    if (level == L.nlev - 1) { if (use_initial) { nx = nx*sc; ny = ny*sc; } else { nx = ppx; ny = ppy; } }
    else { nx = nx*2.f; ny = ny*2.f; }
    ppx -= halfWin; ppy -= halfWin;
    const int ipx = (int)floorf(ppx), ipy = (int)floorf(ppy);
    if (ipx < -win || ipx >= w || ipy < -win || ipy >= h) { if (level == 0) { st = false; e = 0.f; } continue; }
    float a = ppx - ipx, b = ppy - ipy;
    int iw00 = __float2int_rn((1.f - a)*(1.f - b)*16384.f), iw01 = __float2int_rn(a*(1.f - b)*16384.f),
        iw10 = __float2int_rn((1.f - a)*b*16384.f), iw11 = 16384 - iw00 - iw01 - iw10;
    long long sA11 = 0, sA12 = 0, sA22 = 0;
    for (int q = lane; q < area; q += 32) {
      const int y = q/win, x = q - y*win, gx = ipx + x, gy = ipy + y;
      const int ival = DESCALE(img_at(L.I[level], w, h, gx, gy)*iw00 + img_at(L.I[level], w, h, gx + 1, gy)*iw01 +
                               img_at(L.I[level], w, h, gx, gy + 1)*iw10 + img_at(L.I[level], w, h, gx + 1, gy + 1)*iw11, 9);
      const int ixv = DESCALE(der_at(L.D[level], w, h, gx, gy, 0)*iw00 + der_at(L.D[level], w, h, gx + 1, gy, 0)*iw01 +
                              der_at(L.D[level], w, h, gx, gy + 1, 0)*iw10 + der_at(L.D[level], w, h, gx + 1, gy + 1, 0)*iw11, 14);
      const int iyv = DESCALE(der_at(L.D[level], w, h, gx, gy, 1)*iw00 + der_at(L.D[level], w, h, gx + 1, gy, 1)*iw01 +
                              der_at(L.D[level], w, h, gx, gy + 1, 1)*iw10 + der_at(L.D[level], w, h, gx + 1, gy + 1, 1)*iw11, 14);
      Ipatch[q] = (short)ival; dI[2*q] = (short)ixv; dI[2*q + 1] = (short)iyv;
      sA11 += (long long)ixv*ixv; sA12 += (long long)ixv*iyv; sA22 += (long long)iyv*iyv;
    }
    for (int o = 16; o > 0; o >>= 1) { sA11 += __shfl_xor_sync(0xffffffffu, sA11, o); sA12 += __shfl_xor_sync(0xffffffffu, sA12, o); sA22 += __shfl_xor_sync(0xffffffffu, sA22, o); }
    __syncwarp();
    const float FLT_SCALE = 1.f/(1 << 20);
    const float A11 = (float)sA11*FLT_SCALE, A12 = (float)sA12*FLT_SCALE, A22 = (float)sA22*FLT_SCALE;
    float D = A11*A22 - A12*A12;
    const float minEig = (A22 + A11 - sqrtf((A11 - A22)*(A11 - A22) + 4.f*A12*A12))/(2*win*win);
    if (eig_out && level == 0 && lane == 0) { eig_out[2*pt] = minEig; eig_out[2*pt + 1] = (A11 + A22)/(2*win*win); }
    if (minEig < minEigThreshold || D < 1.1920929e-07f) { if (level == 0) st = false; continue; }
    D = 1.f/D;
    nx -= halfWin; ny -= halfWin;
    float pdx = 0.f, pdy = 0.f;
    float outx = nx + halfWin, outy = ny + halfWin;
    for (int j = 0; j < maxCount; j++) {
      const int inx = (int)floorf(nx), iny = (int)floorf(ny);
      if (inx < -win || inx >= w || iny < -win || iny >= h) { if (level == 0) st = false; break; }
      a = nx - inx; b = ny - iny;
      iw00 = __float2int_rn((1.f - a)*(1.f - b)*16384.f); iw01 = __float2int_rn(a*(1.f - b)*16384.f);
      iw10 = __float2int_rn((1.f - a)*b*16384.f); iw11 = 16384 - iw00 - iw01 - iw10;
      long long sb1 = 0, sb2 = 0;
      for (int q = lane; q < area; q += 32) {
        const int y = q/win, x = q - y*win, gx = inx + x, gy = iny + y;
        const int diff = DESCALE(img_at(L.J[level], w, h, gx, gy)*iw00 + img_at(L.J[level], w, h, gx + 1, gy)*iw01 +
                                 img_at(L.J[level], w, h, gx, gy + 1)*iw10 + img_at(L.J[level], w, h, gx + 1, gy + 1)*iw11, 9) - Ipatch[q];
        sb1 += (long long)diff*dI[2*q]; sb2 += (long long)diff*dI[2*q + 1];
      }
      for (int o = 16; o > 0; o >>= 1) { sb1 += __shfl_xor_sync(0xffffffffu, sb1, o); sb2 += __shfl_xor_sync(0xffffffffu, sb2, o); }
      const float b1 = (float)sb1*FLT_SCALE, b2 = (float)sb2*FLT_SCALE;
      const float dx = (A12*b2 - A22*b1)*D, dy = (A12*b1 - A11*b2)*D;
      nx += dx; ny += dy;
      outx = nx + halfWin; outy = ny + halfWin;
      if (dx*dx + dy*dy <= eps2) break;
      if (j > 0 && fabsf(dx + pdx) < 0.01f && fabsf(dy + pdy) < 0.01f) { outx -= dx*0.5f; outy -= dy*0.5f; break; }
      pdx = dx; pdy = dy;
    }
    nx = outx; ny = outy;
    if (st && level == 0) {     // residual error of the final position (status can still flip here)
      const float fx = nx - halfWin, fy = ny - halfWin;
      const int inx = (int)floorf(fx), iny = (int)floorf(fy);
      if (inx < -win || inx >= w || iny < -win || iny >= h) st = false;
      else {
        const float aa = fx - inx, bb = fy - iny;
        iw00 = __float2int_rn((1.f - aa)*(1.f - bb)*16384.f); iw01 = __float2int_rn(aa*(1.f - bb)*16384.f);
        iw10 = __float2int_rn((1.f - aa)*bb*16384.f); iw11 = 16384 - iw00 - iw01 - iw10;
        long long se = 0;
        for (int q = lane; q < area; q += 32) {
          const int y = q/win, x = q - y*win, gx = inx + x, gy = iny + y;
          const int diff = DESCALE(img_at(L.J[0], w, h, gx, gy)*iw00 + img_at(L.J[0], w, h, gx + 1, gy)*iw01 +
                                   img_at(L.J[0], w, h, gx, gy + 1)*iw10 + img_at(L.J[0], w, h, gx + 1, gy + 1)*iw11, 9) - Ipatch[q];
          se += diff < 0 ? -diff : diff;
        }
        for (int o = 16; o > 0; o >>= 1) se += __shfl_xor_sync(0xffffffffu, se, o);
        e = (float)se*(1.f/(32*win*win));
      }
    }
  }
  if (lane == 0) { nextPts[2*pt] = nx; nextPts[2*pt + 1] = ny; status[pt] = st ? 1 : 0; if (err) err[pt] = e; }
}

// ---------------------------------------------------------------------------------------------------- forward-backward KLT
// KltFeatureTracker::trackPoints after the two cv::calcOpticalFlowPyrLK calls (StaticFeatureTracker.cc:505-534): a track
// survives when both passes succeeded and the backward pass returns to within 0.5 px of where it started (float
// arithmetic, as the reference's lambda), then the per-point checks of :575-592 / :628-646 -- background label at the
// truncated key-point, inside the image and the shrunken image, age + 1 <= max_feature_track_age.
__global__ void klt_fb_filter_kernel(int n, const float* __restrict__ prev, const float* __restrict__ next, const float* __restrict__ back,
                                     const uint8_t* __restrict__ st_f, const uint8_t* __restrict__ st_b, float max_dist, uint8_t* __restrict__ status,
                                     int check, const int32_t* __restrict__ mask, int W, int H, dynofront_track_params prm, const int32_t* __restrict__ age,
                                     int max_age, uint8_t* __restrict__ keep, int* __restrict__ count) {
  const int i = blockIdx.x*blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float dx = prev[2*i] - back[2*i], dy = prev[2*i + 1] - back[2*i + 1];
  const bool ok = st_f[i] && st_b[i] && sqrtf(dx*dx + dy*dy) <= max_dist;
  status[i] = ok ? 1 : 0;
  bool k = ok;
  if (check && ok) {
    const double kx = (double)next[2*i], ky = (double)next[2*i + 1];
    const int x = (int)kx, y = (int)ky;                                       // functional_keypoint::u / v: truncation
    const bool contained = kx >= 0.0 && kx < (double)W && ky >= 0.0 && ky < (double)H;
    const bool shrunk = y > prm.shrink_row && y < H - prm.shrink_row && x > prm.shrink_col && x < W - prm.shrink_col;
    k = contained && shrunk && mask[(size_t)y*W + x] == 0 && age[i] + 1 <= max_age;
  }
  keep[i] = k ? 1 : 0;
  if (ok) atomicAdd(count, 1);
  if (k) atomicAdd(count + 1, 1);
}
__global__ void count_status_kernel(int n, const uint8_t* st, int* count) {
  const int i = blockIdx.x*blockDim.x + threadIdx.x;
  if (i < n && st[i]) atomicAdd(count, 1);
}

// ---------------------------------------------------------------------------------------------------- external-flow static tracker
// ExternalFlowFeatureTracker::trackStatic / constructStaticFeature (StaticFeatureTracker.cc:70-220).  The reference walks
// the previous features in order and the FIRST one that passes every check claims its grid cell (cells are only marked by
// successful constructions): in parallel, the passing feature with the smallest index per cell wins (atomicMin).  New
// detections do the same among the cells the tracked features left free, in detection order, until the frame holds
// max_features (a prefix count); tracklet ids are handed out in that order.
__device__ __forceinline__ bool sf_construct(const float* flow, const int32_t* mask, int W, int H, int x, int y, double kx, double ky, double* out) {
  if (mask[(size_t)y*W + x] != 0) return false;
  const double fx = (double)flow[2*((size_t)y*W + x)], fy = (double)flow[2*((size_t)y*W + x) + 1];
  if (!(fx != 0 && fy != 0)) return false;
  const double px = kx + fx, py = ky + fy;
  if (!(px >= 0.0 && px < (double)W && py >= 0.0 && py < (double)H)) return false;
  out[0] = fx; out[1] = fy; out[2] = px; out[3] = py;
  return true;
}
__global__ void sf_prev_kernel(int n, const double* __restrict__ kp, const uint8_t* __restrict__ usable, const float* flow, const int32_t* mask, int W, int H,
                               int cell_size, int ncols, int* __restrict__ cell, uint8_t* __restrict__ pass, double* __restrict__ out, int* __restrict__ win) {
  const int i = blockIdx.x*blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double kx = kp[2*i], ky = kp[2*i + 1];
  pass[i] = 0; cell[i] = -1;
  if (!(kx >= 0.0 && kx < (double)W && ky >= 0.0 && ky < (double)H)) return;
  const int x = (int)kx, y = (int)ky;
  const int c = (int)floor(ky/cell_size)*ncols + (int)floor(kx/cell_size);
  cell[i] = c;
  if (!usable[i]) return;
  if (!sf_construct(flow, mask, W, H, x, y, kx, ky, out + 4*(size_t)i)) return;
  pass[i] = 1;
  atomicMin(win + c, i);
}
__global__ void sf_prev_resolve_kernel(int n, const int* cell, const uint8_t* pass, const int* win, const int32_t* age, uint8_t* acc, double* out, int32_t* oage, int* cnt) {
  const int i = blockIdx.x*blockDim.x + threadIdx.x;
  if (i >= n) return;
  const bool a = pass[i] && win[cell[i]] == i;
  acc[i] = a ? 1 : 0; oage[i] = a ? age[i] + 1 : 0;
  if (!a) { out[4*(size_t)i] = out[4*(size_t)i + 1] = out[4*(size_t)i + 2] = out[4*(size_t)i + 3] = 0.0; }
  else atomicAdd(cnt, 1);
}
__global__ void sf_det_kernel(int n, const int32_t* __restrict__ xy, const float* flow, const int32_t* mask, int W, int H, int cell_size, int ncols,
                              const int* __restrict__ win_prev, int* __restrict__ cell, uint8_t* __restrict__ pass, double* __restrict__ out, int* __restrict__ win) {
  const int j = blockIdx.x*blockDim.x + threadIdx.x;
  if (j >= n) return;
  const int x = xy[2*j], y = xy[2*j + 1];
  pass[j] = 0; cell[j] = -1;
  if (x < 0 || x >= W || y < 0 || y >= H) return;
  if (mask[(size_t)y*W + x] != 0) return;
  const int c = (int)floor((double)y/cell_size)*ncols + (int)floor((double)x/cell_size);
  cell[j] = c;
  if (win_prev[c] != 0x7fffffff) return;                       // cell taken by a tracked feature
  if (!sf_construct(flow, mask, W, H, x, y, (double)x, (double)y, out + 4*(size_t)j)) return;
  pass[j] = 1;
  atomicMin(win + c, j);
}
// one CTA: in-order prefix count of the accepted detections, truncated at `room`; tracklet ids follow the order
__global__ void __launch_bounds__(1024) sf_det_resolve_kernel(int n, const int* cell, const uint8_t* pass, const int* win, const int* cnt_prev, int max_features,
                                                              long long base_id, uint8_t* acc, double* out, long long* otid, int* cnt_det) {
  __shared__ int s_scan[1024]; __shared__ int s_base;
  const int room = max(0, max_features - *cnt_prev);
  if (threadIdx.x == 0) s_base = 0;
  __syncthreads();
  for (int j0 = 0; j0 < n; j0 += 1024) {
    const int j = j0 + threadIdx.x;
    const int a = (j < n && pass[j] && win[cell[j]] == j) ? 1 : 0;
    s_scan[threadIdx.x] = a;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) { const int v = threadIdx.x >= o ? s_scan[threadIdx.x - o] : 0; __syncthreads(); s_scan[threadIdx.x] += v; __syncthreads(); }
    const int rank = s_base + s_scan[threadIdx.x] - a;           // accepted detections before j
    if (j < n) {
      const bool fin = a && rank < room;
      acc[j] = fin ? 1 : 0; otid[j] = fin ? base_id + rank : 0;
      if (!fin) { out[4*(size_t)j] = out[4*(size_t)j + 1] = out[4*(size_t)j + 2] = out[4*(size_t)j + 3] = 0.0; }
    }
    __syncthreads();
    if (threadIdx.x == 1023) s_base += s_scan[1023];
    __syncthreads();
  }
  if (threadIdx.x == 0) *cnt_det = min(s_base, room);
}

// ---------------------------------------------------------------------------------------------------- host API
extern "C" {

const char* dynofront_last_error(dynofront_handle h) { return h ? h->err.c_str() : "null handle"; }

int dynofront_create(int device, int width, int height, dynofront_handle* out) {
  if (!out || width <= 0 || height <= 0) return -1;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return -3;
  cudaDeviceProp prop; if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major < 10) return -3;
  dynofront_ctx* h = new dynofront_ctx(); h->dev = device; h->W = width; h->H = height;
  cudaSetDevice(device);
  if (cudaStreamCreateWithFlags(&h->s, cudaStreamNonBlocking) != cudaSuccess) { delete h; return -3; }
  cudaEventCreate(&h->e0); cudaEventCreate(&h->e1);
  const size_t npx = (size_t)width*height;
  int rc = 0;
  rc |= falloc(h, &h->flow, 2*npx); rc |= falloc(h, &h->mask, npx); rc |= falloc(h, &h->det, npx); rc |= falloc(h, &h->det_work, npx);
  rc |= falloc(h, &h->trk, npx); rc |= falloc(h, &h->trk_idx, npx); rc |= falloc(h, &h->cell, npx); rc |= falloc(h, &h->nextid, 1);
  rc |= falloc(h, &h->tile_cnt, ((npx + ST_TILE - 1)/ST_TILE)*ST_MAXOBJ); rc |= falloc(h, &h->obj_tot, ST_MAXOBJ);
  rc |= falloc(h, &h->d_objs, ST_MAXOBJ); rc |= falloc(h, &h->d_zero, ST_MAXOBJ);
  rc |= falloc(h, &h->pmask, npx); rc |= falloc(h, &h->pflow, 2*npx); rc |= falloc(h, &h->cmask, npx); rc |= falloc(h, &h->pflag, 1);
  if (rc) { dynofront_destroy(h); return -3; }
  *out = h;
  return 0;
}
int dynofront_destroy(dynofront_handle h) {
  if (!h) return -1;
  cudaSetDevice(h->dev);
  for (void* p : h->allocs) cudaFree(p);
  if (h->e0) cudaEventDestroy(h->e0); if (h->e1) cudaEventDestroy(h->e1);
  if (h->s) cudaStreamDestroy(h->s);
  if (h->sd_host) cudaFreeHost(h->sd_host);
  delete h; return 0;
}
int dynofront_set_frame(dynofront_handle h, const float* flow, const int32_t* motion_mask, const uint8_t* detection_mask) {
  if (!h) return -1; cudaSetDevice(h->dev);
  const size_t npx = (size_t)h->W*h->H;
  if (flow) FCK(cudaMemcpyAsync(h->flow, flow, 2*npx*sizeof(float), cudaMemcpyHostToDevice, h->s));
  if (motion_mask) FCK(cudaMemcpyAsync(h->mask, motion_mask, npx*sizeof(int32_t), cudaMemcpyHostToDevice, h->s));
  if (detection_mask) { FCK(cudaMemcpyAsync(h->det, detection_mask, npx, cudaMemcpyHostToDevice, h->s)); h->has_det = true; }
  else h->has_det = false;
  h->det_work_valid = false;
  FCK(cudaStreamSynchronize(h->s));
  return 0;
}
static int build_pyramid(dynofront_ctx* h, int which, const uint8_t* host_img, int max_level, int win, bool with_deriv);
// Streaming: the frame that was current becomes the previous one WITHOUT moving data (the device buffers swap roles:
// flow / motion mask for propogateMask, gray pyramid + Scharr derivatives for the KLT), then only the new frame's images
// cross PCIe (asynchronously when the host buffers are pinned, dynofront_pin_host) and only its pyramid is built.
int dynofront_next_frame(dynofront_handle h, const uint8_t* gray, const float* flow, const int32_t* motion_mask, const uint8_t* detection_mask) {
  if (!h || !gray || !flow || !motion_mask) return -1;
  cudaSetDevice(h->dev);
  const size_t npx = (size_t)h->W*h->H;
  std::swap(h->flow, h->pflow); std::swap(h->mask, h->pmask);
  FCK(cudaMemcpyAsync(h->flow, flow, 2*npx*sizeof(float), cudaMemcpyHostToDevice, h->s));
  FCK(cudaMemcpyAsync(h->mask, motion_mask, npx*sizeof(int32_t), cudaMemcpyHostToDevice, h->s));
  if (detection_mask) { FCK(cudaMemcpyAsync(h->det, detection_mask, npx, cudaMemcpyHostToDevice, h->s)); h->has_det = true; } else h->has_det = false;
  h->det_work_valid = false;
  h->have_prev = h->have_cur; h->have_cur = true;
  if (!h->lw.empty()) { std::swap(h->pyr[0], h->pyr[1]); std::swap(h->der, h->der2); }
  h->have_pyr = h->have_pyr_cur; h->have_pyr_cur = true;
  if (build_pyramid(h, 1, gray, 5, 21, true)) return -3;       // (levels that are too small for a window are simply never read)
  return 0;                                                     // no synchronisation: the next call's work is ordered behind on the stream
}
static int ensure_features(dynofront_ctx* h, int n) {
  if (n <= h->cap) return 0;
  const int cap = std::max(n, 4096);
  int rc = 0;
  rc |= falloc(h, &h->f_kp, 2*(size_t)cap); rc |= falloc(h, &h->f_lab, cap); rc |= falloc(h, &h->f_age, cap); rc |= falloc(h, &h->f_tid, cap);
  rc |= falloc(h, &h->f_x, cap); rc |= falloc(h, &h->f_y, cap); rc |= falloc(h, &h->f_state, cap); rc |= falloc(h, &h->f_next, cap);
  rc |= falloc(h, &h->f_out, 4*(size_t)cap); rc |= falloc(h, &h->f_oage, cap); rc |= falloc(h, &h->f_otid, cap); rc |= falloc(h, &h->f_olab, cap);
  rc |= falloc(h, &h->f_acc, cap);
  if (rc) return -3;
  h->cap = cap; return 0;
}
static void prepare_det_work(dynofront_ctx* h) {
  const size_t npx = (size_t)h->W*h->H;
  if (h->has_det) cudaMemcpyAsync(h->det_work, h->det, npx, cudaMemcpyDeviceToDevice, h->s);
  else fill_u8_kernel<<<(unsigned)((npx + 255)/256), 256, 0, h->s>>>(h->det_work, npx, 255);
  h->det_work_valid = true;
}

int dynofront_track_dynamic(dynofront_handle h, int32_t n, const double* kp, const int32_t* lab, const int32_t* age, const int64_t* tid,
                            const dynofront_track_params* prm, int64_t* next_tracklet_id, uint8_t* accepted, double* pred_kp, double* flow_out,
                            int32_t* oage, int64_t* otid, int32_t* olab, uint8_t* det_out, uint8_t* trk_out) {
  if (!h || !prm || n < 0 || !next_tracklet_id) return -1;
  if (prm->min_distance < 0 || prm->min_distance > 15) { h->err = "min_distance must be in [0,15]"; return -1; }
  cudaSetDevice(h->dev);
  if (ensure_features(h, n)) return -3;
  const size_t npx = (size_t)h->W*h->H; const int W = h->W, H = h->H;
  const Disc disc = make_disc(prm->min_distance);
  FCK(cudaMemcpyAsync(h->f_kp, kp, 2*(size_t)n*8, cudaMemcpyHostToDevice, h->s));
  FCK(cudaMemcpyAsync(h->f_lab, lab, (size_t)n*4, cudaMemcpyHostToDevice, h->s));
  FCK(cudaMemcpyAsync(h->f_age, age, (size_t)n*4, cudaMemcpyHostToDevice, h->s));
  FCK(cudaMemcpyAsync(h->f_tid, tid, (size_t)n*8, cudaMemcpyHostToDevice, h->s));
  long long nid = *next_tracklet_id;
  FCK(cudaMemcpyAsync(h->nextid, &nid, 8, cudaMemcpyHostToDevice, h->s));
  prepare_det_work(h);
  fill_i32_kernel<<<(unsigned)((npx + 255)/256), 256, 0, h->s>>>(h->cell, npx, -1);
  fill_i32_kernel<<<(unsigned)((npx + 255)/256), 256, 0, h->s>>>(h->trk_idx, npx, 0);
  if (n > 0) {
    const int g = (n + 127)/128;
    td_candidate_kernel<<<g, 128, 0, h->s>>>(n, h->f_kp, h->f_lab, h->f_age, h->flow, h->mask, h->has_det ? h->det : nullptr, W, H, *prm,
                                             h->f_x, h->f_y, h->f_state, h->f_out, h->f_oage, h->f_olab);
    td_link_kernel<<<g, 128, 0, h->s>>>(n, h->f_x, h->f_y, h->f_state, W, h->cell, h->f_next);
    td_resolve_kernel<<<1, 1024, 0, h->s>>>(n, h->f_x, h->f_y, h->f_state, h->cell, h->f_next, W, H, disc, prm->max_dynamic_feature_age,
                                            (const int64_t*)h->f_tid, h->f_oage, h->f_otid, h->f_acc, h->nextid);
    td_clear_rejected_kernel<<<g, 128, 0, h->s>>>(n, h->f_acc, h->f_out, h->f_olab);
    td_masks_kernel<<<g, 128, 0, h->s>>>(n, h->f_x, h->f_y, h->f_acc, W, H, disc, h->det_work, h->trk_idx);
  }
  td_trk_final_kernel<<<(unsigned)((npx + 255)/256), 256, 0, h->s>>>(npx, h->trk_idx, h->f_olab, h->trk);
  std::vector<double> out4((size_t)4*n);
  if (n) {
    FCK(cudaMemcpyAsync(out4.data(), h->f_out, out4.size()*8, cudaMemcpyDeviceToHost, h->s));
    if (accepted) FCK(cudaMemcpyAsync(accepted, h->f_acc, n, cudaMemcpyDeviceToHost, h->s));
    if (oage) FCK(cudaMemcpyAsync(oage, h->f_oage, (size_t)n*4, cudaMemcpyDeviceToHost, h->s));
    if (otid) FCK(cudaMemcpyAsync(otid, h->f_otid, (size_t)n*8, cudaMemcpyDeviceToHost, h->s));
    if (olab) FCK(cudaMemcpyAsync(olab, h->f_olab, (size_t)n*4, cudaMemcpyDeviceToHost, h->s));
  }
  FCK(cudaMemcpyAsync(&nid, h->nextid, 8, cudaMemcpyDeviceToHost, h->s));
  if (det_out) FCK(cudaMemcpyAsync(det_out, h->det_work, npx, cudaMemcpyDeviceToHost, h->s));
  if (trk_out) FCK(cudaMemcpyAsync(trk_out, h->trk, npx, cudaMemcpyDeviceToHost, h->s));
  FCK(cudaStreamSynchronize(h->s));
  FCK(cudaGetLastError());
  *next_tracklet_id = nid;
  for (int i = 0; i < n; i++) {
    if (pred_kp) { pred_kp[2*i] = out4[4*i]; pred_kp[2*i+1] = out4[4*i+1]; }
    if (flow_out) { flow_out[2*i] = out4[4*i+2]; flow_out[2*i+1] = out4[4*i+3]; }
  }
  return 0;
}

int dynofront_sample_candidates(dynofront_handle h, int32_t nobj, const int32_t* objects, const dynofront_track_params* prm, int32_t* counts,
                                int32_t* offsets, int32_t* zero_flow, int32_t* indices, int64_t capacity) {
  if (!h || !prm || nobj < 0 || nobj > ST_MAXOBJ || !counts || !offsets) return -1;
  cudaSetDevice(h->dev);
  const size_t npx = (size_t)h->W*h->H; const int ntiles = (int)((npx + ST_TILE - 1)/ST_TILE);
  if (!h->det_work_valid) prepare_det_work(h);
  if ((size_t)capacity > h->idx_cap) { if (falloc(h, &h->d_idx, (size_t)capacity)) return -3; h->idx_cap = (size_t)capacity; }
  FCK(cudaMemcpyAsync(h->d_objs, objects, (size_t)nobj*4, cudaMemcpyHostToDevice, h->s));
  FCK(cudaMemsetAsync(h->d_zero, 0, ST_MAXOBJ*4, h->s));
  sc_count_kernel<<<ntiles, ST_TILE, 0, h->s>>>(npx, h->W, h->H, h->det_work, h->mask, h->flow, h->d_objs, nobj, *prm, h->tile_cnt, h->d_zero);
  sc_scan_kernel<<<1, ST_MAXOBJ, 0, h->s>>>(ntiles, nobj, h->tile_cnt, h->obj_tot);
  std::vector<int> tot(ST_MAXOBJ), zc(ST_MAXOBJ);
  FCK(cudaMemcpyAsync(tot.data(), h->obj_tot, ST_MAXOBJ*4, cudaMemcpyDeviceToHost, h->s));
  FCK(cudaMemcpyAsync(zc.data(), h->d_zero, ST_MAXOBJ*4, cudaMemcpyDeviceToHost, h->s));
  FCK(cudaStreamSynchronize(h->s));
  int run = 0;
  for (int o = 0; o < nobj; o++) { counts[o] = tot[o]; offsets[o] = run; run += tot[o]; if (zero_flow) zero_flow[o] = zc[o]; }
  if (indices && capacity > 0) {
    FCK(cudaMemcpyAsync(h->obj_tot, offsets, (size_t)nobj*4, cudaMemcpyHostToDevice, h->s));
    sc_scatter_kernel<<<ntiles, ST_TILE, 0, h->s>>>(npx, h->W, h->H, h->det_work, h->mask, h->flow, h->d_objs, nobj, *prm, h->tile_cnt, h->obj_tot,
                                                    h->d_idx, (long long)capacity);
    const size_t ncopy = std::min<size_t>((size_t)run, (size_t)capacity);
    FCK(cudaMemcpyAsync(indices, h->d_idx, ncopy*4, cudaMemcpyDeviceToHost, h->s));
    FCK(cudaStreamSynchronize(h->s));
  }
  FCK(cudaGetLastError());
  return 0;
}

int dynofront_propagate_mask(dynofront_handle h, int32_t n, const double* kp, const int32_t* lab, const int32_t* prev_mask, const float* prev_flow,
                             const dynofront_track_params* prm, int32_t min_votes, int32_t* current_mask) {
  if (!h || !prm || n < 0) return -1;
  const bool resident = !prev_mask && !prev_flow && !current_mask;       // previous / current frame already on the device (dynofront_next_frame)
  if (!resident && (!prev_mask || !prev_flow || !current_mask)) { h->err = "pass all three images, or none for the resident frames"; return -1; }
  if (resident && !h->have_prev) { h->err = "no previous frame on the device"; return -2; }
  cudaSetDevice(h->dev);
  if (ensure_features(h, n)) return -3;
  const size_t npx = (size_t)h->W*h->H;
  FCK(cudaMemcpyAsync(h->f_kp, kp, 2*(size_t)n*8, cudaMemcpyHostToDevice, h->s));
  FCK(cudaMemcpyAsync(h->f_lab, lab, (size_t)n*4, cudaMemcpyHostToDevice, h->s));
  const int32_t* pmask = h->pmask; const float* pflow = h->pflow; int32_t* cmask = resident ? h->mask : h->cmask;
  if (!resident) {
    FCK(cudaMemcpyAsync(h->pmask, prev_mask, npx*4, cudaMemcpyHostToDevice, h->s));
    FCK(cudaMemcpyAsync(h->pflow, prev_flow, 2*npx*4, cudaMemcpyHostToDevice, h->s));
    FCK(cudaMemcpyAsync(h->cmask, current_mask, npx*4, cudaMemcpyHostToDevice, h->s));
    h->have_prev = false;               // the resident previous frame was overwritten
  }
  std::vector<int32_t> labels(lab, lab + n);
  std::sort(labels.begin(), labels.end()); labels.erase(std::unique(labels.begin(), labels.end()), labels.end());
  for (int32_t l : labels) {      // objects in ascending label order, sequentially (FeatureTracker.cc:1262)
    pm_vote_kernel<<<1, 256, 0, h->s>>>(n, h->f_kp, h->f_lab, l, cmask, h->W, h->H, min_votes, h->pflag);
    pm_warp_kernel<<<(unsigned)((npx + 255)/256), 256, 0, h->s>>>(npx, h->W, h->H, pmask, pflow, l, *prm, h->pflag, cmask);
  }
  if (!resident) FCK(cudaMemcpyAsync(current_mask, h->cmask, npx*4, cudaMemcpyDeviceToHost, h->s));
  FCK(cudaStreamSynchronize(h->s));
  FCK(cudaGetLastError());
  return 0;
}
int dynofront_get_motion_mask(dynofront_handle h, int32_t* out) {
  if (!h || !out) return -1;
  cudaSetDevice(h->dev);
  FCK(cudaMemcpyAsync(out, h->mask, (size_t)h->W*h->H*4, cudaMemcpyDeviceToHost, h->s)); FCK(cudaStreamSynchronize(h->s));
  return 0;
}
int dynofront_pin_host(dynofront_handle h, void* ptr, size_t bytes) {
  if (!h || !ptr) return -1;
  cudaSetDevice(h->dev);
  FCK(cudaHostRegister(ptr, bytes, cudaHostRegisterDefault));
  return 0;
}
int dynofront_unpin_host(dynofront_handle h, void* ptr) {
  if (!h || !ptr) return -1;
  cudaSetDevice(h->dev);
  FCK(cudaHostUnregister(ptr));
  return 0;
}
static int klt_scratch(dynofront_ctx* h, int cap) {
  if (falloc(h, &h->k_prev, 2*(size_t)cap) || falloc(h, &h->k_next, 2*(size_t)cap) || falloc(h, &h->k_err, cap) || falloc(h, &h->k_st, cap) ||
      falloc(h, &h->k_back, 2*(size_t)cap) || falloc(h, &h->k_eig, 2*(size_t)cap) || falloc(h, &h->k_st2, cap) || falloc(h, &h->k_keep, cap) ||
      falloc(h, &h->k_age, cap) || falloc(h, &h->k_count, 2)) return -3;
  h->k_cap = cap; return 0;
}
static int build_pyramid(dynofront_ctx* h, int which, const uint8_t* host_img, int max_level, int win, bool with_deriv) {
  const int W = h->W, H = h->H;
  if (h->lw.empty()) {
    int w = W, hh = H;
    for (int l = 0; l < 8; l++) {
      h->lw.push_back(w); h->lh.push_back(hh);
      uint8_t *a, *b; short* d;
      if (falloc(h, &a, (size_t)w*hh) || falloc(h, &b, (size_t)w*hh) || falloc(h, &d, 2*(size_t)w*hh)) return -3;
      h->pyr[0].push_back(a); h->pyr[1].push_back(b); h->der.push_back(d);
      short* d2; if (falloc(h, &d2, 2*(size_t)w*hh)) return -3; h->der2.push_back(d2);
      w = (w + 1)/2; hh = (hh + 1)/2;
      if (w < 2 || hh < 2) break;
    }
  }
  FCK(cudaMemcpyAsync(h->pyr[which][0], host_img, (size_t)W*H, cudaMemcpyHostToDevice, h->s));
  const dim3 blk(32, 8);
  for (int l = 0; l <= max_level && l < (int)h->lw.size(); l++) {
    const int w = h->lw[l], hh = h->lh[l];
    if (l > 0) pyr_down_kernel<<<dim3((w + 31)/32, (hh + 7)/8), blk, 0, h->s>>>(h->pyr[which][l-1], h->lw[l-1], h->lh[l-1], h->pyr[which][l], w, hh);
    if (with_deriv) scharr_kernel<<<dim3((w + 31)/32, (hh + 7)/8), blk, 0, h->s>>>(h->pyr[which][l], w, hh, which == 0 ? h->der[l] : h->der2[l]);
  }
  return 0;
}

int dynofront_klt_track(dynofront_handle h, const uint8_t* prev_gray, const uint8_t* cur_gray, int32_t n, const float* prev_pts, float* next_pts,
                        uint8_t* status, float* err, int32_t win, int32_t max_level, int32_t max_count, double epsilon, int32_t use_initial,
                        double min_eig, float* ms_device) {
  if (!h || !prev_gray || !cur_gray || n < 0 || !prev_pts || !next_pts || !status) return -1;
  if (win < 3 || win > KLT_MAXWIN || max_level < 0) { h->err = "win must be in [3,31]"; return -1; }
  cudaSetDevice(h->dev);
  // buildOpticalFlowPyramid: stop when a level is not larger than the window (lkpyramid.cpp)
  int levels = 0; { int w = h->W, hh = h->H; for (int l = 0; l <= max_level && l < 8; l++) { levels = l; if (l < max_level) { const int w2 = (w + 1)/2, h2 = (hh + 1)/2; if (w2 <= win || h2 <= win) break; w = w2; hh = h2; } } }
  if (n > h->k_cap) { const int cap = std::max(n, 4096); if (klt_scratch(h, cap)) return -3; }
  FCK(cudaEventRecord(h->e0, h->s));
  if (build_pyramid(h, 0, prev_gray, levels, win, true)) return -3;
  if (build_pyramid(h, 1, cur_gray, levels, win, false)) return -3;
  h->have_pyr = h->have_pyr_cur = false;      // (the resident pyramids of the streaming mode were overwritten)
  FCK(cudaMemcpyAsync(h->k_prev, prev_pts, 2*(size_t)n*4, cudaMemcpyHostToDevice, h->s));
  FCK(cudaMemcpyAsync(h->k_next, use_initial ? next_pts : prev_pts, 2*(size_t)n*4, cudaMemcpyHostToDevice, h->s));
  KltLevels L; L.nlev = levels + 1;
  for (int l = 0; l <= levels; l++) { L.I[l] = h->pyr[0][l]; L.J[l] = h->pyr[1][l]; L.D[l] = h->der[l]; L.w[l] = h->lw[l]; L.h[l] = h->lh[l]; }
  max_count = std::min(std::max(max_count, 0), 100);
  double eps = std::min(std::max(epsilon, 0.0), 10.0); eps *= eps;
  if (n > 0) {
    const size_t smem = (size_t)KLT_WARPS*win*win*3*sizeof(short);
    klt_kernel<<<(n + KLT_WARPS - 1)/KLT_WARPS, KLT_WARPS*32, smem, h->s>>>(L, n, h->k_prev, h->k_next, h->k_st, h->k_err, win, max_count, (float)eps,
                                                                            use_initial, (float)min_eig, h->k_eig);
  }
  FCK(cudaMemcpyAsync(next_pts, h->k_next, 2*(size_t)n*4, cudaMemcpyDeviceToHost, h->s));
  FCK(cudaMemcpyAsync(status, h->k_st, n, cudaMemcpyDeviceToHost, h->s));
  if (err) FCK(cudaMemcpyAsync(err, h->k_err, (size_t)n*4, cudaMemcpyDeviceToHost, h->s));
  FCK(cudaEventRecord(h->e1, h->s));
  FCK(cudaStreamSynchronize(h->s));
  FCK(cudaGetLastError());
  if (ms_device) FCK(cudaEventElapsedTime(ms_device, h->e0, h->e1));
  return 0;
}

int dynofront_klt_track_fb(dynofront_handle h, const uint8_t* prev_gray, const uint8_t* cur_gray, int32_t n, const float* prev_pts, float* next_pts,
                           uint8_t* status, float* back_pts, const dynofront_klt_fb_params* P, const int32_t* prev_age, uint8_t* keep,
                           int32_t* n_status, int32_t* n_keep, float* ms_device) {
  if (!h || n < 0 || !prev_pts || !next_pts || !status || !P) return -1;
  const bool resident = !prev_gray && !cur_gray;           // both pyramids already on the device (dynofront_next_frame, twice)
  if (!resident && (!prev_gray || !cur_gray)) { h->err = "pass both images, or none for the resident frames"; return -1; }
  if (resident && !(h->have_pyr && h->have_pyr_cur)) { h->err = "two frames are needed on the device"; return -2; }
  if (P->win < 3 || P->win > KLT_MAXWIN || P->win_back < 3 || P->win_back > KLT_MAXWIN || P->max_level < 0 || P->max_level_back < 0) { h->err = "win must be in [3,31]"; return -1; }
  if (P->check_static && (!prev_age || !keep)) { h->err = "check_static needs prev_age and keep"; return -1; }
  cudaSetDevice(h->dev);
  auto nlevels = [&](int max_level, int win) { int levels = 0; int w = h->W, hh = h->H;
    for (int l = 0; l <= max_level && l < 8; l++) { levels = l; if (l < max_level) { const int w2 = (w + 1)/2, h2 = (hh + 1)/2; if (w2 <= win || h2 <= win) break; w = w2; hh = h2; } } return levels; };
  const int lf = nlevels(P->max_level, P->win), lb = nlevels(P->max_level_back, P->win_back), lmax = std::max(lf, lb);
  if (n > h->k_cap) { if (klt_scratch(h, std::max(n, 4096))) return -3; }
  FCK(cudaEventRecord(h->e0, h->s));
  if (!resident) {
    if (build_pyramid(h, 0, prev_gray, lmax, P->win, true)) return -3;      // both images with derivatives: each is "previous" once
    if (build_pyramid(h, 1, cur_gray, lmax, P->win, true)) return -3;
    h->have_pyr = h->have_pyr_cur = true;
  }
  FCK(cudaMemcpyAsync(h->k_prev, prev_pts, 2*(size_t)n*4, cudaMemcpyHostToDevice, h->s));
  FCK(cudaMemcpyAsync(h->k_next, P->use_initial_flow ? next_pts : prev_pts, 2*(size_t)n*4, cudaMemcpyHostToDevice, h->s));
  if (P->check_static) FCK(cudaMemcpyAsync(h->k_age, prev_age, (size_t)n*4, cudaMemcpyHostToDevice, h->s));
  FCK(cudaMemsetAsync(h->k_count, 0, 2*sizeof(int), h->s));
  auto levels_of = [&](int nl, int fwd) { KltLevels L; L.nlev = nl + 1;
    for (int l = 0; l <= nl; l++) { L.I[l] = h->pyr[fwd ? 0 : 1][l]; L.J[l] = h->pyr[fwd ? 1 : 0][l]; L.D[l] = fwd ? h->der[l] : h->der2[l]; L.w[l] = h->lw[l]; L.h[l] = h->lh[l]; } return L; };
  auto run = [&](const KltLevels& L, const float* from, float* to, uint8_t* st, int win, int max_count, double epsilon, int use_initial, float* eig) {
    const int mc = std::min(std::max(max_count, 0), 100); double eps = std::min(std::max(epsilon, 0.0), 10.0); eps *= eps;
    if (n > 0) klt_kernel<<<(n + KLT_WARPS - 1)/KLT_WARPS, KLT_WARPS*32, (size_t)KLT_WARPS*win*win*3*sizeof(short), h->s>>>(L, n, from, to, st, h->k_err, win, mc, (float)eps,
                                                                                                                        use_initial, (float)P->min_eig_threshold, eig);
  };
  const KltLevels LF = levels_of(lf, 1), LB = levels_of(lb, 0);
  run(LF, h->k_prev, h->k_next, h->k_st, P->win, P->max_count, P->epsilon, P->use_initial_flow, h->k_eig);
  if (P->use_initial_flow && n > 0) {
    // StaticFeatureTracker.cc:491-503: with OPTFLOW_USE_INITIAL_FLOW fewer than 10 successes -> track again from scratch
    int succ = 0;
    count_status_kernel<<<(n + 255)/256, 256, 0, h->s>>>(n, h->k_st, h->k_count);
    FCK(cudaMemcpyAsync(&succ, h->k_count, sizeof(int), cudaMemcpyDeviceToHost, h->s)); FCK(cudaStreamSynchronize(h->s));
    FCK(cudaMemsetAsync(h->k_count, 0, 2*sizeof(int), h->s));
    if (succ < 10) { FCK(cudaMemcpyAsync(h->k_next, h->k_prev, 2*(size_t)n*4, cudaMemcpyDeviceToDevice, h->s)); run(LF, h->k_prev, h->k_next, h->k_st, P->win, P->max_count, P->epsilon, 0, h->k_eig); }
  }
  FCK(cudaMemcpyAsync(h->k_back, h->k_next, 2*(size_t)n*4, cudaMemcpyDeviceToDevice, h->s));       // flags = 0: the backward search starts at the forward result
  run(LB, h->k_next, h->k_back, h->k_st2, P->win_back, P->max_count_back, P->epsilon_back, 0, nullptr);
  if (n > 0) klt_fb_filter_kernel<<<(n + 255)/256, 256, 0, h->s>>>(n, h->k_prev, h->k_next, h->k_back, h->k_st, h->k_st2, (float)P->max_fb_distance, h->k_st,
                                                                  P->check_static, h->mask, h->W, h->H, P->track, h->k_age, P->max_feature_track_age, h->k_keep, h->k_count);
  int counts[2] = {0, 0};
  FCK(cudaMemcpyAsync(next_pts, h->k_next, 2*(size_t)n*4, cudaMemcpyDeviceToHost, h->s));
  FCK(cudaMemcpyAsync(status, h->k_st, n, cudaMemcpyDeviceToHost, h->s));
  if (back_pts) FCK(cudaMemcpyAsync(back_pts, h->k_back, 2*(size_t)n*4, cudaMemcpyDeviceToHost, h->s));
  if (keep) FCK(cudaMemcpyAsync(keep, h->k_keep, n, cudaMemcpyDeviceToHost, h->s));
  FCK(cudaMemcpyAsync(counts, h->k_count, sizeof(counts), cudaMemcpyDeviceToHost, h->s));
  FCK(cudaEventRecord(h->e1, h->s));
  FCK(cudaStreamSynchronize(h->s));
  FCK(cudaGetLastError());
  if (n_status) *n_status = counts[0]; if (n_keep) *n_keep = counts[1];
  if (ms_device) FCK(cudaEventElapsedTime(ms_device, h->e0, h->e1));
  return 0;
}

// FeatureTracker::stereoTrack (FeatureTracker.cc:194-337): left -> right LK (21x21, 5 levels, OpenCV default criteria), then per
// matched point disparity = uL - uR, rejected when <= 1 px or uR < 0, depth = fx * baseline / disparity.  (The reference also
// runs the right -> left pass but its round-trip filter is commented out, :240-253, and a fundamental-matrix RANSAC sits between
// the LK status and the disparity test: host code outside section 8 -- final = status & ransac_mask & valid.)
__global__ void stereo_post_kernel(int n, const float* __restrict__ left, const float* __restrict__ right, const uint8_t* __restrict__ st, double fx,
                                   double baseline, double* __restrict__ depth, uint8_t* __restrict__ valid) {
  const int i = blockIdx.x*blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double uL = (double)left[2*i], uR = (double)right[2*i];
  const double disparity = uL - uR;
  const bool ok = st[i] && !(disparity <= 1.0 || right[2*i] < 0.0f);
  valid[i] = ok ? 1 : 0;
  depth[i] = ok ? fx*baseline/disparity : 0.0;
}
int dynofront_stereo_track(dynofront_handle h, const uint8_t* left_gray, const uint8_t* right_gray, int32_t n, const float* left_pts, float* right_pts,
                           uint8_t* status, double fx, double baseline, double* depth, uint8_t* valid, float* ms_device) {
  if (!h || !left_gray || !right_gray || n < 0 || !left_pts || !right_pts || !status || !depth || !valid) return -1;
  cudaSetDevice(h->dev);
  const int win = 21, max_level = 5;
  int levels = 0; { int w = h->W, hh = h->H; for (int l = 0; l <= max_level && l < 8; l++) { levels = l; if (l < max_level) { const int w2 = (w + 1)/2, h2 = (hh + 1)/2; if (w2 <= win || h2 <= win) break; w = w2; hh = h2; } } }
  if (n > h->k_cap) { if (klt_scratch(h, std::max(n, 4096))) return -3; }
  double* d_depth = nullptr;
  if (n > h->st_cap) { if (falloc(h, &h->st_depth, (size_t)std::max(n, 4096))) return -3; h->st_cap = std::max(n, 4096); }
  d_depth = h->st_depth;
  FCK(cudaEventRecord(h->e0, h->s));
  if (build_pyramid(h, 0, left_gray, levels, win, true)) return -3;
  if (build_pyramid(h, 1, right_gray, levels, win, false)) return -3;
  h->have_pyr = h->have_pyr_cur = false;
  FCK(cudaMemcpyAsync(h->k_prev, left_pts, 2*(size_t)n*4, cudaMemcpyHostToDevice, h->s));
  FCK(cudaMemcpyAsync(h->k_next, left_pts, 2*(size_t)n*4, cudaMemcpyHostToDevice, h->s));
  KltLevels L; L.nlev = levels + 1;
  for (int l = 0; l <= levels; l++) { L.I[l] = h->pyr[0][l]; L.J[l] = h->pyr[1][l]; L.D[l] = h->der[l]; L.w[l] = h->lw[l]; L.h[l] = h->lh[l]; }
  if (n > 0) {
    klt_kernel<<<(n + KLT_WARPS - 1)/KLT_WARPS, KLT_WARPS*32, (size_t)KLT_WARPS*win*win*3*sizeof(short), h->s>>>(L, n, h->k_prev, h->k_next, h->k_st, h->k_err, win, 30, 0.01f*0.01f,
                                                                                                                0, 1e-4f, h->k_eig);
    stereo_post_kernel<<<(n + 255)/256, 256, 0, h->s>>>(n, h->k_prev, h->k_next, h->k_st, fx, baseline, d_depth, h->k_keep);
  }
  FCK(cudaMemcpyAsync(right_pts, h->k_next, 2*(size_t)n*4, cudaMemcpyDeviceToHost, h->s));
  FCK(cudaMemcpyAsync(status, h->k_st, n, cudaMemcpyDeviceToHost, h->s));
  FCK(cudaMemcpyAsync(depth, d_depth, (size_t)n*8, cudaMemcpyDeviceToHost, h->s));
  FCK(cudaMemcpyAsync(valid, h->k_keep, n, cudaMemcpyDeviceToHost, h->s));
  FCK(cudaEventRecord(h->e1, h->s));
  FCK(cudaStreamSynchronize(h->s));
  FCK(cudaGetLastError());
  if (ms_device) FCK(cudaEventElapsedTime(ms_device, h->e0, h->e1));
  return 0;
}

int dynofront_klt_last_min_eig(dynofront_handle h, int32_t n, float* out) {
  if (!h || !out || n < 0 || n > h->k_cap || !h->k_eig) return -1;
  cudaSetDevice(h->dev);
  FCK(cudaMemcpy(out, h->k_eig, 2*(size_t)n*4, cudaMemcpyDeviceToHost));
  return 0;
}

int dynofront_track_static_flow(dynofront_handle h, int32_t n_prev, const double* prev_pred_kp, const int32_t* prev_age, const uint8_t* prev_usable,
                                int32_t n_det, const int32_t* det_xy, int32_t cell_size, int32_t max_features, int64_t* next_tracklet_id,
                                uint8_t* acc_prev, double* flow_prev, double* pred_prev, int32_t* age_out,
                                uint8_t* acc_det, double* flow_det, double* pred_det, int64_t* tracklet_det, int32_t* n_tracked, int32_t* n_detected) {
  if (!h || n_prev < 0 || n_det < 0 || cell_size <= 0 || !next_tracklet_id) return -1;
  if ((n_prev && (!prev_pred_kp || !prev_age || !prev_usable || !acc_prev || !flow_prev || !pred_prev || !age_out)) ||
      (n_det && (!det_xy || !acc_det || !flow_det || !pred_det || !tracklet_det))) { h->err = "null array"; return -1; }
  cudaSetDevice(h->dev);
  const int ncols = (int)std::ceil((double)h->W/cell_size), nrows = (int)std::ceil((double)h->H/cell_size), ncell = ncols*nrows;
  const int nmax = std::max(std::max(n_prev, n_det), 1);
  if (nmax > h->sf_cap || ncell > h->sf_cells) {
    const int cap = std::max(nmax, 4096), cells = std::max(ncell, h->sf_cells);
    int rc = 0;
    rc |= falloc(h, &h->sf_kp, 2*(size_t)cap); rc |= falloc(h, &h->sf_age, cap); rc |= falloc(h, &h->sf_use, cap); rc |= falloc(h, &h->sf_det, 2*(size_t)cap);
    rc |= falloc(h, &h->sf_cell, cap); rc |= falloc(h, &h->sf_win, cells); rc |= falloc(h, &h->sf_win2, cells); rc |= falloc(h, &h->sf_cnt, 2);
    rc |= falloc(h, &h->sf_pass, cap); rc |= falloc(h, &h->sf_acc, cap); rc |= falloc(h, &h->sf_out, 4*(size_t)cap); rc |= falloc(h, &h->sf_oage, cap); rc |= falloc(h, &h->sf_otid, cap);
    if (rc) return -3;
    h->sf_cap = cap; h->sf_cells = cells;
  }
  fill_i32_kernel<<<(ncell + 255)/256, 256, 0, h->s>>>(h->sf_win, ncell, 0x7fffffff);
  fill_i32_kernel<<<(ncell + 255)/256, 256, 0, h->s>>>(h->sf_win2, ncell, 0x7fffffff);
  FCK(cudaMemsetAsync(h->sf_cnt, 0, 2*sizeof(int), h->s));
  std::vector<double> o4; std::vector<uint8_t> acc; int cnt[2] = {0, 0};
  if (n_prev) {
    FCK(cudaMemcpyAsync(h->sf_kp, prev_pred_kp, 2*(size_t)n_prev*8, cudaMemcpyHostToDevice, h->s));
    FCK(cudaMemcpyAsync(h->sf_age, prev_age, (size_t)n_prev*4, cudaMemcpyHostToDevice, h->s));
    FCK(cudaMemcpyAsync(h->sf_use, prev_usable, (size_t)n_prev, cudaMemcpyHostToDevice, h->s));
    sf_prev_kernel<<<(n_prev + 255)/256, 256, 0, h->s>>>(n_prev, h->sf_kp, h->sf_use, h->flow, h->mask, h->W, h->H, cell_size, ncols, h->sf_cell, h->sf_pass, h->sf_out, h->sf_win);
    sf_prev_resolve_kernel<<<(n_prev + 255)/256, 256, 0, h->s>>>(n_prev, h->sf_cell, h->sf_pass, h->sf_win, h->sf_age, h->sf_acc, h->sf_out, h->sf_oage, h->sf_cnt);
    o4.resize(4*(size_t)n_prev);
    FCK(cudaMemcpyAsync(acc_prev, h->sf_acc, n_prev, cudaMemcpyDeviceToHost, h->s));
    FCK(cudaMemcpyAsync(o4.data(), h->sf_out, o4.size()*8, cudaMemcpyDeviceToHost, h->s));
    FCK(cudaMemcpyAsync(age_out, h->sf_oage, (size_t)n_prev*4, cudaMemcpyDeviceToHost, h->s));
    FCK(cudaStreamSynchronize(h->s));
    for (int i = 0; i < n_prev; i++) { flow_prev[2*i] = o4[4*(size_t)i]; flow_prev[2*i + 1] = o4[4*(size_t)i + 1]; pred_prev[2*i] = o4[4*(size_t)i + 2]; pred_prev[2*i + 1] = o4[4*(size_t)i + 3]; }
  }
  if (n_det) {
    FCK(cudaMemcpyAsync(h->sf_det, det_xy, 2*(size_t)n_det*4, cudaMemcpyHostToDevice, h->s));
    sf_det_kernel<<<(n_det + 255)/256, 256, 0, h->s>>>(n_det, h->sf_det, h->flow, h->mask, h->W, h->H, cell_size, ncols, h->sf_win, h->sf_cell, h->sf_pass, h->sf_out, h->sf_win2);
    sf_det_resolve_kernel<<<1, 1024, 0, h->s>>>(n_det, h->sf_cell, h->sf_pass, h->sf_win2, h->sf_cnt, max_features, (long long)*next_tracklet_id, h->sf_acc, h->sf_out, h->sf_otid, h->sf_cnt + 1);
    o4.resize(4*(size_t)n_det);
    FCK(cudaMemcpyAsync(acc_det, h->sf_acc, n_det, cudaMemcpyDeviceToHost, h->s));
    FCK(cudaMemcpyAsync(o4.data(), h->sf_out, o4.size()*8, cudaMemcpyDeviceToHost, h->s));
    FCK(cudaMemcpyAsync(tracklet_det, h->sf_otid, (size_t)n_det*8, cudaMemcpyDeviceToHost, h->s));
    FCK(cudaStreamSynchronize(h->s));
    for (int j = 0; j < n_det; j++) { flow_det[2*j] = o4[4*(size_t)j]; flow_det[2*j + 1] = o4[4*(size_t)j + 1]; pred_det[2*j] = o4[4*(size_t)j + 2]; pred_det[2*j + 1] = o4[4*(size_t)j + 3]; }
  }
  FCK(cudaMemcpyAsync(cnt, h->sf_cnt, sizeof(cnt), cudaMemcpyDeviceToHost, h->s)); FCK(cudaStreamSynchronize(h->s));
  FCK(cudaGetLastError());
  *next_tracklet_id += cnt[1];
  if (n_tracked) *n_tracked = cnt[0]; if (n_detected) *n_detected = cnt[1];
  return 0;
}

// ---------------------------------------------------------------------------------------------------- ANMS / sampleDynamic host side
static int anms_prepare(dynofront_ctx* h) {       // the ANMS kernel may use all the shared memory a block can opt into
  if (h->anms_smem) return 0;
  int optin = 0; cudaFuncAttributes fa;
  FCK(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->dev));
  FCK(cudaFuncGetAttributes(&fa, anms_range_tree_kernel));
  const int dyn = (optin - (int)fa.sharedSizeBytes) & ~15;
  FCK(cudaFuncSetAttribute(anms_range_tree_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn));
  h->anms_smem = dyn;
  return 0;
}
static int sd_scratch(dynofront_ctx* h, long long capacity) {
  if (anms_prepare(h)) return -3;
  const size_t npx = (size_t)h->W*h->H;
  if (!h->sd_idx) {
    const long long bmw = (long long)((h->W + 31)/32)*h->H;       // a bounding box of cells is at most the whole image
    int rc = 0;
    rc |= falloc(h, &h->sd_idx, npx); rc |= falloc(h, &h->sd_off, ST_MAXOBJ); rc |= falloc(h, &h->sd_K, ST_MAXOBJ); rc |= falloc(h, &h->sd_nsel, ST_MAXOBJ);
    rc |= falloc(h, &h->sd_sel, 2*npx); rc |= falloc(h, &h->sd_out, npx); rc |= falloc(h, &h->sd_pts, npx);
    rc |= falloc(h, &h->sd_bm, (size_t)(ST_MAXOBJ*bmw)); rc |= falloc(h, &h->sd_bm_off, ST_MAXOBJ);
    if (rc) return -3;
    std::vector<long long> bo(ST_MAXOBJ);
    for (int o = 0; o < ST_MAXOBJ; o++) bo[o] = o*bmw;
    FCK(cudaMemcpy(h->sd_bm_off, bo.data(), ST_MAXOBJ*sizeof(long long), cudaMemcpyHostToDevice));
  }
  if (capacity > h->sd_host_cap) {                 // mapped pinned staging: inputs, per-object stats, features
    if (h->sd_host) { cudaFreeHost(h->sd_host); h->sd_host = h->sd_host_dev = nullptr; h->sd_host_cap = -1; }
    const long long cap = std::max<long long>(capacity, 1024);
    FCK(cudaHostAlloc((void**)&h->sd_host, 6*ST_MAXOBJ*4 + (size_t)cap*(6*8 + 8), cudaHostAllocMapped));
    FCK(cudaHostGetDevicePointer((void**)&h->sd_host_dev, h->sd_host, 0));
    h->sd_host_cap = cap;
  }
  return 0;
}

int dynofront_sample_dynamic(dynofront_handle h, int32_t nobj, const int32_t* objects, const int32_t* num_track, int32_t max_features,
                             float tolerance, const dynofront_track_params* prm, int64_t* next_tracklet_id, int32_t* candidates,
                             int32_t* zero_flow, int32_t* selected, int32_t* selected_offset, double* keypoint, double* flow_out,
                             double* predicted_keypoint, int64_t* tracklet, int64_t capacity, float* ms_device) {
  if (!h || !prm || !next_tracklet_id || nobj < 0 || nobj > ST_MAXOBJ || capacity < 0) return -1;
  if (nobj && (!objects || !num_track || !candidates || !selected || !selected_offset)) { h->err = "null per-object array"; return -1; }
  if (capacity && (!keypoint || !flow_out || !predicted_keypoint || !tracklet)) { h->err = "null per-feature array"; return -1; }
  cudaSetDevice(h->dev);
  if (sd_scratch(h, capacity)) return -3;
  const size_t npx = (size_t)h->W*h->H; const int ntiles = (int)((npx + ST_TILE - 1)/ST_TILE);
  int32_t* in = (int32_t*)h->sd_host; int32_t* stats = in + 2*ST_MAXOBJ;
  int32_t* stats_dev = (int32_t*)h->sd_host_dev + 2*ST_MAXOBJ;
  double* feat = (double*)(h->sd_host + 6*ST_MAXOBJ*4); long long* tid = (long long*)(feat + 6*h->sd_host_cap);
  double* feat_dev = (double*)(h->sd_host_dev + 6*ST_MAXOBJ*4); long long* tid_dev = (long long*)(feat_dev + 6*h->sd_host_cap);
  std::memcpy(in, objects, (size_t)nobj*4); std::memcpy(in + ST_MAXOBJ, num_track, (size_t)nobj*4);
  FCK(cudaEventRecord(h->e0, h->s));
  if (!h->det_work_valid) prepare_det_work(h);
  if (nobj > 0) {
    FCK(cudaMemcpyAsync(h->d_objs, in, (size_t)nobj*4, cudaMemcpyHostToDevice, h->s));
    FCK(cudaMemcpyAsync(h->sd_K, in + ST_MAXOBJ, (size_t)nobj*4, cudaMemcpyHostToDevice, h->s));
    FCK(cudaMemsetAsync(h->d_zero, 0, ST_MAXOBJ*4, h->s));
    sc_count_kernel<<<ntiles, ST_TILE, 0, h->s>>>(npx, h->W, h->H, h->det_work, h->mask, h->flow, h->d_objs, nobj, *prm, h->tile_cnt, h->d_zero);
    sc_scan_kernel<<<1, ST_MAXOBJ, 0, h->s>>>(ntiles, nobj, h->tile_cnt, h->obj_tot);
    sd_plan_kernel<<<1, 32, 0, h->s>>>(nobj, h->obj_tot, h->sd_K, max_features, h->sd_off, h->sd_K);
    sc_scatter_kernel<<<ntiles, ST_TILE, 0, h->s>>>(npx, h->W, h->H, h->det_work, h->mask, h->flow, h->d_objs, nobj, *prm, h->tile_cnt, h->sd_off,
                                                    h->sd_idx, (long long)npx);
    AnmsArgs a{h->sd_off, h->obj_tot, h->sd_K, nullptr, h->sd_idx, h->W, tolerance, h->W, h->H, h->sd_pts, h->sd_bm, h->sd_bm_off,
               h->sd_sel, (long long)npx, h->sd_out, h->sd_nsel, h->anms_smem};
    anms_range_tree_kernel<<<nobj, ANMS_THREADS, h->anms_smem, h->s>>>(a);
    sd_construct_kernel<<<nobj, 128, 0, h->s>>>(nobj, h->sd_off, h->obj_tot, h->d_zero, h->sd_nsel, h->sd_out, h->sd_idx, h->W, h->flow,
                                                capacity, (long long)*next_tracklet_id, stats_dev, feat_dev, tid_dev);
  }
  FCK(cudaEventRecord(h->e1, h->s));
  FCK(cudaStreamSynchronize(h->s));
  FCK(cudaGetLastError());
  long long total = 0;
  for (int o = 0; o < nobj; o++) {
    candidates[o] = stats[o]; if (zero_flow) zero_flow[o] = stats[ST_MAXOBJ + o];
    selected[o] = stats[2*ST_MAXOBJ + o]; selected_offset[o] = stats[3*ST_MAXOBJ + o]; total += selected[o];
  }
  if (ms_device) FCK(cudaEventElapsedTime(ms_device, h->e0, h->e1));
  if (total > capacity) { h->err = "capacity < " + std::to_string(total) + " selected features"; return -1; }
  for (long long f = 0; f < total; f++) {
    keypoint[2*f] = feat[6*f]; keypoint[2*f + 1] = feat[6*f + 1]; flow_out[2*f] = feat[6*f + 2]; flow_out[2*f + 1] = feat[6*f + 3];
    predicted_keypoint[2*f] = feat[6*f + 4]; predicted_keypoint[2*f + 1] = feat[6*f + 5]; tracklet[f] = tid[f];
  }
  *next_tracklet_id += total;
  return 0;
}

int dynofront_anms_range_tree(dynofront_handle h, int32_t n_lists, const int32_t* counts, const float* xy, const int32_t* num_ret_points,
                              float tolerance, int32_t cols, int32_t rows, int32_t* indices, int32_t* n_selected) {
  if (!h || n_lists < 0 || (n_lists && (!counts || !num_ret_points || !n_selected))) return -1;
  if (cols <= 0 || rows <= 0 || cols > 65535 || rows > 65535) { h->err = "cols / rows must be in [1, 65535] (u16 cells)"; return -1; }
  cudaSetDevice(h->dev);
  if (anms_prepare(h)) return -3;
  std::vector<int> meta(4*(size_t)n_lists);         // off, count, K, (selected)
  std::vector<long long> bm_off(std::max(n_lists, 1));
  long long total = 0, bm_total = 0;
  for (int l = 0; l < n_lists; l++) {
    if (counts[l] < 0) { h->err = "negative list length"; return -1; }
    meta[l] = (int)total; meta[n_lists + l] = counts[l]; meta[2*n_lists + l] = num_ret_points[l];
    float bx0 = 65536.f, bx1 = -1.f, by0 = 65536.f, by1 = -1.f;
    for (long long i = total; i < total + counts[l]; i++) {
      const float x = xy[2*i], y = xy[2*i + 1];
      if (!(x >= 0.f && x < 65536.f && y >= 0.f && y < 65536.f)) { h->err = "coordinates must lie in [0, 65536) (u16 cells)"; return -1; }
      bx0 = std::min(bx0, x); bx1 = std::max(bx1, x); by0 = std::min(by0, y); by1 = std::max(by1, y);
    }
    total += counts[l];
    if (total > INT32_MAX/2) { h->err = "too many points"; return -1; }
    bm_off[l] = bm_total;                            // global bitmap only where the kernel cannot keep it in shared memory
    if (counts[l] > 0) {
      const long long words = (long long)((((int)bx1 - (int)bx0) >> 5) + 1)*((int)by1 - (int)by0 + 1);
      if (4*words > h->anms_smem) bm_total += words;
    }
  }
  if (n_lists == 0) return 0;
  if (total > h->an_cap) {
    const int cap = (int)std::max<long long>(2*total, 4096);
    if (falloc(h, &h->an_xy, 2*(size_t)cap) || falloc(h, &h->an_pts, cap) || falloc(h, &h->an_sel, 2*(size_t)cap) || falloc(h, &h->an_out, cap)) return -3;
    h->an_cap = cap;
  }
  if (n_lists > h->an_lists) {
    const int cap = std::max(2*n_lists, 64);
    if (falloc(h, &h->an_meta, 4*(size_t)cap) || falloc(h, &h->an_bm_off, cap)) return -3;
    h->an_lists = cap;
  }
  if (bm_total > h->an_bm_cap) { if (falloc(h, &h->an_bm, (size_t)bm_total)) return -3; h->an_bm_cap = bm_total; }
  FCK(cudaMemcpyAsync(h->an_meta, meta.data(), meta.size()*4, cudaMemcpyHostToDevice, h->s));
  FCK(cudaMemcpyAsync(h->an_bm_off, bm_off.data(), (size_t)n_lists*8, cudaMemcpyHostToDevice, h->s));
  if (total) FCK(cudaMemcpyAsync(h->an_xy, xy, 2*(size_t)total*4, cudaMemcpyHostToDevice, h->s));
  AnmsArgs a{h->an_meta, h->an_meta + n_lists, h->an_meta + 2*n_lists, h->an_xy, nullptr, 0, tolerance, cols, rows, h->an_pts, h->an_bm, h->an_bm_off,
             h->an_sel, (long long)h->an_cap, h->an_out, h->an_meta + 3*n_lists, h->anms_smem};
  anms_range_tree_kernel<<<n_lists, ANMS_THREADS, h->anms_smem, h->s>>>(a);
  if (total && indices) FCK(cudaMemcpyAsync(indices, h->an_out, (size_t)total*4, cudaMemcpyDeviceToHost, h->s));
  FCK(cudaMemcpyAsync(n_selected, h->an_meta + 3*n_lists, (size_t)n_lists*4, cudaMemcpyDeviceToHost, h->s));
  FCK(cudaStreamSynchronize(h->s));
  FCK(cudaGetLastError());
  return 0;
}

int dynofront_anms_tie_order(int32_t n, int32_t* out) {
  if (n < 0 || (n && !out)) return -1;
  for (int k = 0; k < n; k++) out[k] = anms_tie_source(n, k);
  return 0;
}

int dynofront_get_pyramid_level(dynofront_handle h, int32_t which, int32_t level, int32_t* w, int32_t* hgt, uint8_t* img, int16_t* deriv) {
  if (!h || which < 0 || which > 1 || level < 0 || level >= (int)h->lw.size()) return -1;
  cudaSetDevice(h->dev);
  if (w) *w = h->lw[level]; if (hgt) *hgt = h->lh[level];
  const size_t n = (size_t)h->lw[level]*h->lh[level];
  if (img) FCK(cudaMemcpy(img, h->pyr[which][level], n, cudaMemcpyDeviceToHost));
  if (deriv) FCK(cudaMemcpy(deriv, h->der[level], 2*n*sizeof(short), cudaMemcpyDeviceToHost));
  return 0;
}

}  // extern "C"
