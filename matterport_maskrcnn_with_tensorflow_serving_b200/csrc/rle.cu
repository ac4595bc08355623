// rle.cu -- COCO run-length masks straight from the 28x28 tiles (SURVEY.md 8f rank 4: the second
// compact format it names; the output of /root/reference/serve.py:147 re-encoded).
//
// EXTENSION, not the reference layout.  For every kept instance the result is the
// "uncompressed RLE" of pycocotools, {'size': [H, W], 'counts': [...]}: the [H, W] mask read in
// COLUMN-major order as alternating runs of zeros and ones, starting with zeros (a leading 0
// when the first pixel is set).  The mask itself is never materialised: the kernels evaluate the
// same samples as mrx_mask_expand (same exact integer source coordinates, same fp32 weights,
// same two fused multiply-adds -- horizontal then vertical), but with lanes on 32 adjacent
// COLUMNS walking DOWN the box, so each lane meets the pixels of its column in run-length
// order and only has to note where the value changes.
//
//   rle_walk_kernel<false>   per (instance, 32-column block): number of transitions per column
//   rle_scan_kernel          per instance: exclusive scan over its columns, instance total
//   rle_offsets_kernel       exclusive scan of the instance totals (one CTA)
//   rle_walk_kernel<true>    the same walk again, now writing each transition's flat position
//                            x*H + y at (instance base + column offset + running index)
//   rle_counts_kernel        positions -> run lengths (differences, closing run to H*W)
//
// Column seams: column x continues at (x+1, 0) after (x, H-1).  Outside its box an instance is
// zero, so a column starts after a zero unless the box spans the full height (then it starts
// after the previous column's last pixel), and a run still open at the last box row is closed
// by a transition at the first pixel below the box (or at the top of the next column).
//
// Instruction-bound on the in-box samples like the packed expand kernel; the output is a few
// bytes per run (a few MB per batch of real masks).
#include "expand.cuh"

namespace mrx {

namespace rle {

constexpr int kWalkWarps = 8;

struct RleParams {
  const float *tiles;         // [B,R,mh,mw]
  const int *tile_index;      // [B,R] or NULL
  const int4 *boxes;          // [B,R]
  const int *counts;          // [B]
  const int *geom;            // [B,8]
  int *col_count;             // [B,R,max_w]: transitions per column -> exclusive offsets (scan)
  long long *inst_off;        // [B*R + 1]: totals -> exclusive offsets of the instances
  unsigned int *positions;    // [total] flat positions of the transitions (write pass)
  int B, R, mh, mw, max_w;
};

// One warp: instance k of image b, columns [32*cb, 32*cb + 32).
template <bool kWrite>
__global__ void __launch_bounds__(kWalkWarps * 32)
rle_walk_kernel(const RleParams p) {
  const int lane = threadIdx.x & 31;
  const int cb = blockIdx.x * kWalkWarps + (threadIdx.x >> 5);
  const int k = blockIdx.y, b = blockIdx.z;
  if (k >= p.counts[b]) return;
  const int H = p.geom[b * MRX_GEOM_INTS + 0], W = p.geom[b * MRX_GEOM_INTS + 1];
  const int4 bx = __ldg(p.boxes + static_cast<size_t>(b) * p.R + k);   // (y1, x1, y2, x2)
  const bool sane = bx.x >= 0 && bx.y >= 0 && bx.z <= H && bx.w <= W && bx.z > bx.x && bx.w > bx.y;
  if (!sane || (cb << 5) >= bx.w || (cb << 5) + 32 <= bx.y) return;
  const int mh = p.mh, mw = p.mw;
  const int bh = bx.z - bx.x, bw = bx.w - bx.y;
  const int D = 2 * bw, Dy = 2 * bh;
  const float invD = __fdiv_rn(1.0f, static_cast<float>(D));
  const float invDy = __fdiv_rn(1.0f, static_cast<float>(Dy));
  const int tile = p.tile_index != nullptr ? __ldg(p.tile_index + static_cast<size_t>(b) * p.R + k) : k;
  const bool lanecol = lane >= 1 && lane <= mw;      // lane l holds tile column l - 1
  const int lcol = min(max(lane - 1, 0), mw - 1);
  const float *tp = p.tiles + (static_cast<size_t>(b) * p.R + tile) * mh * mw + lcol;
  auto raw = [&](int j) -> float {   // tile row j in lane-column layout, zero outside the tile
    const float v = __ldg(tp + static_cast<unsigned>(min(max(j, 0), mh - 1) * mw));
    return (lanecol && j >= 0 && j < mh) ? v : 0.f;
  };
  // horizontal source coordinate of column x: taps idx, idx + 1 of the zero-padded tile row
  auto hcoord = [&](int x, int &idx, float &wx) {
    const int A = mw * (2 * (x - bx.y) + 1) - bw;
    int i0 = __float2int_rd(static_cast<float>(A) * invD);
    int rem = A - i0 * D;
    if (rem < 0) {
      --i0;
      rem += D;
    } else if (rem >= D) {
      ++i0;
      rem -= D;
    }
    idx = min(max(i0 + 1, 0), 30);
    wx = static_cast<float>(rem) * invD;
  };
  const int x = (cb << 5) + lane;
  const bool colvalid = x >= bx.y && x < bx.w;
  int idx;
  float wx;
  hcoord(x, idx, wx);
  auto hrow = [&](float rv, int id, float w) -> float {
    const float lo = __shfl_sync(0xffffffffu, rv, id);
    const float hi = __shfl_sync(0xffffffffu, rv, id + 1);
    return fmaf(w, hi - lo, lo);
  };
  const float thr = colvalid ? 0.5f : __int_as_float(0x7f800000);

  // exact vertical source coordinate of the first box row
  int jcur, remy;
  {
    const int Ay = mh - bh;   // mh * (2*0 + 1) - bh
    int j0 = __float2int_rd(static_cast<float>(Ay) * invDy);
    int rem = Ay - j0 * Dy;
    if (rem < 0) {
      --j0;
      rem += Dy;
    } else if (rem >= Dy) {
      ++j0;
      rem -= Dy;
    }
    jcur = j0;
    remy = rem;
  }
  int stepQy = 0;
  if (Dy <= 2 * mh) stepQy = (2 * mh) / Dy;
  const int stepRy = 2 * mh - stepQy * Dy;

  const bool full = bx.x == 0 && bx.z == H;          // column seams carry the previous column's bit
  unsigned int *out = nullptr;
  if (kWrite) {
    const size_t inst = static_cast<size_t>(b) * p.R + k;
    out = p.positions + p.inst_off[inst] + (colvalid ? p.col_count[inst * p.max_w + x] : 0);
  }
  const unsigned base = static_cast<unsigned>(x) * static_cast<unsigned>(H);
  int n = 0;
  bool prev = false;
  // With a full-height box the first row's predecessor is the previous column's LAST pixel:
  // one extra sample (column x - 1, row H - 1), evaluated exactly as that column's own walk
  // evaluates it.
  bool prev_top = false;
  if (full) {
    // last row's vertical coordinate (same exact arithmetic, from the row index)
    const int Ay = mh * (2 * (bh - 1) + 1) - bh;
    int jl = __float2int_rd(static_cast<float>(Ay) * invDy);
    int reml = Ay - jl * Dy;
    if (reml < 0) {
      --jl;
      reml += Dy;
    } else if (reml >= Dy) {
      ++jl;
      reml -= Dy;
    }
    int idp;
    float wxp;
    hcoord(x - 1, idp, wxp);
    const float rt = raw(jl), rbv = raw(jl + 1);
    const float htl = hrow(rt, idp, wxp), hbl = hrow(rbv, idp, wxp);
    const float vl = fmaf(static_cast<float>(reml) * invDy, hbl - htl, htl);
    prev_top = colvalid && x - 1 >= bx.y && vl >= 0.5f;
  }
  prev = prev_top;

  int j0 = jcur;
  float ht = hrow(raw(jcur), idx, wx), hb = hrow(raw(jcur + 1), idx, wx);
  float rawn = raw(jcur + 2);
  float dh = hb - ht;
  bool cur = false;
  for (int r = bx.x; r < bx.z; ++r) {
    if (j0 != jcur) {   // warp-uniform
      if (j0 == jcur + 1) {
        ht = hb;
        hb = hrow(rawn, idx, wx);
      } else {
        ht = hrow(raw(j0), idx, wx);
        hb = hrow(raw(j0 + 1), idx, wx);
      }
      jcur = j0;
      rawn = raw(jcur + 2);
      dh = hb - ht;
    }
    const float v = fmaf(static_cast<float>(remy) * invDy, dh, ht);
    cur = v >= thr;
    if (cur != prev) {
      if (kWrite) out[n] = base + static_cast<unsigned>(r);
      ++n;
    }
    prev = cur;
    remy += stepRy;
    j0 += stepQy;
    if (remy >= Dy) {
      remy -= Dy;
      ++j0;
    }
  }
  // a run still open at the last box row ends at the next pixel in column-major order -- below
  // the box, or the top of the next column -- unless that pixel is the next column of a
  // full-height box (its own top comparison sees it) or lies past the end of the image
  if (cur) {
    const bool next_is_box = full && x + 1 < bx.w;
    const unsigned long long pend = bx.z < H ? static_cast<unsigned long long>(base) + bx.z
                                             : static_cast<unsigned long long>(base) + H;
    if (!next_is_box && pend < static_cast<unsigned long long>(H) * W) {
      if (kWrite) out[n] = static_cast<unsigned>(pend);
      ++n;
    }
  }
  if (!kWrite && colvalid) p.col_count[(static_cast<size_t>(b) * p.R + k) * p.max_w + x] = n;
}

// One CTA per instance: exclusive scan of its columns' transition counts (in place), total out.
__global__ void __launch_bounds__(256)
rle_scan_kernel(const RleParams p) {
  const int k = blockIdx.x, b = blockIdx.y;
  const size_t inst = static_cast<size_t>(b) * p.R + k;
  __shared__ int s_warp[8];
  __shared__ int s_carry;
  if (k >= p.counts[b]) {
    if (threadIdx.x == 0) p.inst_off[inst] = 0;
    return;
  }
  const int H = p.geom[b * MRX_GEOM_INTS + 0], W = p.geom[b * MRX_GEOM_INTS + 1];
  const int4 bx = p.boxes[inst];
  const bool sane = bx.x >= 0 && bx.y >= 0 && bx.z <= H && bx.w <= W && bx.z > bx.x && bx.w > bx.y;
  const int x1 = sane ? bx.y : 0, x2 = sane ? bx.w : 0;
  int *cc = p.col_count + inst * p.max_w;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (int base = x1; base < x2; base += 256) {
    const int x = base + threadIdx.x;
    const int v = x < x2 ? cc[x] : 0;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += u;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    int before = s_carry;
    for (int w = 0; w < warp; ++w) before += s_warp[w];
    if (x < x2) cc[x] = before + incl - v;
    __syncthreads();
    if (threadIdx.x == 255) s_carry = before + incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) p.inst_off[inst] = s_carry;
}

// Exclusive scan of the n instance totals in place; inst_off[n] = grand total.  One CTA.
__global__ void __launch_bounds__(1024)
rle_offsets_kernel(long long *inst_off, int n) {
  __shared__ long long s_warp[32];
  __shared__ long long s_carry;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (int base = 0; base < n; base += 1024) {
    const int i = base + threadIdx.x;
    const long long v = i < n ? inst_off[i] : 0;
    long long incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const long long u = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += u;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    long long before = s_carry;
    for (int w = 0; w < warp; ++w) before += s_warp[w];
    if (i < n) inst_off[i] = before + incl - v;
    __syncthreads();
    if (threadIdx.x == 1023) s_carry = before + incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) inst_off[n] = s_carry;
}

// positions -> run lengths.  Instance i has T = inst_off[i+1] - inst_off[i] transitions and
// T + 1 runs; its runs start at counts + inst_off[i] + i.
__global__ void __launch_bounds__(256)
rle_counts_kernel(const unsigned int *__restrict__ positions, const long long *__restrict__ inst_off,
                  const int *__restrict__ counts_per_image, const int *__restrict__ geom, int R,
                  unsigned int *__restrict__ counts) {
  const int k = blockIdx.x, b = blockIdx.y;
  if (k >= counts_per_image[b]) return;
  const size_t inst = static_cast<size_t>(b) * R + k;
  const long long lo = inst_off[inst], hi = inst_off[inst + 1];
  const unsigned total = static_cast<unsigned>(geom[b * MRX_GEOM_INTS + 0]) *
                         static_cast<unsigned>(geom[b * MRX_GEOM_INTS + 1]);
  unsigned int *o = counts + lo + inst;
  const long long T = hi - lo;
  for (long long j = threadIdx.x; j <= T; j += 256) {
    const unsigned a = j == 0 ? 0u : positions[lo + j - 1];
    const unsigned e = j == T ? total : positions[lo + j];
    o[j] = e - a;
  }
}

}  // namespace rle

int exclusive_scan_i64(long long *d, int n, cudaStream_t stream) {
  rle::rle_offsets_kernel<<<1, 1024, 0, stream>>>(d, n);
  MRX_LAUNCH_CHECK("rle_offsets_kernel");
  return MRX_OK;
}

}  // namespace mrx

using namespace mrx;

static int fill_rle_params(rle::RleParams &prm, const float *d_tiles, const int *d_tile_index,
                           const int *d_boxes, const int *d_counts, const int *d_geom,
                           int *d_col_count, long long *d_inst_off, unsigned int *d_positions,
                           int B, int R, int mh, int mw, int max_w) {
  MRX_CHECK_ARG(d_tiles && d_boxes && d_counts && d_geom && d_col_count && d_inst_off,
                "mrx_rle: null pointer");
  MRX_CHECK_ARG(B >= 1 && B <= 65535 && R >= 1 && R <= 65535 && max_w >= 1,
                "mrx_rle: bad sizes B=%d R=%d max_w=%d", B, R, max_w);
  MRX_CHECK_SUPPORTED(mh >= 2 && mh <= MRX_MAX_MASK_DIM && mw >= 4 && mw <= 30,
                      "mrx_rle: mask tile %dx%d unsupported (2<=mh<=%d, 4<=mw<=30)", mh, mw,
                      MRX_MAX_MASK_DIM);
  prm.tiles = d_tiles;
  prm.tile_index = d_tile_index;
  prm.boxes = reinterpret_cast<const int4 *>(d_boxes);
  prm.counts = d_counts;
  prm.geom = d_geom;
  prm.col_count = d_col_count;
  prm.inst_off = d_inst_off;
  prm.positions = d_positions;
  prm.B = B;
  prm.R = R;
  prm.mh = mh;
  prm.mw = mw;
  prm.max_w = max_w;
  return MRX_OK;
}

extern "C" int mrx_rle_count(const float *d_tiles, const int *d_tile_index, const int *d_boxes,
                             const int *d_counts, const int *d_geom, int *d_col_count,
                             long long *d_inst_off, int B, int R, int mh, int mw, int max_w,
                             void *stream) {
  if (B == 0) return MRX_OK;
  rle::RleParams prm;
  if (int rc = fill_rle_params(prm, d_tiles, d_tile_index, d_boxes, d_counts, d_geom, d_col_count,
                               d_inst_off, nullptr, B, R, mh, mw, max_w))
    return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int cblocks = (max_w + 31) >> 5;
  dim3 grid((cblocks + rle::kWalkWarps - 1) / rle::kWalkWarps, R, B);
  rle::rle_walk_kernel<false><<<grid, rle::kWalkWarps * 32, 0, st>>>(prm);
  MRX_LAUNCH_CHECK("rle_walk_kernel<count>");
  rle::rle_scan_kernel<<<dim3(R, B), 256, 0, st>>>(prm);
  MRX_LAUNCH_CHECK("rle_scan_kernel");
  return exclusive_scan_i64(d_inst_off, B * R, st);
}

extern "C" int mrx_rle_write(const float *d_tiles, const int *d_tile_index, const int *d_boxes,
                             const int *d_counts, const int *d_geom, int *d_col_count,
                             long long *d_inst_off, unsigned int *d_positions,
                             unsigned int *d_run_lengths, int B, int R, int mh, int mw, int max_w,
                             void *stream) {
  if (B == 0) return MRX_OK;
  MRX_CHECK_ARG(d_positions && d_run_lengths, "mrx_rle_write: null pointer");
  rle::RleParams prm;
  if (int rc = fill_rle_params(prm, d_tiles, d_tile_index, d_boxes, d_counts, d_geom, d_col_count,
                               d_inst_off, d_positions, B, R, mh, mw, max_w))
    return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int cblocks = (max_w + 31) >> 5;
  dim3 grid((cblocks + rle::kWalkWarps - 1) / rle::kWalkWarps, R, B);
  rle::rle_walk_kernel<true><<<grid, rle::kWalkWarps * 32, 0, st>>>(prm);
  MRX_LAUNCH_CHECK("rle_walk_kernel<write>");
  rle::rle_counts_kernel<<<dim3(R, B), 256, 0, st>>>(d_positions, d_inst_off, d_counts, d_geom, R,
                                                     d_run_lengths);
  MRX_LAUNCH_CHECK("rle_counts_kernel");
  return MRX_OK;
}
