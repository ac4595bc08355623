// contours.cu -- mask outlines as closed polygons: what visualize.display_instances traces for
// every instance (skimage.measure.find_contours(padded_mask, 0.5), serve.py:160-169), computed
// from the bit-packed masks (the layout of mrx_mask_expand_packed / mrx_pack_masks).
//
// Marching squares on the mask padded by one zero pixel on every side: cell (r, c) of the padded
// grid is the 2x2 square of padded pixels (r..r+1, c..c+1), i.e. mask pixels (r-1..r, c-1..c).
// Its case code ul + 2 ur + 4 ll + 8 lr selects 0, 1 or 2 directed segments between the
// midpoints of the cell's edges (table in include/mrx.h); cells are emitted in row-major order,
// which numbers every segment of an instance.  For 0/1 data each edge midpoint has exactly one
// segment in and one out, so the segments form cycles; skimage's assembly then yields, per cycle,
// the polygon that starts at the `to` point of the cycle's LAST-emitted segment, follows segment
// direction and repeats its start point, and orders the polygons by the emission index of each
// cycle's FIRST-emitted segment.  That rule is what the kernels implement.
//
//   contour_rows_kernel<false>  per (instance, cell row): number of segments of the row
//   contour_scan_kernel         per instance: exclusive scan over its rows, instance total
//   (exclusive scan of the instance totals: the RLE offsets kernel)
//   contour_rows_kernel<true>   per (instance, cell row): every segment's successor (the segment
//                               leaving the edge midpoint it enters, found in the neighbouring
//                               cell across that edge) and its `to` point, into the scratch
//   contour_walk_kernel         one warp per instance: cycles in emission order, two walks each
//                               (mark + find the largest index, then write the vertices), on a
//                               shared-memory copy of the successors when they fit
//
// Only the cells of the box plus one ring are visited: a mask is read as zero outside its box.
#include "common.cuh"

namespace mrx {

namespace contours {

constexpr int kRowWarps = 8;
constexpr int kScanThreads = 256;
constexpr int kSmemSegments = 16384;    // walk kernel: successors cached in 64 KB of shared memory

struct Params {
  const unsigned char *packed;   // image b at packed + packed_off[b]: uint8 [N_b, H_b, ceil(W_b/8)]
  const long long *packed_off;   // [B]
  const int4 *boxes;             // [B,R] (y1, x1, y2, x2)
  const int *counts;             // [B]
  const int *geom;               // [B,8]
  int *row_seg;                  // [B,R,max_h+1]: segments per cell row -> exclusive row offsets
  const long long *seg_off;      // [B*R+1]
  int *succ;                     // [T] successor of every segment (instance-local index)
  unsigned int *to;              // [T] its `to` point, (2*row) << 16 | (2*col) in the padded grid
  int B, R, max_h, max_w;
};

struct Inst {
  const unsigned char *plane;    // the instance's [H, ceil(W/8)] bit plane
  int wb;                        // bytes per row
  int y1, x1, y2, x2;            // box; empty (y2 <= y1) when the instance has no sane box
};

__device__ __forceinline__ Inst load_inst(const Params &p, int b, int k) {
  Inst in;
  const int H = p.geom[b * MRX_GEOM_INTS + 0], W = p.geom[b * MRX_GEOM_INTS + 1];
  in.wb = (W + 7) >> 3;
  in.plane = p.packed + p.packed_off[b] + static_cast<size_t>(k) * H * in.wb;
  const int4 bx = p.boxes[static_cast<size_t>(b) * p.R + k];
  const bool sane = k < p.counts[b] && bx.x >= 0 && bx.y >= 0 && bx.z <= H && bx.w <= W &&
                    bx.z > bx.x && bx.w > bx.y;
  in.y1 = sane ? bx.x : 0;
  in.x1 = sane ? bx.y : 0;
  in.y2 = sane ? bx.z : 0;
  in.x2 = sane ? bx.w : 0;
  return in;
}

__device__ __forceinline__ unsigned range_mask(int lo, int hi) {   // bits [lo, hi), 0 <= lo, hi <= 32
  const unsigned below_hi = hi >= 32 ? 0xffffffffu : (1u << max(hi, 0)) - 1u;
  const unsigned below_lo = lo >= 32 ? 0xffffffffu : (1u << max(lo, 0)) - 1u;
  return below_hi & ~below_lo;
}

// Mask pixels (y, 32*wi .. 32*wi+31) as bits 0..31, zero outside the box (which also drops the
// bits past W in a row's last byte).
__device__ __forceinline__ unsigned pixel_word(const Inst &in, int y, int wi) {
  if (y < in.y1 || y >= in.y2 || wi < 0) return 0u;
  const int x0 = wi << 5;
  const unsigned m = range_mask(in.x1 - x0, in.x2 - x0);
  if (m == 0u) return 0u;
  const unsigned char *row = in.plane + static_cast<size_t>(y) * in.wb;
  const int byte0 = wi << 2;
  unsigned w = 0;
#pragma unroll
  for (int t = 0; t < 4; ++t)
    w |= static_cast<unsigned>(byte0 + t < in.wb ? row[byte0 + t] : 0) << (24 - 8 * t);
  return __brev(w) & m;    // most significant bit first within a byte -> bit k = pixel x0 + k
}

// Edge codes and the segment table (from, to) per case; fully_connected='low' pairs the saddles.
enum { kTop = 0, kBottom = 1, kLeft = 2, kRight = 3 };
__device__ __forceinline__ int seg_count(int cs) {
  return (cs == 0 || cs == 15) ? 0 : ((cs == 6 || cs == 9) ? 2 : 1);
}
// packed as from | to << 2 (first segment) | from2 << 4 | to2 << 6 (second, saddles only)
__constant__ unsigned char kSegTable[16] = {
    0,
    kTop | kLeft << 2,                                        // 1
    kRight | kTop << 2,                                       // 2
    kRight | kLeft << 2,                                      // 3
    kLeft | kBottom << 2,                                     // 4
    kTop | kBottom << 2,                                      // 5
    kRight | kTop << 2 | kLeft << 4 | kBottom << 6,           // 6
    kRight | kBottom << 2,                                    // 7
    kBottom | kRight << 2,                                    // 8
    kTop | kLeft << 2 | kBottom << 4 | kRight << 6,           // 9
    kBottom | kTop << 2,                                      // 10
    kBottom | kLeft << 2,                                     // 11
    kLeft | kRight << 2,                                      // 12
    kTop | kRight << 2,                                       // 13
    kLeft | kTop << 2,                                        // 14
    0};

// Which segment of a cell with case `cs` leaves edge `from` (only saddles have two).
__device__ __forceinline__ int seg_leaving(int cs, int from) {
  if (cs == 6) return from == kLeft ? 1 : 0;
  if (cs == 9) return from == kBottom ? 1 : 0;
  return 0;
}

// Bit x - 32*wi + d of a row given its words wi-1 (prev), wi (cur), wi+1 (next); lane-relative.
__device__ __forceinline__ int bit_at(unsigned prev, unsigned cur, unsigned next, int k) {
  if (k >= 32) return (next >> (k - 32)) & 1;
  if (k < 0) return (prev >> (k + 32)) & 1;
  return (cur >> k) & 1;
}

__device__ __forceinline__ int case_of(int ul, int ur, int ll, int lr) {
  return ul | (ur << 1) | (ll << 2) | (lr << 3);
}

// One warp per padded cell row r of one instance.  Lane k of a step handles cell c = 32*wi + k,
// which reads mask pixels (r-1..r, c-1..c); the write pass also needs the cells around it, so the
// words of mask rows r-2 .. r+1 are kept for wi-1, wi, wi+1.
template <bool kWrite>
__global__ void __launch_bounds__(kRowWarps * 32)
contour_rows_kernel(const Params p) {
  const int lane = threadIdx.x & 31;
  const int k = blockIdx.y, b = blockIdx.z;
  const Inst in = load_inst(p, b, k);
  const int r = in.y1 + blockIdx.x * kRowWarps + (threadIdx.x >> 5);
  if (in.y2 <= in.y1 || r > in.y2) return;
  const size_t inst = static_cast<size_t>(b) * p.R + k;
  int *rows = p.row_seg + inst * (p.max_h + 1);
  const int wlo = in.x1 >> 5, whi = in.x2 >> 5;   // cells x1 .. x2
  int row_base[3] = {0, 0, 0};                    // first segment of cell rows r-1, r, r+1
  int S = 0;
  int *succ = nullptr;
  unsigned *to = nullptr;
  if (kWrite) {
    const long long sb = p.seg_off[inst];
    S = static_cast<int>(p.seg_off[inst + 1] - sb);
    succ = p.succ + sb;
    to = p.to + sb;
    for (int d = 0; d < 3; ++d) {
      const int rr = r - 1 + d;
      row_base[d] = (rr >= in.y1 && rr <= in.y2) ? rows[rr - in.y1] : 0;
    }
  }
  // words of mask rows r-2+i (i = 0..3) at wi-1, wi, wi+1
  unsigned wp[4], wc[4], wn[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    wp[i] = pixel_word(in, r - 2 + i, wlo - 1);
    wc[i] = pixel_word(in, r - 2 + i, wlo);
    wn[i] = pixel_word(in, r - 2 + i, wlo + 1);
  }
  int carry[3] = {0, 0, 0};
  for (int wi = wlo; wi <= whi; ++wi) {
    // 4x4 patch of mask bits: rows r-2..r+1, columns c-2..c+1
    int pt[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) pt[i][j] = bit_at(wp[i], wc[i], wn[i], lane - 2 + j);
    const int cs = case_of(pt[1][1], pt[1][2], pt[2][1], pt[2][2]);   // cell (r, c)
    const int n = seg_count(cs);
    if (!kWrite) {
      carry[1] += __reduce_add_sync(0xffffffffu, n);
    } else {
      const int cs_up = case_of(pt[0][1], pt[0][2], pt[1][1], pt[1][2]);   // (r-1, c)
      const int cs_dn = case_of(pt[2][1], pt[2][2], pt[3][1], pt[3][2]);   // (r+1, c)
      const int cs_lf = case_of(pt[1][0], pt[1][1], pt[2][0], pt[2][1]);   // (r, c-1)
      const int cs_rt = case_of(pt[1][2], pt[1][3], pt[2][2], pt[2][3]);   // (r, c+1)
      // inclusive warp scan of the three rows' counts, packed 10 bits each (<= 64 per step)
      int v = seg_count(cs_up) | (n << 10) | (seg_count(cs_dn) << 20);
      const int own = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += u;
      }
      const int excl = v - own;
      const int tot = __shfl_sync(0xffffffffu, v, 31);
      const int start_up = row_base[0] + carry[0] + (excl & 1023);
      const int start = row_base[1] + carry[1] + ((excl >> 10) & 1023);
      const int start_dn = row_base[2] + carry[2] + ((excl >> 20) & 1023);
      const int c = (wi << 5) + lane;
      const unsigned tbl = kSegTable[cs];
      for (int s = 0; s < n; ++s) {
        const int dst = (tbl >> (4 * s + 2)) & 3;
        int nxt;
        unsigned pt2;   // (2*row) << 16 | (2*col), padded grid
        if (dst == kTop) {
          nxt = start_up + seg_leaving(cs_up, kBottom);
          pt2 = (static_cast<unsigned>(2 * r) << 16) | static_cast<unsigned>(2 * c + 1);
        } else if (dst == kBottom) {
          nxt = start_dn + seg_leaving(cs_dn, kTop);
          pt2 = (static_cast<unsigned>(2 * r + 2) << 16) | static_cast<unsigned>(2 * c + 1);
        } else if (dst == kLeft) {
          nxt = start - seg_count(cs_lf) + seg_leaving(cs_lf, kRight);
          pt2 = (static_cast<unsigned>(2 * r + 1) << 16) | static_cast<unsigned>(2 * c);
        } else {
          nxt = start + n + seg_leaving(cs_rt, kLeft);
          pt2 = (static_cast<unsigned>(2 * r + 1) << 16) | static_cast<unsigned>(2 * c + 2);
        }
        const int j = start + s;
        if (j < S) {
          succ[j] = nxt;
          to[j] = pt2;
        }
      }
      carry[0] += tot & 1023;
      carry[1] += (tot >> 10) & 1023;
      carry[2] += (tot >> 20) & 1023;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      wp[i] = wc[i];
      wc[i] = wn[i];
      wn[i] = pixel_word(in, r - 2 + i, wi + 2);
    }
  }
  if (!kWrite && lane == 0) rows[r - in.y1] = carry[1];
}

// One CTA per instance: exclusive scan of its cell rows' segment counts (in place), total out.
__global__ void __launch_bounds__(kScanThreads)
contour_scan_kernel(const Params p, long long *seg_total) {
  const int k = blockIdx.x, b = blockIdx.y;
  const size_t inst = static_cast<size_t>(b) * p.R + k;
  __shared__ int s_warp[kScanThreads / 32];
  __shared__ int s_carry;
  const Inst in = load_inst(p, b, k);
  const int n = in.y2 > in.y1 ? in.y2 - in.y1 + 1 : 0;
  int *rows = p.row_seg + inst * (p.max_h + 1);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (int base = 0; base < n; base += kScanThreads) {
    const int i = base + threadIdx.x;
    const int v = i < n ? rows[i] : 0;
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
    if (i < n) rows[i] = before + incl - v;
    __syncthreads();
    if (threadIdx.x == kScanThreads - 1) s_carry = before + incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) seg_total[inst] = s_carry;
}

struct Out {
  float2 *vertices;      // instance i's vertices from seg_off[i] + seg_off[i]/4
  int *contour_len;      // instance i's contour lengths from seg_off[i]/4
  int *inst_contours;    // [B*R]
};

// One warp per instance.  Cycles are found in emission order; a visited segment's successor is
// stored complemented (negative).  Lane 0 walks; the warp scans for unvisited segments.
__global__ void __launch_bounds__(32)
contour_walk_kernel(const Params p, const Out o) {
  extern __shared__ int s_succ[];
  const int lane = threadIdx.x;
  const size_t inst = static_cast<size_t>(blockIdx.y) * p.R + blockIdx.x;
  const long long sb = p.seg_off[inst];
  const int S = static_cast<int>(p.seg_off[inst + 1] - sb);
  int *succ = p.succ + sb;
  const unsigned *to = p.to + sb;
  if (S <= kSmemSegments) {
    for (int j = lane; j < S; j += 32) s_succ[j] = succ[j];
    __syncwarp();
    succ = s_succ;
  }
  float2 *vout = o.vertices + sb + sb / 4;
  int *lens = o.contour_len + sb / 4;
  auto vertex = [](unsigned t) {
    return make_float2(0.5f * static_cast<float>(static_cast<int>(t & 0xffffu) - 2),
                       0.5f * static_cast<float>(static_cast<int>(t >> 16) - 2));
  };
  int nc = 0;
  long long nv = 0;
  for (int base = 0; base < S; base += 32) {
    const int jj = base + lane;
    unsigned m = __ballot_sync(0xffffffffu, jj < S && succ[jj] >= 0);
    if (lane == 0) {
      while (m) {
        const int i = base + __ffs(m) - 1;
        m &= m - 1;
        if (succ[i] < 0) continue;
        // walk 1: mark the cycle, its length and its last-emitted segment
        int j = i, last = i, L = 0;
        do {
          const int nx = succ[j];
          if (static_cast<unsigned>(nx) >= static_cast<unsigned>(S)) break;   // (inconsistent input)
          succ[j] = ~nx;
          last = max(last, j);
          ++L;
          j = nx;
        } while (j != i);
        // walk 2: vertices from the last-emitted segment's `to` point, closed
        float2 *vo = vout + nv;
        vo[0] = vertex(to[last]);
        int q = ~succ[last];
        for (int t = 1; t <= L; ++t) {
          vo[t] = vertex(to[q]);
          q = ~succ[q];
        }
        lens[nc++] = L + 1;
        nv += L + 1;
      }
    }
    __syncwarp();
  }
  if (lane == 0) o.inst_contours[inst] = nc;
}

}  // namespace contours

}  // namespace mrx

using namespace mrx;

static int fill_contour_params(contours::Params &prm, const char *what,
                               const unsigned char *d_packed, const long long *d_packed_off,
                               const int *d_boxes, const int *d_counts, const int *d_geom,
                               int *d_row_seg, const long long *d_seg_off, int B, int R, int max_h,
                               int max_w) {
  MRX_CHECK_ARG(d_packed && d_packed_off && d_boxes && d_counts && d_geom && d_row_seg && d_seg_off,
                "%s: null pointer", what);
  MRX_CHECK_ARG(B >= 1 && B <= 65535 && R >= 1 && R <= 65535 && max_h >= 1 && max_w >= 1,
                "%s: bad sizes B=%d R=%d max_h=%d max_w=%d", what, B, R, max_h, max_w);
  MRX_CHECK_SUPPORTED(max_h <= MRX_CONTOUR_MAX_DIM && max_w <= MRX_CONTOUR_MAX_DIM,
                      "%s: image %dx%d too large for contours (sides <= %d)", what, max_h, max_w,
                      MRX_CONTOUR_MAX_DIM);
  prm.packed = d_packed;
  prm.packed_off = d_packed_off;
  prm.boxes = reinterpret_cast<const int4 *>(d_boxes);
  prm.counts = d_counts;
  prm.geom = d_geom;
  prm.row_seg = d_row_seg;
  prm.seg_off = d_seg_off;
  prm.succ = nullptr;
  prm.to = nullptr;
  prm.B = B;
  prm.R = R;
  prm.max_h = max_h;
  prm.max_w = max_w;
  return MRX_OK;
}

extern "C" int mrx_contours_count(const unsigned char *d_packed, const long long *d_packed_off,
                                  const int *d_boxes, const int *d_counts, const int *d_geom,
                                  int *d_row_seg, long long *d_seg_off, int B, int R, int max_h,
                                  int max_w, void *stream) {
  contours::Params prm;
  if (int rc = fill_contour_params(prm, "mrx_contours_count", d_packed, d_packed_off, d_boxes,
                                   d_counts, d_geom, d_row_seg, d_seg_off, B, R, max_h, max_w))
    return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  dim3 grid((max_h + 1 + contours::kRowWarps - 1) / contours::kRowWarps, R, B);
  contours::contour_rows_kernel<false><<<grid, contours::kRowWarps * 32, 0, st>>>(prm);
  MRX_LAUNCH_CHECK("contour_rows_kernel<count>");
  contours::contour_scan_kernel<<<dim3(R, B), contours::kScanThreads, 0, st>>>(prm, d_seg_off);
  MRX_LAUNCH_CHECK("contour_scan_kernel");
  return exclusive_scan_i64(d_seg_off, B * R, st);
}

extern "C" int mrx_contours_write(const unsigned char *d_packed, const long long *d_packed_off,
                                  const int *d_boxes, const int *d_counts, const int *d_geom,
                                  int *d_row_seg, const long long *d_seg_off, int *d_scratch,
                                  float *d_vertices, int *d_contour_len, int *d_inst_contours,
                                  long long total_segments, int B, int R, int max_h, int max_w,
                                  void *stream) {
  contours::Params prm;
  if (int rc = fill_contour_params(prm, "mrx_contours_write", d_packed, d_packed_off, d_boxes,
                                   d_counts, d_geom, d_row_seg, d_seg_off, B, R, max_h, max_w))
    return rc;
  MRX_CHECK_ARG(d_inst_contours && total_segments >= 0, "mrx_contours_write: null pointer or "
                "negative total");
  MRX_CHECK_ARG(total_segments == 0 || (d_scratch && d_vertices && d_contour_len),
                "mrx_contours_write: null pointer");
  prm.succ = d_scratch;
  prm.to = reinterpret_cast<unsigned int *>(d_scratch) + total_segments;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DevInfo dev;
  if (int rc = current_device_info(&dev)) return rc;
  const int smem = contours::kSmemSegments * static_cast<int>(sizeof(int));
  static SmemCache cache;
  if (int rc = ensure_dynamic_smem(reinterpret_cast<const void *>(contours::contour_walk_kernel),
                                   &cache, dev.device, smem))
    return rc;
  dim3 grid((max_h + 1 + contours::kRowWarps - 1) / contours::kRowWarps, R, B);
  contours::contour_rows_kernel<true><<<grid, contours::kRowWarps * 32, 0, st>>>(prm);
  MRX_LAUNCH_CHECK("contour_rows_kernel<write>");
  contours::Out o;
  o.vertices = reinterpret_cast<float2 *>(d_vertices);
  o.contour_len = d_contour_len;
  o.inst_contours = d_inst_contours;
  contours::contour_walk_kernel<<<dim3(R, B), 32, smem, st>>>(prm, o);
  MRX_LAUNCH_CHECK("contour_walk_kernel");
  return MRX_OK;
}
