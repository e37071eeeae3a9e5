// Point-to-plane ICP / gradICP odometry for sm_100a, batched over B elements, no host synchronisation.
//
//   k_icp_gather_src     live frame -> source cloud: lattice pixels (every ds-th row/column) with valid depth,
//                        world-frame vertex at the PREVIOUS pose, stable row-major compaction
//                        (downsample_rgbdimages, gradslam/odometry/icputils.py:623-669)
//   k_icp_gather_tgt     map -> target cloud: map points inside the previous frame's frustum whose pixel lies on
//                        the lattice, stable compaction in point order (find_active_map_points +
//                        downsample_pointclouds, slam/fusionutils.py:198-287, odometry/icputils.py:548-620)
//   k_icp_knn_linearize  exact 1-NN of every source point in the target cloud (brute force over shared-memory
//                        tiles, lowest index wins ties; restates chamferdist knn_points, icputils.py:200) fused
//                        with the point-to-plane row build and the reduction of J^T J (21), J^T r (6), r^T r (1)
//                        (gauss_newton_solve + the normal equations, icputils.py:85-90, 203-232).  A pending
//                        4x4 transform is applied to the source on load (transform_pointcloud, geometryutils.py
//                        :737-794) and optionally written back.
//   k_icp_solve          one warp per element: fixed-order reduction of the block partials, damped 6x6 solve
//                        (solve_linear_system, icputils.py:22-90), se3_exp (geometry/se3utils.py:77-115)
//   k_icp_update         one warp per element: look-ahead error, LM accept/reject (icputils.py:356-365) or gradLM
//                        smooth gates (icputils.py:527-543), pose accumulation
#include "gsx_common.cuh"
#include "../../include/gsx.h"

namespace gsx {

constexpr int kIcpBlock = 256;
constexpr int kTgtTile = 1024;  // target points staged in shared memory per step (16 KB as float4)
constexpr int kNumSums = 28;    // 21 upper-triangular J^T J + 6 J^T r + r^T r

// ---------------------------------------------------------------------------------------------------------
// gather: source cloud
// ---------------------------------------------------------------------------------------------------------
struct GatherSrcArgs {
  const float *depth;
  int64_t depth_bstride;
  const float *K;
  int64_t K_bstride;
  const float *poses;  // pose to place the frame at (the previous frame's pose)
  int64_t pose_bstride;
  int B, H, W, ds;
  float *src;        // (B, ns_cap, 3)
  int32_t *src_count;  // (B)
  int ns_cap;
};

__global__ void __launch_bounds__(1024) k_icp_gather_src(GatherSrcArgs a) {
  __shared__ int s_warp[32];
  __shared__ int s_base;
  __shared__ KInv s_k;
  __shared__ Rigid s_pose;
  const int b = blockIdx.x;
  if (threadIdx.x == 0) {
    s_k = load_kinv(a.K + b * a.K_bstride);
    s_base = 0;
  }
  if (threadIdx.x == 32) s_pose = load_rigid(a.poses + b * a.pose_bstride);
  __syncthreads();
  const int Hs = (a.H + a.ds - 1) / a.ds, Ws = (a.W + a.ds - 1) / a.ds;
  const int total = Hs * Ws;
  const float *dimg = a.depth + b * a.depth_bstride;
  float *out = a.src + (int64_t)b * a.ns_cap * 3;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int base = 0; base < total; base += 1024) {
    const int i = base + threadIdx.x;
    bool flag = false;
    float3 gv = make_float3(0.f, 0.f, 0.f);
    if (i < total) {
      const int hs = i / Ws, ws = i - hs * Ws;
      const FrameSample f = frame_sample<false>(dimg, s_k, &s_pose, hs * a.ds, ws * a.ds, a.H, a.W);
      flag = f.d > 0.0f;
      gv = f.gv;
    }
    const unsigned int ballot = __ballot_sync(0xffffffffu, flag);
    if (lane == 0) s_warp[warp] = __popc(ballot);
    __syncthreads();
    int excl = s_base, tot = 0;
    for (int w = 0; w < 32; ++w) {
      const int c = s_warp[w];
      if (w < warp) excl += c;
      tot += c;
    }
    excl += __popc(ballot & ((1u << lane) - 1u));
    if (flag && excl < a.ns_cap) {
      out[(int64_t)excl * 3 + 0] = gv.x;
      out[(int64_t)excl * 3 + 1] = gv.y;
      out[(int64_t)excl * 3 + 2] = gv.z;
    }
    __syncthreads();
    if (threadIdx.x == 0) s_base += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) a.src_count[b] = min(s_base, a.ns_cap);
}

// ---------------------------------------------------------------------------------------------------------
// gather: target cloud (stable compaction of lattice-active map points; decoupled look-back over tiles)
// ---------------------------------------------------------------------------------------------------------
constexpr int kGeoW = 8;  // floats per packed geometry row (px,py,pz,nx,ny,nz,ccount,0), see gsx_fusion.cu
struct GatherTgtArgs {
  const float *geo;  // (B,cap,8)
  const int32_t *counts;
  int64_t cap;
  const float *poses;
  int64_t pose_bstride;
  const float *K;
  int64_t K_bstride;
  int B, H, W, ds;
  float u_hi, v_hi;
  float *tgt_p, *tgt_n;  // (B, nt_cap, 3)
  int32_t *tgt_count;    // (B)
  int nt_cap;
  unsigned long long *tile_state;  // (B, tiles)
  unsigned int *ticket;            // (B)
  int tiles;                       // tiles per element (= ceil(max_count / 1024))
  unsigned int epoch;
  int32_t *overflow;  // set to 1 if the target cloud did not fit nt_cap (may be null)
};

constexpr unsigned long long kAgg = 1ull, kPrefix = 2ull;
__device__ __forceinline__ unsigned long long icp_pack(unsigned int epoch, unsigned long long flag, unsigned int v) {
  return ((unsigned long long)epoch << 34) | (flag << 32) | v;
}
__device__ __forceinline__ unsigned long long icp_ld_acquire(const unsigned long long *p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void icp_st_release(unsigned long long *p, unsigned long long v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__global__ void __launch_bounds__(kIcpBlock) k_icp_gather_tgt(GatherTgtArgs a) {
  __shared__ Rigid s_tinv;
  __shared__ float s_k[12];
  __shared__ int s_tile, s_excl;
  __shared__ int s_warp[4][kIcpBlock / 32];
  const int b = blockIdx.x % a.B;  // elements interleaved in the grid (short look-back chains)
  if (threadIdx.x == 0) {
    // dynamic tile id.  The block that draws the last ticket re-arms the counter for the next launch (nobody
    // else will touch it any more in this one), so the number of tiles may differ from launch to launch.
    const unsigned int t = atomicAdd(a.ticket + b, 1u);
    if (t == (unsigned int)a.tiles - 1u) a.ticket[b] = 0u;
    s_tile = (int)t;
    s_tinv = rigid_inverse(load_rigid(a.poses + b * a.pose_bstride));
  }
  if (threadIdx.x >= 32 && threadIdx.x < 44) s_k[threadIdx.x - 32] = __ldg(a.K + b * a.K_bstride + (threadIdx.x - 32));
  __syncthreads();
  const int tile = s_tile;
  const int count = a.counts[b];
  const float *geo = a.geo + (int64_t)b * a.cap * kGeoW;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int n[4], wexcl[4];
  bool keep[4];
  float px[4], py[4], pz[4], nx[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    n[j] = tile * 1024 + j * kIcpBlock + threadIdx.x;
    keep[j] = n[j] < count;
    const int nn = keep[j] ? n[j] : 0;
    const float4 g = __ldg(reinterpret_cast<const float4 *>(geo + (int64_t)nn * kGeoW));
    px[j] = g.x;
    py[j] = g.y;
    pz[j] = g.z;
    nx[j] = g.w;
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    // identical to the projection of k_project_select (fusionutils.py:249-274)
    const float3 q = rigid_apply(s_tinv, px[j], py[j], pz[j]);
    const float hx = ((s_k[0] * q.x + s_k[1] * q.y) + s_k[2] * q.z) + s_k[3];
    const float hy = ((s_k[4] * q.x + s_k[5] * q.y) + s_k[6] * q.z) + s_k[7];
    const float hz = ((s_k[8] * q.x + s_k[9] * q.y) + s_k[10] * q.z) + s_k[11];
    const float den = (hz != 0.0f) ? hz : 1.0f;
    const float u = hx / den, v = hy / den;
    keep[j] = keep[j] && (u > -1e-3f) && (u < a.u_hi) && (v > -1e-3f) && (v < a.v_hi) && (q.z > 0.0f);
    int w = (int)rintf(u), h = (int)rintf(v);
    w = min(max(w, 0), a.W - 1);
    h = min(max(h, 0), a.H - 1);
    keep[j] = keep[j] && (h % a.ds == 0) && (w % a.ds == 0);  // icputils.py:596-597
    const unsigned int ballot = __ballot_sync(0xffffffffu, keep[j]);
    wexcl[j] = __popc(ballot & ((1u << lane) - 1u));
    if (lane == 0) s_warp[j][warp] = __popc(ballot);
  }
  __syncthreads();
  int total = 0, bexcl[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    bexcl[j] = total;
#pragma unroll
    for (int i = 0; i < kIcpBlock / 32; ++i) {
      const int c = s_warp[j][i];
      if (i < warp) bexcl[j] += c;
      total += c;
    }
  }
  unsigned long long *state = a.tile_state + (int64_t)b * a.tiles;
  if (threadIdx.x == 0 && tile + 1 < a.tiles) icp_st_release(state + tile, icp_pack(a.epoch, kAgg, (unsigned)total));
  if (warp == 0) {
    unsigned int excl = 0;
    for (int base = tile - 1; base >= 0; base -= 32) {
      const int j = base - lane;
      unsigned long long s = 0ull;
      if (j >= 0) {
        do {
          s = icp_ld_acquire(state + j);
        } while ((unsigned int)(s >> 34) != a.epoch);
      }
      const bool is_prefix = (j >= 0) && (((s >> 32) & 3ull) == kPrefix);
      const unsigned int pm = __ballot_sync(0xffffffffu, is_prefix);
      const int first = pm ? (__ffs(pm) - 1) : 32;
      const unsigned int v = (j >= 0 && lane <= first) ? (unsigned int)s : 0u;
      excl += __reduce_add_sync(0xffffffffu, v);
      if (pm) break;
    }
    if (lane == 0) {
      if (tile + 1 < a.tiles) icp_st_release(state + tile, icp_pack(a.epoch, kPrefix, excl + (unsigned)total));
      s_excl = (int)excl;
    }
  }
  __syncthreads();
  float *op = a.tgt_p + (int64_t)b * a.nt_cap * 3;
  float *on = a.tgt_n + (int64_t)b * a.nt_cap * 3;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (keep[j]) {
      const int pos = s_excl + bexcl[j] + wexcl[j];
      if (pos < a.nt_cap) {
        op[(int64_t)pos * 3 + 0] = px[j];
        op[(int64_t)pos * 3 + 1] = py[j];
        op[(int64_t)pos * 3 + 2] = pz[j];
        const float2 g = __ldg(reinterpret_cast<const float2 *>(geo + (int64_t)n[j] * kGeoW + 4));
        on[(int64_t)pos * 3 + 0] = nx[j];
        on[(int64_t)pos * 3 + 1] = g.x;
        on[(int64_t)pos * 3 + 2] = g.y;
      } else if (a.overflow) {
        *a.overflow = 1;
      }
    }
  }
  if (tile == a.tiles - 1 && threadIdx.x == 0) a.tgt_count[b] = min(s_excl + total, a.nt_cap);
}

// ---------------------------------------------------------------------------------------------------------
// uniform grid over the target cloud (built once per ICP call: the target does not move during the loop)
// ---------------------------------------------------------------------------------------------------------
constexpr int kGridMaxDim = 64;                                                          // cells per axis
constexpr int kGridMaxCells = (kGridMaxDim + 1) * (kGridMaxDim + 1) * (kGridMaxDim + 1);  // 274 625
constexpr int kGridMaxRing = 3;  // rings searched before a query falls back to the full scan

struct GridParams {  // per element
  float ox, oy, oz;  // origin (bbox min)
  float inv_c, c;    // cells are cubes of edge c
  int nx, ny, nz;
};

struct TargetGrid {
  GridParams *params;   // (B)
  int *cell_start;      // (B, kGridMaxCells + 1) exclusive prefix of the per-cell counts
  int *cursor;          // (B, kGridMaxCells)     counts, then scatter cursors
  float4 *sorted;       // (B, nt_stride)         (x, y, z, original index as int bits), grouped by cell
};

__device__ __forceinline__ int cell_coord(float p, float o, float inv_c, int n) {
  const int i = (int)floorf((p - o) * inv_c);
  return min(max(i, 0), n - 1);
}

__global__ void __launch_bounds__(256) k_grid_bbox(const float *tgt_p, const int32_t *tgt_count, int nt_stride,
                                                   TargetGrid g) {
  __shared__ float s_lo[3][8], s_hi[3][8];
  const int b = blockIdx.x;
  const int nt = tgt_count[b];
  const float *p = tgt_p + (int64_t)b * nt_stride * 3;
  float lo[3] = {3.0e38f, 3.0e38f, 3.0e38f}, hi[3] = {-3.0e38f, -3.0e38f, -3.0e38f};
  for (int i = threadIdx.x; i < nt; i += 256)
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      const float v = __ldg(p + (int64_t)i * 3 + a);
      lo[a] = fminf(lo[a], v);
      hi[a] = fmaxf(hi[a], v);
    }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
      hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
    }
    if ((threadIdx.x & 31) == 0) {
      s_lo[a][threadIdx.x >> 5] = lo[a];
      s_hi[a][threadIdx.x >> 5] = hi[a];
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float l[3], h[3];
    for (int a = 0; a < 3; ++a) {
      l[a] = s_lo[a][0];
      h[a] = s_hi[a][0];
      for (int w = 1; w < 8; ++w) {
        l[a] = fminf(l[a], s_lo[a][w]);
        h[a] = fmaxf(h[a], s_hi[a][w]);
      }
    }
    GridParams gp;
    if (nt <= 0) {
      gp = GridParams{0.f, 0.f, 0.f, 1.f, 1.f, 1, 1, 1};
    } else {
      const float ext = fmaxf(fmaxf(h[0] - l[0], h[1] - l[1]), fmaxf(h[2] - l[2], 1e-6f));
      const float c = ext / (float)kGridMaxDim;
      gp.ox = l[0]; gp.oy = l[1]; gp.oz = l[2];
      gp.c = c;
      gp.inv_c = 1.0f / c;
      gp.nx = min(kGridMaxDim + 1, (int)floorf((h[0] - l[0]) * gp.inv_c) + 1);
      gp.ny = min(kGridMaxDim + 1, (int)floorf((h[1] - l[1]) * gp.inv_c) + 1);
      gp.nz = min(kGridMaxDim + 1, (int)floorf((h[2] - l[2]) * gp.inv_c) + 1);
    }
    g.params[b] = gp;
  }
}

__global__ void __launch_bounds__(256) k_grid_clear(TargetGrid g, int B) {
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i < (int64_t)B * kGridMaxCells) g.cursor[i] = 0;
}

__global__ void __launch_bounds__(256) k_grid_count(const float *tgt_p, const int32_t *tgt_count, int nt_stride,
                                                    TargetGrid g) {
  const int b = blockIdx.y;
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= tgt_count[b]) return;
  const GridParams gp = g.params[b];
  const float *p = tgt_p + ((int64_t)b * nt_stride + i) * 3;
  const int cx = cell_coord(__ldg(p), gp.ox, gp.inv_c, gp.nx), cy = cell_coord(__ldg(p + 1), gp.oy, gp.inv_c, gp.ny),
            cz = cell_coord(__ldg(p + 2), gp.oz, gp.inv_c, gp.nz);
  atomicAdd(g.cursor + (int64_t)b * kGridMaxCells + (cz * gp.ny + cy) * gp.nx + cx, 1);
}

__global__ void __launch_bounds__(1024) k_grid_scan(TargetGrid g) {
  __shared__ int s_warp[32];
  __shared__ int s_base;
  const int b = blockIdx.x;
  const GridParams gp = g.params[b];
  const int ncell = gp.nx * gp.ny * gp.nz;
  int *cnt = g.cursor + (int64_t)b * kGridMaxCells;
  int *start = g.cell_start + (int64_t)b * (kGridMaxCells + 1);
  if (threadIdx.x == 0) s_base = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int base = 0; base < ncell; base += 1024) {
    const int i = base + threadIdx.x;
    const int v = (i < ncell) ? cnt[i] : 0;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    int off = s_base;
    for (int w = 0; w < warp; ++w) off += s_warp[w];
    if (i < ncell) {
      start[i] = off + x - v;
      cnt[i] = off + x - v;  // becomes the scatter cursor
    }
    __syncthreads();
    if (threadIdx.x == 1023) s_base = off + x;
    __syncthreads();
  }
  if (threadIdx.x == 0) start[ncell] = s_base;
}

__global__ void __launch_bounds__(256) k_grid_scatter(const float *tgt_p, const int32_t *tgt_count, int nt_stride,
                                                      TargetGrid g) {
  const int b = blockIdx.y;
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= tgt_count[b]) return;
  const GridParams gp = g.params[b];
  const float *p = tgt_p + ((int64_t)b * nt_stride + i) * 3;
  const float x = __ldg(p), y = __ldg(p + 1), z = __ldg(p + 2);
  const int cx = cell_coord(x, gp.ox, gp.inv_c, gp.nx), cy = cell_coord(y, gp.oy, gp.inv_c, gp.ny),
            cz = cell_coord(z, gp.oz, gp.inv_c, gp.nz);
  const int pos = atomicAdd(g.cursor + (int64_t)b * kGridMaxCells + (cz * gp.ny + cy) * gp.nx + cx, 1);
  g.sorted[(int64_t)b * nt_stride + pos] = make_float4(x, y, z, __int_as_float(i));
}

// Exact nearest neighbour of (sx,sy,sz) through the grid.  Candidates are compared on (squared distance, original
// index) so the result is identical to an ascending brute-force scan with a strict '<' (lowest index on ties),
// whatever the order of the points inside a cell.  Rings of cells are visited outwards; the search stops as soon
// as the best distance is provably not larger than the distance to anything not yet visited; queries that do not
// terminate within kGridMaxRing rings fall back to scanning every target point.
__device__ __forceinline__ void nn_update(float d, int idx, float &best, int &bi) {
  if (bi < 0 || d < best || (d == best && idx < bi)) {
    best = d;
    bi = idx;
  }
}

__device__ void search_grid(const TargetGrid &g, int b, int nt, int nt_stride, float sx, float sy, float sz, float &best,
                            int &bi) {
  const GridParams gp = g.params[b];
  const int *start = g.cell_start + (int64_t)b * (kGridMaxCells + 1);
  const float4 *pts = g.sorted + (int64_t)b * nt_stride;
  const float gx = (sx - gp.ox) * gp.inv_c, gy = (sy - gp.oy) * gp.inv_c, gz = (sz - gp.oz) * gp.inv_c;
  const int cx = min(max((int)floorf(gx), 0), gp.nx - 1), cy = min(max((int)floorf(gy), 0), gp.ny - 1),
            cz = min(max((int)floorf(gz), 0), gp.nz - 1);
  bool done = false;
  for (int r = 0; r <= kGridMaxRing && !done; ++r) {
    const int z0 = max(cz - r, 0), z1 = min(cz + r, gp.nz - 1);
    const int y0 = max(cy - r, 0), y1 = min(cy + r, gp.ny - 1);
    const int x0 = max(cx - r, 0), x1 = min(cx + r, gp.nx - 1);
    for (int z = z0; z <= z1; ++z)
      for (int y = y0; y <= y1; ++y) {
        const bool shell_row = (abs(z - cz) == r) || (abs(y - cy) == r);
        const int row = (z * gp.ny + y) * gp.nx;
        if (shell_row) {  // the whole x-run belongs to the shell: cells are contiguous in the sorted array
          const int e0 = start[row + x0], e1 = start[row + x1 + 1];
          for (int e = e0; e < e1; ++e) {
            const float4 p = pts[e];
            const float dx = sx - p.x, dy = sy - p.y, dz = sz - p.z;
            nn_update((dx * dx + dy * dy) + dz * dz, __float_as_int(p.w), best, bi);
          }
        } else {  // only the two end cells of the run are new
          for (int side = 0; side < 2; ++side) {
            const int x = side ? cx + r : cx - r;
            if (x < 0 || x >= gp.nx || (side && r == 0)) continue;
            const int e0 = start[row + x], e1 = start[row + x + 1];
            for (int e = e0; e < e1; ++e) {
              const float4 p = pts[e];
              const float dx = sx - p.x, dy = sy - p.y, dz = sz - p.z;
              nn_update((dx * dx + dy * dy) + dz * dz, __float_as_int(p.w), best, bi);
            }
          }
        }
      }
    // distance (in cells) from the query to the nearest face of the visited cube that still has cells behind it
    float m = 3.0e38f;
    bool open = false;
    if (cx - r > 0) { m = fminf(m, gx - (float)(cx - r)); open = true; }
    if (cx + r < gp.nx - 1) { m = fminf(m, (float)(cx + r + 1) - gx); open = true; }
    if (cy - r > 0) { m = fminf(m, gy - (float)(cy - r)); open = true; }
    if (cy + r < gp.ny - 1) { m = fminf(m, (float)(cy + r + 1) - gy); open = true; }
    if (cz - r > 0) { m = fminf(m, gz - (float)(cz - r)); open = true; }
    if (cz + r < gp.nz - 1) { m = fminf(m, (float)(cz + r + 1) - gz); open = true; }
    if (!open) {
      done = true;  // the cube covers the whole grid
    } else if (bi >= 0 && m > 1e-3f) {
      // 1e-3 cells of slack covers the rounding of the cell assignment (|error| < 2e-5 cells for <= 65 cells)
      const float lim = (m - 1e-3f) * gp.c;
      if (best <= lim * lim) done = true;
    }
  }
  if (!done) {  // rare: a query far from every target point -> exact full scan
    for (int e = 0; e < nt; ++e) {
      const float4 p = pts[e];
      const float dx = sx - p.x, dy = sy - p.y, dz = sz - p.z;
      nn_update((dx * dx + dy * dy) + dz * dz, __float_as_int(p.w), best, bi);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------
// exact 1-NN + point-to-plane linearisation + block reduction
// ---------------------------------------------------------------------------------------------------------
struct KnnArgs {
  float *src;  // (B, ns_stride, 3); read, optionally rewritten with the transformed points
  const int32_t *src_count;
  int ns_stride;
  const float *tgt_p, *tgt_n;  // (B, nt_stride, 3)
  const int32_t *tgt_count;
  int nt_stride;
  const float *pre;  // (B,16) transform applied to src on load, or null
  int write_back;
  float dist_thresh;  // compared with the SQUARED nn distance as the reference does (icputils.py:206)
  int use_thresh;
  float *partials;  // (B, gridDim.x, 28)
  int64_t *nn_idx;  // optional (B, ns_stride): nn index per source point (-1 = filtered / invalid)
  float *nn_d2;     // optional (B, ns_stride)
  TargetGrid grid;  // used by the kGrid variant
};

// point-to-plane row of one association and its 28 products (gauss_newton_solve, icputils.py:227-230)
__device__ __forceinline__ void row_products(float sx, float sy, float sz, const float *__restrict__ tp,
                                             const float *__restrict__ tn, int64_t bi, float *acc) {
  const float dx = __ldg(tp + bi * 3), dy = __ldg(tp + bi * 3 + 1), dz = __ldg(tp + bi * 3 + 2);
  const float nx = __ldg(tn + bi * 3), ny = __ldg(tn + bi * 3 + 1), nz = __ldg(tn + bi * 3 + 2);
  float A[6];
  A[0] = nx; A[1] = ny; A[2] = nz;
  A[3] = nz * sy - ny * sz;
  A[4] = nx * sz - nz * sx;
  A[5] = ny * sx - nx * sy;
  const float r = (nx * (dx - sx) + ny * (dy - sy)) + nz * (dz - sz);
  int k = 0;
#pragma unroll
  for (int p = 0; p < 6; ++p)
#pragma unroll
    for (int q = p; q < 6; ++q) acc[k++] = A[p] * A[q];
#pragma unroll
  for (int p = 0; p < 6; ++p) acc[21 + p] = A[p] * r;
  acc[27] = r * r;
}

// deterministic block reduction of the 28 sums: butterfly inside the warp, then warps in index order
__device__ __forceinline__ void block_reduce_sums(float *acc, float (*s_red)[kNumSums], float *out) {
#pragma unroll
  for (int k = 0; k < kNumSums; ++k) {
    float v = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    acc[k] = v;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < kNumSums; ++k) s_red[warp][k] = acc[k];
  }
  __syncthreads();
  if (threadIdx.x < kNumSums) {
    float v = 0.0f;
#pragma unroll
    for (int w = 0; w < kIcpBlock / 32; ++w) v += s_red[w][threadIdx.x];
    out[threadIdx.x] = v;
  }
}

template <bool kGrid>
__global__ void __launch_bounds__(kIcpBlock) k_icp_knn_linearize(KnnArgs a) {
  __shared__ float4 s_t[kGrid ? 1 : kTgtTile];
  __shared__ float s_red[kIcpBlock / 32][kNumSums];
  __shared__ Rigid s_pre;
  const int b = blockIdx.y;
  const int ns = a.src_count[b], nt = a.tgt_count[b];
  const int i = blockIdx.x * kIcpBlock + threadIdx.x;
  if (a.pre && threadIdx.x == 0) s_pre = load_rigid(a.pre + b * 16);
  __syncthreads();
  float *src = a.src + (int64_t)b * a.ns_stride * 3;
  const float *tp = a.tgt_p + (int64_t)b * a.nt_stride * 3;
  const float *tn = a.tgt_n + (int64_t)b * a.nt_stride * 3;
  const bool valid = i < ns;
  float sx = 0.f, sy = 0.f, sz = 0.f;
  if (valid) {
    sx = src[(int64_t)i * 3];
    sy = src[(int64_t)i * 3 + 1];
    sz = src[(int64_t)i * 3 + 2];
    if (a.pre) {
      const float3 q = rigid_apply(s_pre, sx, sy, sz);
      sx = q.x; sy = q.y; sz = q.z;
      if (a.write_back) {
        src[(int64_t)i * 3] = sx;
        src[(int64_t)i * 3 + 1] = sy;
        src[(int64_t)i * 3 + 2] = sz;
      }
    }
  }
  float best = 0.0f;
  int bi = -1;
  if (kGrid) {
    if (valid && nt > 0) search_grid(a.grid, b, nt, a.nt_stride, sx, sy, sz, best, bi);
  } else if (blockIdx.x * kIcpBlock < ns) {  // whole block idle otherwise (uniform)
    for (int base = 0; base < nt; base += kTgtTile) {
      const int m = min(kTgtTile, nt - base);
      __syncthreads();
      for (int t = threadIdx.x; t < m; t += kIcpBlock) {
        const float *p = tp + (int64_t)(base + t) * 3;
        s_t[t] = make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), 0.0f);
      }
      __syncthreads();
      if (valid) {
#pragma unroll 8
        for (int t = 0; t < m; ++t) {
          const float4 p = s_t[t];
          const float dx = sx - p.x, dy = sy - p.y, dz = sz - p.z;
          const float d = (dx * dx + dy * dy) + dz * dz;
          if (bi < 0 || d < best) {  // strict '<' on an ascending scan: lowest index wins ties
            best = d;
            bi = base + t;
          }
        }
      }
    }
  }
  bool use = valid && bi >= 0;
  if (use && a.use_thresh) use = best < a.dist_thresh;
  if (a.nn_idx && valid) {
    a.nn_idx[(int64_t)b * a.ns_stride + i] = use ? (int64_t)bi : -1;
    if (a.nn_d2) a.nn_d2[(int64_t)b * a.ns_stride + i] = best;
  }
  float acc[kNumSums];
#pragma unroll
  for (int k = 0; k < kNumSums; ++k) acc[k] = 0.0f;
  if (use) row_products(sx, sy, sz, tp, tn, (int64_t)bi, acc);
  block_reduce_sums(acc, s_red, a.partials + ((int64_t)b * gridDim.x + blockIdx.x) * kNumSums);
}

// ---------------------------------------------------------------------------------------------------------
// normal equations for a GIVEN association (the differentiable op of the taped ICP): forward + backward
// ---------------------------------------------------------------------------------------------------------
// (batched: element b = blockIdx.y lives at b * ns_stride / b * nt_stride rows; counts may be null = ns_stride rows each)
__global__ void __launch_bounds__(kIcpBlock) k_icp_linearize_idx(const float *src, int ns_stride, const int32_t *counts,
                                                                 const float *tp, const float *tn, int nt_stride,
                                                                 const int64_t *idx, float *partials) {
  __shared__ float s_red[kIcpBlock / 32][kNumSums];
  const int b = blockIdx.y;
  const int ns = counts ? counts[b] : ns_stride;
  src += (int64_t)b * ns_stride * 3;
  tp += (int64_t)b * nt_stride * 3;
  tn += (int64_t)b * nt_stride * 3;
  idx += (int64_t)b * ns_stride;
  partials += (int64_t)b * gridDim.x * kNumSums;
  const int i = blockIdx.x * kIcpBlock + threadIdx.x;
  float acc[kNumSums];
#pragma unroll
  for (int k = 0; k < kNumSums; ++k) acc[k] = 0.0f;
  if (i < ns) {
    const int64_t j = idx[i];
    if (j >= 0) row_products(src[(int64_t)i * 3], src[(int64_t)i * 3 + 1], src[(int64_t)i * 3 + 2], tp, tn, j, acc);
  }
  block_reduce_sums(acc, s_red, partials + (int64_t)blockIdx.x * kNumSums);
}

__global__ void k_icp_reduce_partials(const float *partials, int nblocks, float *sums) {
  partials += (int64_t)blockIdx.x * nblocks * kNumSums;  // (one block per batch element)
  sums += (int64_t)blockIdx.x * kNumSums;
  if (threadIdx.x < kNumSums) {
    float v = 0.0f;
    for (int j = 0; j < nblocks; ++j) v += partials[(int64_t)j * kNumSums + threadIdx.x];
    sums[threadIdx.x] = v;
  }
}

// d(loss)/d(source point), d/d(associated target point), d/d(associated target normal) from d(loss)/d(28 sums).
// One thread per source point; the target gradients are written per SOURCE row (the caller scatters them with the
// association), so there are no atomics.
__global__ void __launch_bounds__(kIcpBlock) k_icp_linearize_bwd(const float *src, int ns_stride, const int32_t *counts,
                                                                 const float *tp, const float *tn, int nt_stride,
                                                                 const int64_t *idx, const float *g, float *g_src,
                                                                 float *g_tp, float *g_tn) {
  __shared__ float s_g[kNumSums];
  const int b = blockIdx.y;
  const int ns = counts ? counts[b] : ns_stride;
  src += (int64_t)b * ns_stride * 3;
  tp += (int64_t)b * nt_stride * 3;
  tn += (int64_t)b * nt_stride * 3;
  idx += (int64_t)b * ns_stride;
  g += (int64_t)b * kNumSums;
  g_src += (int64_t)b * ns_stride * 3;
  g_tp += (int64_t)b * ns_stride * 3;
  g_tn += (int64_t)b * ns_stride * 3;
  if (threadIdx.x < kNumSums) s_g[threadIdx.x] = g[threadIdx.x];
  __syncthreads();
  const int i = blockIdx.x * kIcpBlock + threadIdx.x;
  if (i >= ns_stride) return;
  if (i >= ns) {  // padding rows of a batched call: zero gradients
#pragma unroll
    for (int c = 0; c < 3; ++c) g_src[(int64_t)i * 3 + c] = g_tp[(int64_t)i * 3 + c] = g_tn[(int64_t)i * 3 + c] = 0.0f;
    return;
  }
  float gs[3] = {0.f, 0.f, 0.f}, gp[3] = {0.f, 0.f, 0.f}, gn[3] = {0.f, 0.f, 0.f};
  const int64_t j = idx[i];
  if (j >= 0) {
    const float sx = src[(int64_t)i * 3], sy = src[(int64_t)i * 3 + 1], sz = src[(int64_t)i * 3 + 2];
    const float px = tp[j * 3], py = tp[j * 3 + 1], pz = tp[j * 3 + 2];
    const float nx = tn[j * 3], ny = tn[j * 3 + 1], nz = tn[j * 3 + 2];
    float A[6] = {nx, ny, nz, nz * sy - ny * sz, nx * sz - nz * sx, ny * sx - nx * sy};
    const float r = (nx * (px - sx) + ny * (py - sy)) + nz * (pz - sz);
    // dL/dA_p = sum_{q>=p} G[p,q] A_q + sum_{q<=p} G[q,p] A_q + h_p r ;  dL/dr = sum_p h_p A_p + 2 g_rr r
    float a[6];
    float gr = 2.0f * s_g[27] * r;
#pragma unroll
    for (int p = 0; p < 6; ++p) {
      float v = s_g[21 + p] * r;
      gr += s_g[21 + p] * A[p];
#pragma unroll
      for (int q = 0; q < 6; ++q) {
        const int lo = p < q ? p : q, hi = p < q ? q : p;
        const int k = lo * 6 - lo * (lo - 1) / 2 + (hi - lo);  // index of (lo,hi) in the upper-triangular order
        v += s_g[k] * A[q] * ((p == q) ? 2.0f : 1.0f);
      }
      a[p] = v;
    }
    // A3 = nz sy - ny sz, A4 = nx sz - nz sx, A5 = ny sx - nx sy ;  r = n . (p - s)
    gs[0] = (-nz * a[4] + ny * a[5]) - gr * nx;
    gs[1] = (nz * a[3] - nx * a[5]) - gr * ny;
    gs[2] = (-ny * a[3] + nx * a[4]) - gr * nz;
    gn[0] = (a[0] + sz * a[4] - sy * a[5]) + gr * (px - sx);
    gn[1] = (a[1] - sz * a[3] + sx * a[5]) + gr * (py - sy);
    gn[2] = (a[2] + sy * a[3] - sx * a[4]) + gr * (pz - sz);
    gp[0] = gr * nx; gp[1] = gr * ny; gp[2] = gr * nz;
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    g_src[(int64_t)i * 3 + c] = gs[c];
    g_tp[(int64_t)i * 3 + c] = gp[c];
    g_tn[(int64_t)i * 3 + c] = gn[c];
  }
}

// ---------------------------------------------------------------------------------------------------------
// small per-element kernels: solve, update
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mat4_mul(const float *A, const float *B, float *C) {
  // plain 4x4 product, k accumulated left to right (torch.mm on 4x4, icputils.py:362, 543)
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) {
      float acc = A[i * 4 + 0] * B[0 * 4 + j];
      for (int k = 1; k < 4; ++k) acc = acc + A[i * 4 + k] * B[k * 4 + j];
      C[i * 4 + j] = acc;
    }
}

// se3_exp (se3utils.py:77-115): xi = (v, omega) -> 4x4; for ||omega|| < 1e-6 both R and V are I + hat(omega)
__device__ void se3_exp_dev(const float *xi, float *T) {
  const float vx = xi[0], vy = xi[1], vz = xi[2], wx = xi[3], wy = xi[4], wz = xi[5];
  const float W[9] = {0.f, -wz, wy, wz, 0.f, -wx, -wy, wx, 0.f};
  const float theta = sqrtf((wx * wx + wy * wy) + wz * wz);
  float R[9], V[9];
  if (theta < 1e-6f) {
    for (int i = 0; i < 9; ++i) {
      const float I = (i % 4 == 0) ? 1.0f : 0.0f;
      R[i] = I + W[i];
      V[i] = I + W[i];
    }
  } else {
    const float s = sinf(theta), c = cosf(theta);
    float W2[9];
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) {
        float acc = W[i * 3 + 0] * W[0 * 3 + j];
        for (int k = 1; k < 3; ++k) acc = acc + W[i * 3 + k] * W[k * 3 + j];
        W2[i * 3 + j] = acc;
      }
    const float Ac = s / theta;
    const float Bc = (1.0f - c) / (theta * theta);
    const float Cc = (theta - s) / ((theta * theta) * theta);
    for (int i = 0; i < 9; ++i) {
      const float I = (i % 4 == 0) ? 1.0f : 0.0f;
      R[i] = (I + Ac * W[i]) + Bc * W2[i];
      V[i] = (I + Bc * W[i]) + Cc * W2[i];
    }
  }
  for (int i = 0; i < 3; ++i) {
    T[i * 4 + 0] = R[i * 3 + 0];
    T[i * 4 + 1] = R[i * 3 + 1];
    T[i * 4 + 2] = R[i * 3 + 2];
    T[i * 4 + 3] = (V[i * 3 + 0] * vx + V[i * 3 + 1] * vy) + V[i * 3 + 2] * vz;
  }
  T[12] = 0.f; T[13] = 0.f; T[14] = 0.f; T[15] = 1.f;
}

struct IcpState {     // per element, device resident
  float *T_total;     // (B,16) accumulated transform
  float *T_pend;      // (B,16) transform still to be applied to the source cloud
  float *dT;          // (B,16) Gauss-Newton step of this iteration
  float *xi;          // (B,6)
  float *err;         // (B)
  float *damp;        // (B)
};

__device__ float reduce_partial(const float *partials, int nblocks, int k) {
  float v = 0.0f;
  for (int j = 0; j < nblocks; ++j) v += partials[(int64_t)j * kNumSums + k];
  return v;
}

__global__ void k_icp_solve(const float *partials, int nblocks, IcpState st) {
  __shared__ float s_sum[kNumSums];
  const int b = blockIdx.x;
  const float *p = partials + (int64_t)b * nblocks * kNumSums;
  if (threadIdx.x < kNumSums) s_sum[threadIdx.x] = reduce_partial(p, nblocks, threadIdx.x);
  __syncwarp();
  if (threadIdx.x != 0) return;
  // (A^T A + damp I) x = A^T b by Gauss-Jordan inversion with partial pivoting, then x = inv * A^T b
  float M[6][12];
  int k = 0;
  for (int i = 0; i < 6; ++i)
    for (int j = i; j < 6; ++j) {
      M[i][j] = s_sum[k];
      M[j][i] = s_sum[k];
      ++k;
    }
  const float damp = st.damp[b];
  for (int i = 0; i < 6; ++i) {
    M[i][i] = M[i][i] + damp;
    for (int j = 0; j < 6; ++j) M[i][6 + j] = (i == j) ? 1.0f : 0.0f;
  }
  for (int c = 0; c < 6; ++c) {
    int piv = c;
    float mx = fabsf(M[c][c]);
    for (int r = c + 1; r < 6; ++r)
      if (fabsf(M[r][c]) > mx) {
        mx = fabsf(M[r][c]);
        piv = r;
      }
    if (piv != c)
      for (int j = 0; j < 12; ++j) {
        const float t = M[c][j];
        M[c][j] = M[piv][j];
        M[piv][j] = t;
      }
    const float inv = 1.0f / M[c][c];
    for (int j = 0; j < 12; ++j) M[c][j] *= inv;
    for (int r = 0; r < 6; ++r) {
      if (r == c) continue;
      const float f = M[r][c];
      for (int j = 0; j < 12; ++j) M[r][j] -= f * M[c][j];
    }
  }
  float xi[6];
  for (int i = 0; i < 6; ++i) {
    float acc = 0.0f;
    for (int j = 0; j < 6; ++j) acc += M[i][6 + j] * s_sum[21 + j];
    xi[i] = acc;
    st.xi[b * 6 + i] = acc;
  }
  se3_exp_dev(xi, st.dT + b * 16);
  st.err[b] = s_sum[27];
}

struct UpdateArgs {
  int mode;  // 0 = LM accept/reject (point_to_plane_ICP), 1 = gradLM (point_to_plane_gradICP)
  float lambda_min, lambda_max, B, B2, inv_nu;
};

__global__ void k_icp_update(const float *partials, int nblocks, IcpState st, UpdateArgs u) {
  const int b = blockIdx.x;
  if (threadIdx.x != 0) return;
  const float new_err = reduce_partial(partials + (int64_t)b * nblocks * kNumSums, nblocks, 27);
  const float err = st.err[b];
  float Tn[16], Tp[16];
  float *T = st.T_total + b * 16;
  if (u.mode == 0) {
    if (new_err < err) {  // trust region: accept the step
      for (int i = 0; i < 16; ++i) Tp[i] = st.dT[b * 16 + i];
      st.damp[b] = st.damp[b] / 2.0f;
      mat4_mul(Tp, T, Tn);
      for (int i = 0; i < 16; ++i) T[i] = Tn[i];
    } else {
      for (int i = 0; i < 16; ++i) Tp[i] = (i % 5 == 0) ? 1.0f : 0.0f;
      st.damp[b] = st.damp[b] * 2.0f;
    }
  } else {
    float diff = new_err - err;
    diff = fminf(fmaxf(diff, -70.0f), 70.0f);
    const float gate = u.lambda_min + (u.lambda_max - u.lambda_min) / (1.0f + expf(-u.B * diff));
    st.damp[b] = st.damp[b] * gate;
    const float sig = 1.0f / powf(1.0f + expf(-u.B2 * diff), u.inv_nu);
    float xs[6];
    for (int i = 0; i < 6; ++i) xs[i] = sig * st.xi[b * 6 + i];
    se3_exp_dev(xs, Tp);
    mat4_mul(Tp, T, Tn);
    for (int i = 0; i < 16; ++i) T[i] = Tn[i];
  }
  for (int i = 0; i < 16; ++i) st.T_pend[b * 16 + i] = Tp[i];
}

__global__ void k_icp_init(IcpState st, const float *T0, float damp0, int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  for (int i = 0; i < 16; ++i) {
    const float v = T0 ? T0[b * 16 + i] : ((i % 5 == 0) ? 1.0f : 0.0f);
    st.T_total[b * 16 + i] = v;
    st.T_pend[b * 16 + i] = v;
  }
  st.damp[b] = damp0;
}

// new pose = T_icp · prev pose (kornia compose_transformations as used at slam/icpslam.py:245-247)
__global__ void k_pose_compose(const float *T, const float *prev, int64_t prev_bstride, float *out, int64_t out_bstride,
                               int B) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const float *A = T + b * 16;
  const float *P = prev + b * prev_bstride;
  float *O = out + b * out_bstride;
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) O[i * 4 + j] = dot3(A[i * 4], A[i * 4 + 1], A[i * 4 + 2], P[j], P[4 + j], P[8 + j]);
    O[i * 4 + 3] = dot3(A[i * 4], A[i * 4 + 1], A[i * 4 + 2], P[3], P[7], P[11]) + A[i * 4 + 3];
  }
  O[12] = 0.f; O[13] = 0.f; O[14] = 0.f; O[15] = 1.f;
}

// ---------------------------------------------------------------------------------------------------------
// workspace
// ---------------------------------------------------------------------------------------------------------
struct IcpWorkspace {
  float *src;  // (B, ns_cap, 3)
  int32_t *src_count, *tgt_count;
  float *partials;  // (B, nblk, 28)
  IcpState st;
  unsigned long long *tile_state;
  unsigned int *ticket;
  int ns_cap, nblk, tiles_cap;
};

inline int64_t up256(int64_t x) { return (x + 255) / 256 * 256; }

inline int icp_ns_cap(int H, int W, int ds) { return ((H + ds - 1) / ds) * ((W + ds - 1) / ds); }

inline int64_t icp_workspace_bytes(int B, int H, int W, int ds, int64_t map_capacity) {
  const int ns = icp_ns_cap(H, W, ds);
  const int nblk = (ns + kIcpBlock - 1) / kIcpBlock;
  const int64_t tiles = (map_capacity + 1023) / 1024;
  return up256((int64_t)B * ns * 12) + 2 * up256((int64_t)B * 4) + up256((int64_t)B * nblk * kNumSums * 4) +
         4 * up256((int64_t)B * 64) + 3 * up256((int64_t)B * 24) + up256(B * tiles * 8) + up256((int64_t)B * 4);
}

inline IcpWorkspace icp_carve(void *ws, int B, int H, int W, int ds, int64_t map_capacity) {
  IcpWorkspace w;
  w.ns_cap = icp_ns_cap(H, W, ds);
  w.nblk = (w.ns_cap + kIcpBlock - 1) / kIcpBlock;
  w.tiles_cap = (int)((map_capacity + 1023) / 1024);
  char *p = (char *)ws;
  w.src = (float *)p;            p += up256((int64_t)B * w.ns_cap * 12);
  w.src_count = (int32_t *)p;    p += up256((int64_t)B * 4);
  w.tgt_count = (int32_t *)p;    p += up256((int64_t)B * 4);
  w.partials = (float *)p;       p += up256((int64_t)B * w.nblk * kNumSums * 4);
  w.st.T_total = (float *)p;     p += up256((int64_t)B * 64);
  w.st.T_pend = (float *)p;      p += up256((int64_t)B * 64);
  w.st.dT = (float *)p;          p += up256((int64_t)B * 64);
  p += up256((int64_t)B * 64);   // spare
  w.st.xi = (float *)p;          p += up256((int64_t)B * 24);
  w.st.err = (float *)p;         p += up256((int64_t)B * 24);
  w.st.damp = (float *)p;        p += up256((int64_t)B * 24);
  w.tile_state = (unsigned long long *)p;  p += up256((int64_t)B * w.tiles_cap * 8);
  w.ticket = (unsigned int *)p;
  return w;
}

// runs the LM / gradLM loop on clouds that are already in place
constexpr int kGridThreshold = 4096;  // target clouds up to this size use the shared-memory brute force

inline int64_t grid_bytes(int B, int nt_stride) {
  if (nt_stride <= kGridThreshold) return 0;
  return up256((int64_t)B * sizeof(GridParams)) + up256((int64_t)B * (kGridMaxCells + 1) * 4) +
         up256((int64_t)B * kGridMaxCells * 4) + up256((int64_t)B * nt_stride * 16);
}

inline TargetGrid grid_carve(void *mem, int B, int nt_stride) {
  TargetGrid g;
  char *p = (char *)mem;
  g.params = (GridParams *)p;  p += up256((int64_t)B * sizeof(GridParams));
  g.cell_start = (int *)p;     p += up256((int64_t)B * (kGridMaxCells + 1) * 4);
  g.cursor = (int *)p;         p += up256((int64_t)B * kGridMaxCells * 4);
  g.sorted = (float4 *)p;
  return g;
}

int run_icp_loop(float *src, const int32_t *src_count, int ns_stride, const float *tgt_p, const float *tgt_n,
                 const int32_t *tgt_count, int nt_stride, int B, const float *T0, int mode, int numiters, float damp,
                 int use_thresh, float dist_thresh, float lambda_max, float Bp, float B2p, float nu, float *partials,
                 int nblk_cap, IcpState st, int64_t *nn_idx, void *grid_mem, cudaStream_t stream) {
  const int nblk = (ns_stride + kIcpBlock - 1) / kIcpBlock;
  if (nblk > nblk_cap) {
    set_error("icp: source cloud larger than workspace");
    return 1;
  }
  k_icp_init<<<(B + 63) / 64, 64, 0, stream>>>(st, T0, damp, B);
  UpdateArgs u{mode, 1.0f / lambda_max, lambda_max, Bp, B2p, 1.0f / nu};
  KnnArgs ka{src, src_count, ns_stride, tgt_p, tgt_n, tgt_count, nt_stride, nullptr, 0, dist_thresh, use_thresh,
             partials, nullptr, nullptr, TargetGrid{}};
  const bool use_grid = grid_mem != nullptr && nt_stride > kGridThreshold;
  if (use_grid) {  // the target is fixed for the whole loop: bin it once
    ka.grid = grid_carve(grid_mem, B, nt_stride);
    const unsigned nb = (unsigned)((nt_stride + 255) / 256);
    k_grid_bbox<<<B, 256, 0, stream>>>(tgt_p, tgt_count, nt_stride, ka.grid);
    k_grid_clear<<<(unsigned)(((int64_t)B * kGridMaxCells + 255) / 256), 256, 0, stream>>>(ka.grid, B);
    k_grid_count<<<dim3(nb, (unsigned)B), 256, 0, stream>>>(tgt_p, tgt_count, nt_stride, ka.grid);
    k_grid_scan<<<B, 1024, 0, stream>>>(ka.grid);
    k_grid_scatter<<<dim3(nb, (unsigned)B), 256, 0, stream>>>(tgt_p, tgt_count, nt_stride, ka.grid);
  }
  const dim3 grid((unsigned)nblk, (unsigned)B);
  for (int it = 0; it < numiters; ++it) {
    ka.pre = st.T_pend;
    ka.write_back = 1;
    ka.nn_idx = (it == numiters - 1) ? nn_idx : nullptr;
    if (use_grid) k_icp_knn_linearize<true><<<grid, kIcpBlock, 0, stream>>>(ka);
    else k_icp_knn_linearize<false><<<grid, kIcpBlock, 0, stream>>>(ka);
    k_icp_solve<<<B, 32, 0, stream>>>(partials, nblk, st);
    ka.pre = st.dT;
    ka.write_back = 0;
    ka.nn_idx = nullptr;
    if (use_grid) k_icp_knn_linearize<true><<<grid, kIcpBlock, 0, stream>>>(ka);
    else k_icp_knn_linearize<false><<<grid, kIcpBlock, 0, stream>>>(ka);
    k_icp_update<<<B, 32, 0, stream>>>(partials, nblk, st, u);
  }
  GSX_CHECK_LAUNCH("gsx_icp");
  return 0;
}

}  // namespace gsx

using namespace gsx;

extern "C" int64_t gsx_icp_workspace_bytes(int B, int H, int W, int ds, int64_t map_capacity) {
  if (B < 0 || H < 1 || W < 1 || ds < 1 || map_capacity < 0) return -1;
  return icp_workspace_bytes(B, H, W, ds, map_capacity);
}

extern "C" int gsx_icp_align(const float *src_points, const int32_t *src_count, int ns_stride, const float *tgt_points,
                             const float *tgt_normals, const int32_t *tgt_count, int nt_stride, int B,
                             const float *initial_transform, int mode, int numiters, float damp, int use_dist_thresh,
                             float dist_thresh, float lambda_max, float Bp, float B2p, float nu, float *transform_out,
                             int64_t *nn_idx_out, void *scratch, int64_t scratch_bytes, void *stream) {
  GSX_CHECK_ARG(src_points && src_count && tgt_points && tgt_normals && tgt_count && transform_out && scratch,
                "gsx_icp_align: null pointer");
  GSX_CHECK_ARG(B >= 1 && ns_stride >= 1 && nt_stride >= 1 && numiters >= 0, "gsx_icp_align: bad extents");
  GSX_CHECK_ARG(mode == 0 || mode == 1, "gsx_icp_align: mode must be 0 (ICP) or 1 (gradICP)");
  // scratch: working copy of src (B,ns,3) + partials + state
  const int nblk = (ns_stride + kIcpBlock - 1) / kIcpBlock;
  const int64_t need = up256((int64_t)B * ns_stride * 12) + up256((int64_t)B * nblk * kNumSums * 4) +
                       3 * up256((int64_t)B * 64) + 3 * up256((int64_t)B * 24) + grid_bytes(B, nt_stride);
  GSX_CHECK_ARG(scratch_bytes >= need, "gsx_icp_align: scratch too small (%lld < %lld)", (long long)scratch_bytes,
                (long long)need);
  char *p = (char *)scratch;
  float *src = (float *)p;       p += up256((int64_t)B * ns_stride * 12);
  float *partials = (float *)p;  p += up256((int64_t)B * nblk * kNumSums * 4);
  IcpState st;
  st.T_total = (float *)p;       p += up256((int64_t)B * 64);
  st.T_pend = (float *)p;        p += up256((int64_t)B * 64);
  st.dT = (float *)p;            p += up256((int64_t)B * 64);
  st.xi = (float *)p;            p += up256((int64_t)B * 24);
  st.err = (float *)p;           p += up256((int64_t)B * 24);
  st.damp = (float *)p;        p += up256((int64_t)B * 24);
  void *grid_mem = grid_bytes(B, nt_stride) ? (void *)p : nullptr;
  cudaStream_t s = (cudaStream_t)stream;
  cudaMemcpyAsync(src, src_points, (size_t)B * ns_stride * 12, cudaMemcpyDeviceToDevice, s);
  const int rc = run_icp_loop(src, src_count, ns_stride, tgt_points, tgt_normals, tgt_count, nt_stride, B,
                              initial_transform, mode, numiters, damp, use_dist_thresh, dist_thresh, lambda_max, Bp,
                              B2p, nu, partials, nblk, st, nn_idx_out, grid_mem, s);
  if (rc) return rc;
  cudaMemcpyAsync(transform_out, st.T_total, (size_t)B * 64, cudaMemcpyDeviceToDevice, s);
  return 0;
}

extern "C" int64_t gsx_icp_align_scratch_bytes(int B, int ns_stride, int nt_stride) {
  if (B < 1 || ns_stride < 1 || nt_stride < 1) return -1;
  const int nblk = (ns_stride + kIcpBlock - 1) / kIcpBlock;
  return up256((int64_t)B * ns_stride * 12) + up256((int64_t)B * nblk * kNumSums * 4) + 3 * up256((int64_t)B * 64) +
         3 * up256((int64_t)B * 24) + grid_bytes(B, nt_stride);
}

extern "C" int64_t gsx_icp_tgt_scratch_bytes(int B, int64_t tgt_capacity) {
  if (B < 1 || tgt_capacity < 1 || tgt_capacity > (1ll << 30)) return -1;
  return 2 * up256((int64_t)B * tgt_capacity * 12) + grid_bytes(B, (int)tgt_capacity);
}

extern "C" int gsx_icp_localize(const float *map_geometry, const int32_t *counts,
                                int64_t capacity, int64_t max_count, const float *depth, int64_t depth_bstride,
                                const float *intrinsics, int64_t K_bstride, const float *prev_poses,
                                int64_t prev_pose_bstride, int B, int H, int W, int ds, int mode, int numiters,
                                float damp, int use_dist_thresh, float dist_thresh, float lambda_max, float Bp,
                                float B2p, float nu, void *tgt_scratch, int64_t tgt_capacity, float *poses_out,
                                int64_t poses_out_bstride, void *workspace, int64_t workspace_map_capacity,
                                uint32_t epoch, int32_t *overflow_flag, void *stream) {
  GSX_CHECK_ARG(map_geometry && counts && depth && intrinsics && prev_poses && poses_out && workspace && tgt_scratch,
                "gsx_icp_localize: null pointer");
  GSX_CHECK_ARG((reinterpret_cast<uintptr_t>(map_geometry) & 15) == 0,
                "gsx_icp_localize: geometry rows must be 16-byte aligned");
  GSX_CHECK_ARG(B >= 1 && H >= 2 && W >= 2 && ds >= 1, "gsx_icp_localize: bad extents");
  GSX_CHECK_ARG(mode == 0 || mode == 1, "gsx_icp_localize: mode must be 0 (ICP) or 1 (gradICP)");
  GSX_CHECK_ARG(max_count <= capacity && tgt_capacity >= 1, "gsx_icp_localize: bad capacities");
  GSX_CHECK_ARG(epoch >= 1 && epoch < (1u << 30), "gsx_icp_localize: epoch out of range");
  cudaStream_t s = (cudaStream_t)stream;
  GSX_CHECK_ARG(workspace_map_capacity >= max_count, "gsx_icp_localize: workspace sized for a smaller map");
  // the layout of the workspace is fixed by the capacity it was created for, not by today's map capacity
  IcpWorkspace w = icp_carve(workspace, B, H, W, ds, workspace_map_capacity);
  GSX_CHECK_ARG(tgt_capacity < (1ll << 30), "gsx_icp_localize: tgt_capacity too large");
  float *tgt_p = (float *)tgt_scratch;
  float *tgt_n = (float *)((char *)tgt_scratch + up256((int64_t)B * tgt_capacity * 12));
  void *grid_mem = grid_bytes(B, (int)tgt_capacity)
                       ? (void *)((char *)tgt_scratch + 2 * up256((int64_t)B * tgt_capacity * 12))
                       : nullptr;
  GatherSrcArgs gs{depth, depth_bstride, intrinsics, K_bstride, prev_poses, prev_pose_bstride, B, H, W, ds,
                   w.src, w.src_count, w.ns_cap};
  k_icp_gather_src<<<B, 1024, 0, s>>>(gs);
  int tiles = (int)((max_count + 1023) / 1024);
  if (tiles > w.tiles_cap) tiles = w.tiles_cap;
  if (tiles == 0) cudaMemsetAsync(w.tgt_count, 0, (size_t)B * 4, s);
  if (tiles > 0) {
    GatherTgtArgs gt{map_geometry, counts, capacity, prev_poses, prev_pose_bstride, intrinsics, K_bstride,
                     B, H, W, ds, (float)(W - 0.999), (float)(H - 0.999), tgt_p, tgt_n, w.tgt_count,
                     (int)tgt_capacity, w.tile_state, w.ticket, tiles, epoch, overflow_flag};
    k_icp_gather_tgt<<<dim3((unsigned)(tiles * B)), kIcpBlock, 0, s>>>(gt);
  }
  GSX_CHECK_LAUNCH("gsx_icp_localize(gather)");
  const int rc = run_icp_loop(w.src, w.src_count, w.ns_cap, tgt_p, tgt_n, w.tgt_count, (int)tgt_capacity, B, nullptr,
                              mode, numiters, damp, use_dist_thresh, dist_thresh, lambda_max, Bp, B2p, nu, w.partials,
                              w.nblk, w.st, nullptr, grid_mem, s);
  if (rc) return rc;
  k_pose_compose<<<(B + 63) / 64, 64, 0, s>>>(w.st.T_total, prev_poses, prev_pose_bstride, poses_out,
                                              poses_out_bstride, B);
  GSX_CHECK_LAUNCH("gsx_icp_localize(compose)");
  return 0;
}

extern "C" int64_t gsx_knn1_scratch_bytes(int B, int ns_stride, int nt_stride) {
  if (B < 1 || ns_stride < 1 || nt_stride < 1) return -1;
  const int nblk = (ns_stride + kIcpBlock - 1) / kIcpBlock;
  return up256((int64_t)B * nblk * kNumSums * 4) + grid_bytes(B, nt_stride);
}

extern "C" int gsx_knn1(const float *src_points, const int32_t *src_count, int ns_stride, const float *tgt_points,
                        const int32_t *tgt_count, int nt_stride, int B, int64_t *idx_out, float *d2_out,
                        void *scratch, int64_t scratch_bytes, int build_grid, void *stream) {
  GSX_CHECK_ARG(src_points && src_count && tgt_points && tgt_count && idx_out && scratch, "gsx_knn1: null pointer");
  GSX_CHECK_ARG(B >= 1 && ns_stride >= 1 && nt_stride >= 1, "gsx_knn1: bad extents");
  const int nblk = (ns_stride + kIcpBlock - 1) / kIcpBlock;
  const int64_t part = up256((int64_t)B * nblk * kNumSums * 4);
  GSX_CHECK_ARG(scratch_bytes >= part + grid_bytes(B, nt_stride), "gsx_knn1: scratch too small");
  // the target normals are not needed for the association itself: reuse the points as a placeholder
  KnnArgs ka{const_cast<float *>(src_points), src_count, ns_stride, tgt_points, tgt_points, tgt_count, nt_stride,
             nullptr, 0, 0.0f, 0, (float *)scratch, idx_out, d2_out, TargetGrid{}};
  cudaStream_t s = (cudaStream_t)stream;
  const dim3 grid((unsigned)nblk, (unsigned)B);
  if (nt_stride > kGridThreshold) {
    ka.grid = grid_carve((char *)scratch + part, B, nt_stride);
    if (build_grid) {  // (0: `scratch` still holds the grid a previous call built for this very target)
      const unsigned nb = (unsigned)((nt_stride + 255) / 256);
      k_grid_bbox<<<B, 256, 0, s>>>(tgt_points, tgt_count, nt_stride, ka.grid);
      k_grid_clear<<<(unsigned)(((int64_t)B * kGridMaxCells + 255) / 256), 256, 0, s>>>(ka.grid, B);
      k_grid_count<<<dim3(nb, (unsigned)B), 256, 0, s>>>(tgt_points, tgt_count, nt_stride, ka.grid);
      k_grid_scan<<<B, 1024, 0, s>>>(ka.grid);
      k_grid_scatter<<<dim3(nb, (unsigned)B), 256, 0, s>>>(tgt_points, tgt_count, nt_stride, ka.grid);
    }
    k_icp_knn_linearize<true><<<grid, kIcpBlock, 0, s>>>(ka);
  } else {
    k_icp_knn_linearize<false><<<grid, kIcpBlock, 0, s>>>(ka);
  }
  GSX_CHECK_LAUNCH("gsx_knn1");
  return 0;
}

extern "C" int64_t gsx_icp_normal_eq_scratch_bytes(int ns) {
  if (ns < 1) return -1;
  return (int64_t)((ns + kIcpBlock - 1) / kIcpBlock) * kNumSums * 4;
}

extern "C" int gsx_icp_normal_eq_batched_fwd(const float *src_points, const int32_t *src_count, int ns_stride,
                                             const float *tgt_points, const float *tgt_normals, int nt_stride, int B,
                                             const int64_t *nn_idx, float *sums_out, void *scratch, int64_t scratch_bytes,
                                             void *stream) {
  GSX_CHECK_ARG(src_points && tgt_points && tgt_normals && nn_idx && sums_out && scratch,
                "gsx_icp_normal_eq_batched_fwd: null pointer");
  GSX_CHECK_ARG(B >= 1 && ns_stride >= 1 && nt_stride >= 1 &&
                    scratch_bytes >= (int64_t)B * gsx_icp_normal_eq_scratch_bytes(ns_stride),
                "gsx_icp_normal_eq_batched_fwd: bad sizes");
  const int nblk = (ns_stride + kIcpBlock - 1) / kIcpBlock;
  cudaStream_t s = (cudaStream_t)stream;
  k_icp_linearize_idx<<<dim3((unsigned)nblk, (unsigned)B), kIcpBlock, 0, s>>>(src_points, ns_stride, src_count, tgt_points,
                                                                            tgt_normals, nt_stride, nn_idx,
                                                                            (float *)scratch);
  k_icp_reduce_partials<<<B, 32, 0, s>>>((const float *)scratch, nblk, sums_out);
  GSX_CHECK_LAUNCH("gsx_icp_normal_eq_batched_fwd");
  return 0;
}

extern "C" int gsx_icp_normal_eq_batched_bwd(const float *src_points, const int32_t *src_count, int ns_stride,
                                             const float *tgt_points, const float *tgt_normals, int nt_stride, int B,
                                             const int64_t *nn_idx, const float *g_sums, float *g_src,
                                             float *g_tgt_points_rows, float *g_tgt_normals_rows, void *stream) {
  GSX_CHECK_ARG(src_points && tgt_points && tgt_normals && nn_idx && g_sums && g_src && g_tgt_points_rows &&
                    g_tgt_normals_rows,
                "gsx_icp_normal_eq_batched_bwd: null pointer");
  GSX_CHECK_ARG(B >= 1 && ns_stride >= 1 && nt_stride >= 1, "gsx_icp_normal_eq_batched_bwd: bad sizes");
  const int nblk = (ns_stride + kIcpBlock - 1) / kIcpBlock;
  k_icp_linearize_bwd<<<dim3((unsigned)nblk, (unsigned)B), kIcpBlock, 0, (cudaStream_t)stream>>>(
      src_points, ns_stride, src_count, tgt_points, tgt_normals, nt_stride, nn_idx, g_sums, g_src, g_tgt_points_rows,
      g_tgt_normals_rows);
  GSX_CHECK_LAUNCH("gsx_icp_normal_eq_batched_bwd");
  return 0;
}
