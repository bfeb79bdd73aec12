// nope_b200 -- VSD evaluation (src/poses/vsd.py, vsd_utils.py): a z-buffer rasterizer for many
// (mesh, pose) depth renders and the fused Visible Surface Discrepancy error.  Plain SIMT kernels.
//
// Rasterizer conventions (the ones the reference's pyrender IntrinsicsCamera + OpenCV flip implies):
//   camera x right, y down, z forward; pixel (col x, row y) samples the image point (x + 0.5, y + 0.5);
//   depth = camera z of the nearest surface with znear <= z <= zfar, 0 where nothing is hit.
// Geometry is carried in float64 from the vertex pass on, so edges and depths agree with a float64 ray
// cast to ~1e-9 px.  Edge functions are evaluated with the edge's endpoints in a canonical order and
// without FMA contraction, so two triangles sharing an edge compute bit-identical (negated) values and a
// top-left rule gives each sample on the edge to exactly one of them: closed meshes have no cracks.
// Depth is resolved with atomicMin on the bit pattern of positive floats (order-independent, so renders
// are bit-reproducible whatever the launch grouping).
#pragma once

namespace nope {

constexpr int kVsdBigTriPixels = 1024;   // a face whose clipped bbox covers more pixels goes to the CTA path
constexpr int kVsdBigTriCtas = 1184;     // 8 per SM: the CTA path is a grid-stride loop over deferred faces
constexpr int kVsdErrPixelsPerCta = 4096;

struct VsdRenderInfo {       // per render, built on the host from the mesh table
  int nv, nf;                // vertex / face count of the render's mesh
  long long vbase, fbase;    // the mesh's first vertex / face in the packed table
  long long wbase;           // first transformed vertex of this render in the workspace
};

struct VsdPoly {             // a face clipped to znear <= z <= zfar: a convex polygon of up to 5 vertices
  int n;
  double x[5], y[5], iz[5];  // screen position (K's pixel coordinates) and 1/z
};

__global__ void vsd_vertex_kernel(const float* __restrict__ verts, const float* __restrict__ poses,
                                  const VsdRenderInfo* __restrict__ info, double* __restrict__ cam) {
  const int p = blockIdx.y;
  const VsdRenderInfo ri = info[p];
  const float* T = poses + 12 * (size_t)p;
  for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < ri.nv; v += gridDim.x * blockDim.x) {
    const float* X = verts + 3 * (ri.vbase + v);
    const double x = X[0], y = X[1], z = X[2];
    double* o = cam + 3 * (ri.wbase + v);
#pragma unroll
    for (int r = 0; r < 3; ++r)
      o[r] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn((double)T[4 * r], x), __dmul_rn((double)T[4 * r + 1], y)),
                                 __dmul_rn((double)T[4 * r + 2], z)), (double)T[4 * r + 3]);
  }
}

// Sutherland-Hodgman against z >= znear (keep_ge) or z <= zfar.  An intersection is always computed from
// (inside vertex, outside vertex), so the faces on both sides of an edge create the same point bit for bit.
__device__ __forceinline__ int vsd_clip(const double (&ix)[5], const double (&iy)[5], const double (&iz)[5], int n,
                                        double plane, bool keep_ge, double (&ox)[5], double (&oy)[5],
                                        double (&oz)[5]) {
  int m = 0;
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    if (i >= n) break;
    const int j = (i + 1 == n) ? 0 : i + 1;
    const bool in_i = keep_ge ? iz[i] >= plane : iz[i] <= plane;
    const bool in_j = keep_ge ? iz[j] >= plane : iz[j] <= plane;
    if (in_i && m < 5) { ox[m] = ix[i]; oy[m] = iy[i]; oz[m] = iz[i]; ++m; }
    if (in_i != in_j && m < 5) {
      const int a = in_i ? i : j, b = in_i ? j : i;
      const double t = (plane - iz[a]) / (iz[b] - iz[a]);
      ox[m] = __dadd_rn(ix[a], __dmul_rn(t, __dsub_rn(ix[b], ix[a])));
      oy[m] = __dadd_rn(iy[a], __dmul_rn(t, __dsub_rn(iy[b], iy[a])));
      oz[m] = plane;
      ++m;
    }
  }
  return m;
}

// Camera-space face -> clipped, projected polygon.  Returns false for a face with a bad index.
__device__ __forceinline__ bool vsd_setup_face(const int* __restrict__ faces, const double* __restrict__ cam,
                                               const VsdRenderInfo& ri, int f, const double* __restrict__ K,
                                               double znear, double zfar, VsdPoly& poly) {
  const int* F = faces + 3 * (ri.fbase + f);
  double ax[5], ay[5], az[5], bx[5], by[5], bz[5];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const int v = F[c];
    if (v < 0 || v >= ri.nv) return false;
    const double* P = cam + 3 * (ri.wbase + v);
    ax[c] = P[0]; ay[c] = P[1]; az[c] = P[2];
  }
  poly.n = 0;
  if (az[0] < znear && az[1] < znear && az[2] < znear) return true;
  if (az[0] > zfar && az[1] > zfar && az[2] > zfar) return true;
  int n = vsd_clip(ax, ay, az, 3, znear, true, bx, by, bz);
  n = vsd_clip(bx, by, bz, n, zfar, false, ax, ay, az);
  const double fx = K[0], fy = K[1], cx = K[2], cy = K[3];
#pragma unroll
  for (int i = 0; i < 5; ++i) {
    if (i < n) {
      const double iz = 1.0 / az[i];
      poly.x[i] = __dadd_rn(__dmul_rn(fx, __dmul_rn(ax[i], iz)), cx);
      poly.y[i] = __dadd_rn(__dmul_rn(fy, __dmul_rn(ay[i], iz)), cy);
      poly.iz[i] = iz;
    }
  }
  poly.n = n;
  return true;
}

// Pixel bbox of the samples (x + 0.5, y + 0.5) a triangle can cover, clamped to the image.
__device__ __forceinline__ bool vsd_tri_bbox(const double (&x)[3], const double (&y)[3], int H, int W, int& x0,
                                             int& x1, int& y0, int& y1) {
  const double mnx = fmin(x[0], fmin(x[1], x[2])), mxx = fmax(x[0], fmax(x[1], x[2]));
  const double mny = fmin(y[0], fmin(y[1], y[2])), mxy = fmax(y[0], fmax(y[1], y[2]));
  if (!(mxx >= 0.5 && mnx <= W - 0.5 && mxy >= 0.5 && mny <= H - 0.5)) return false;   // also rejects NaN
  x0 = (int)fmax(ceil(mnx - 0.5), 0.0);
  x1 = (int)fmin(floor(mxx - 0.5), (double)(W - 1));
  y0 = (int)fmax(ceil(mny - 0.5), 0.0);
  y1 = (int)fmin(floor(mxy - 0.5), (double)(H - 1));
  return x0 <= x1 && y0 <= y1;
}

// Edge function of sample (sx, sy) against the directed edge a -> b, evaluated with the endpoints in
// lexicographic order (then negated if a > b): both faces of a shared edge get exactly opposite values.
__device__ __forceinline__ double vsd_edge(double ax, double ay, double bx, double by, double sx, double sy) {
  const bool swap = (bx < ax) || (bx == ax && by < ay);
  const double px = swap ? bx : ax, py = swap ? by : ay, qx = swap ? ax : bx, qy = swap ? ay : by;
  const double e = __dsub_rn(__dmul_rn(__dsub_rn(qx, px), __dsub_rn(sy, py)),
                             __dmul_rn(__dsub_rn(qy, py), __dsub_rn(sx, px)));
  return swap ? -e : e;
}

struct VsdTri {
  double x[3], y[3], iz[3];
  double inv_area;     // 1 / signed area
  double sgn;          // sign of the area: the face is rasterized whatever its winding (no culling)
  bool tl[3];          // edge i (opposite vertex i) is a top-left edge of the positively oriented triangle
};

__device__ __forceinline__ bool vsd_tri_from_poly(const VsdPoly& poly, int t, VsdTri& T) {
  const int idx[3] = {0, t + 1, t + 2};
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    T.x[c] = poly.x[idx[c]]; T.y[c] = poly.y[idx[c]]; T.iz[c] = poly.iz[idx[c]];
  }
  const double area = vsd_edge(T.x[0], T.y[0], T.x[1], T.y[1], T.x[2], T.y[2]);
  if (!(area > 0.0 || area < 0.0) || isinf(area)) return false;   // degenerate or NaN
  T.sgn = area > 0 ? 1.0 : -1.0;
  T.inv_area = 1.0 / area;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const int a = (i + 1) % 3, b = (i + 2) % 3;
    // direction of edge i once the triangle is oriented positively; antisymmetric in the direction, so of
    // two faces sharing an edge (traversed in opposite directions) exactly one owns samples on it
    const double dx = T.sgn * (T.x[b] - T.x[a]), dy = T.sgn * (T.y[b] - T.y[a]);
    T.tl[i] = (dy < 0.0) || (dy == 0.0 && dx > 0.0);
  }
  return true;
}

__device__ __forceinline__ void vsd_shade(const VsdTri& T, int px, int py, unsigned int* __restrict__ zbuf, int W) {
  const double sx = px + 0.5, sy = py + 0.5;
  double w[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const int a = (i + 1) % 3, b = (i + 2) % 3;
    w[i] = vsd_edge(T.x[a], T.y[a], T.x[b], T.y[b], sx, sy);
    const double s = T.sgn * w[i];
    if (s < 0.0 || (s == 0.0 && !T.tl[i])) return;
  }
  const double iz = __dadd_rn(__dadd_rn(__dmul_rn(w[0], T.iz[0]), __dmul_rn(w[1], T.iz[1])),
                              __dmul_rn(w[2], T.iz[2]));
  const float z = (float)(1.0 / __dmul_rn(iz, T.inv_area));
  if (z > 0.0f) atomicMin(zbuf + (size_t)py * W + px, __float_as_uint(z));
}

__global__ void vsd_fill_kernel(unsigned int* __restrict__ zbuf, size_t n, unsigned int value) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    zbuf[i] = value;
}

// One thread per face.  Faces whose clipped bbox exceeds kVsdBigTriPixels are appended to `big` (render,
// face) and drawn by vsd_big_face_kernel instead.
__global__ void vsd_face_kernel(const int* __restrict__ faces, const double* __restrict__ cam,
                                const VsdRenderInfo* __restrict__ info, const double* __restrict__ intr, int H, int W,
                                double znear, double zfar, unsigned int* __restrict__ depth, int2* __restrict__ big,
                                unsigned int* __restrict__ n_big) {
  const int p = blockIdx.y;
  const VsdRenderInfo ri = info[p];
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= ri.nf) return;
  VsdPoly poly;
  if (!vsd_setup_face(faces, cam, ri, f, intr + 4 * p, znear, zfar, poly) || poly.n < 3) return;
  unsigned int* zbuf = depth + (size_t)p * H * W;
  long long pixels = 0;
  for (int t = 0; t + 2 < poly.n; ++t) {
    const double x[3] = {poly.x[0], poly.x[t + 1], poly.x[t + 2]};
    const double y[3] = {poly.y[0], poly.y[t + 1], poly.y[t + 2]};
    int x0, x1, y0, y1;
    if (vsd_tri_bbox(x, y, H, W, x0, x1, y0, y1)) pixels += (long long)(x1 - x0 + 1) * (y1 - y0 + 1);
  }
  if (pixels == 0) return;
  if (pixels > kVsdBigTriPixels) {
    big[atomicAdd(n_big, 1u)] = make_int2(p, f);
    return;
  }
  for (int t = 0; t + 2 < poly.n; ++t) {
    VsdTri T;
    if (!vsd_tri_from_poly(poly, t, T)) continue;
    int x0, x1, y0, y1;
    if (!vsd_tri_bbox(T.x, T.y, H, W, x0, x1, y0, y1)) continue;
    for (int py = y0; py <= y1; ++py)
      for (int px = x0; px <= x1; ++px) vsd_shade(T, px, py, zbuf, W);
  }
}

// One CTA per deferred face (grid-stride over the list): the CTA's threads share the face's bbox.
__global__ void __launch_bounds__(256) vsd_big_face_kernel(const int* __restrict__ faces,
                                                           const double* __restrict__ cam,
                                                           const VsdRenderInfo* __restrict__ info,
                                                           const double* __restrict__ intr, int H, int W,
                                                           double znear, double zfar,
                                                           unsigned int* __restrict__ depth,
                                                           const int2* __restrict__ big,
                                                           const unsigned int* __restrict__ n_big) {
  const unsigned int n = *n_big;
  for (unsigned int e = blockIdx.x; e < n; e += gridDim.x) {
    const int2 pf = big[e];
    const VsdRenderInfo ri = info[pf.x];
    VsdPoly poly;
    if (!vsd_setup_face(faces, cam, ri, pf.y, intr + 4 * pf.x, znear, zfar, poly)) continue;
    unsigned int* zbuf = depth + (size_t)pf.x * H * W;
    for (int t = 0; t + 2 < poly.n; ++t) {
      VsdTri T;
      if (!vsd_tri_from_poly(poly, t, T)) continue;
      int x0, x1, y0, y1;
      if (!vsd_tri_bbox(T.x, T.y, H, W, x0, x1, y0, y1)) continue;
      const int bw = x1 - x0 + 1;
      const long long cnt = (long long)bw * (y1 - y0 + 1);
      for (long long i = threadIdx.x; i < cnt; i += blockDim.x)
        vsd_shade(T, x0 + (int)(i % bw), y0 + (int)(i / bw), zbuf, W);
    }
  }
}

// +inf (nothing drawn) -> 0, the background value of the reference's renders
__global__ void vsd_finish_kernel(unsigned int* __restrict__ zbuf, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    if (zbuf[i] == 0x7f800000u) zbuf[i] = 0u;
}

// ------------------------------------------------------------------------------------------------
// VSD error: vsd_obj's inner loop (vsd.py:93-135) with the bop19 masks and the step cost.  Grid
// (pixel slice, hypothesis, frame); integer counts are accumulated with atomics (exact, so the result
// does not depend on the order) and turned into errors by vsd_error_finish_kernel.
// ------------------------------------------------------------------------------------------------

// depth_im_to_dist_im_fast (vsd_utils.py:40-62) for one pixel: pre_X = (x - cx) / fx over pixel indices,
// sqrt((pre_X d)^2 + (pre_Y d)^2 + d^2) with numpy's separate roundings (no FMA contraction).
__device__ __forceinline__ double vsd_dist(double d, double pre_x, double pre_y) {
  const double a = __dmul_rn(pre_x, d), b = __dmul_rn(pre_y, d);
  return sqrt(__dadd_rn(__dadd_rn(__dmul_rn(a, a), __dmul_rn(b, b)), __dmul_rn(d, d)));
}

__global__ void __launch_bounds__(256) vsd_error_kernel(const uint16_t* __restrict__ raw, double scale,
                                                        const double* __restrict__ intr,
                                                        const float* __restrict__ dgt,
                                                        const float* __restrict__ dest, int k, int H, int W,
                                                        float delta, double tau,
                                                        unsigned long long* __restrict__ counts) {
  const int j = blockIdx.y, f = blockIdx.z;
  const size_t HW = (size_t)H * W;
  const uint16_t* R = raw + f * HW;
  const float* G = dgt + f * HW;
  const float* E = dest + ((size_t)f * k + j) * HW;
  const double fx = intr[4 * f], fy = intr[4 * f + 1], cx = intr[4 * f + 2], cy = intr[4 * f + 3];
  unsigned int n_union = 0, n_inter = 0, n_cost = 0;
  const size_t end = min(HW, (size_t)(blockIdx.x + 1) * kVsdErrPixelsPerCta);
  for (size_t i = (size_t)blockIdx.x * kVsdErrPixelsPerCta + threadIdx.x; i < end; i += blockDim.x) {
    const float zg = G[i], ze = E[i];
    if (!(zg > 0.0f) && !(ze > 0.0f)) continue;      // both masks need d_model > 0
    const int y = (int)(i / W), x = (int)(i - (size_t)y * W);
    const double pre_x = ((double)x - cx) / fx, pre_y = ((double)y - cy) / fy;
    const double dt = vsd_dist((double)R[i] / scale, pre_x, pre_y);
    const double dg = vsd_dist((double)zg, pre_x, pre_y), de = vsd_dist((double)ze, pre_x, pre_y);
    const float ft = (float)dt;
    // bop19: (float32(d_model) - float32(d_test) <= delta or d_test == 0) and d_model > 0
    const bool vis_gt = (__fsub_rn((float)dg, ft) <= delta || dt == 0.0) && dg > 0.0;
    const bool vis_est = ((__fsub_rn((float)de, ft) <= delta || dt == 0.0) && de > 0.0) || (vis_gt && de > 0.0);
    n_union += (vis_gt || vis_est);
    const bool inter = vis_gt && vis_est;
    n_inter += inter;
    n_cost += inter && fabs(dg - de) >= tau;
  }
  __shared__ unsigned int s[3];
  if (threadIdx.x < 3) s[threadIdx.x] = 0;
  __syncthreads();
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    n_union += __shfl_xor_sync(0xffffffffu, n_union, o);
    n_inter += __shfl_xor_sync(0xffffffffu, n_inter, o);
    n_cost += __shfl_xor_sync(0xffffffffu, n_cost, o);
  }
  if ((threadIdx.x & 31) == 0) {
    atomicAdd(&s[0], n_union);
    atomicAdd(&s[1], n_inter);
    atomicAdd(&s[2], n_cost);
  }
  __syncthreads();
  if (threadIdx.x < 3 && s[threadIdx.x] != 0)
    atomicAdd(counts + 3 * ((size_t)f * k + j) + threadIdx.x, (unsigned long long)s[threadIdx.x]);
}

// error = (costs + |union| - |inter|) / |union|, 1.0 for an empty union (vsd.py:115-135)
__global__ void vsd_error_finish_kernel(const unsigned long long* __restrict__ counts, int n,
                                        double* __restrict__ err) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long u = (long long)counts[3 * i], in = (long long)counts[3 * i + 1], c = (long long)counts[3 * i + 2];
  err[i] = u == 0 ? 1.0 : (double)(c + (u - in)) / (double)u;
}

}  // namespace nope
