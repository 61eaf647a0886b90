// dts_render.cu — batched software rasteriser for the agent camera (Simulator._render_img,
// simulator.py:1707-1951) on sm_100a.  No tensor cores: there is no dense contraction here.
//
// Stream-ordered kernels per frame batch (k_cull, a work-list pre-pass for k_geometry, and k_raster_solo, the lean
// rasteriser of coarse bins lying inside one prim, are described at their definitions):
//   k_frame_setup  thread per env: camera matrices (f64), gluPerspective, counters -> FrameCtx[env]
//   k_geometry     warp per (env, draw item) over the whole GPU: ground / map tile / placed mesh.  Model-view
//                  f64->f32, fixed-function per-vertex lighting, frustum cull, near + guard-band clip, snap to
//                  1/64 px, triangle setup -> 128-byte PrimRec appended to the env's slab.  A road tile is ONE quad:
//                  its 8x8 lit lattice goes to the env's table and the Gouraud interpolant is evaluated per pixel
//                  (render spec tile mode 1); RenderCfg.tessellate switches to the literal 98 triangles (mode 0).
//   k_bin          warp per env: exact (prim, 32x8-px coarse bin) pairs — count, warp scan, scatter — then, dense
//                  over the pairs (one pair per lane), the 80-byte BinRec each pair needs for visibility: edge
//                  functions re-based to the bin corner (exact in 64 bits, then int32), per-fine-bin reject /
//                  trivial-accept bits, the depth plane.  A bin's records are contiguous in HBM.
//   k_raster       persistent warps pull rows of coarse bins (any env) from one global counter.  The bin's records
//                  arrive in shared memory by bulk-async copy (cp.async.bulk + mbarrier, double-buffered per warp:
//                  the next chunk of 32 records lands while the current one is rasterised).  Visibility first: every
//                  lane owns one pixel of an 8x4 fine bin with its 4 MSAA samples (depth + winning prim) in
//                  registers.  Shading is DEFERRED: once per distinct winner of the pixel (1 for interior pixels,
//                  2 on an edge), fetched from the PrimRec by index — overdraw costs no shading.  Bins with one
//                  fully covering prim skip the depth pass.  Box resolve -> u8, rows packed with shuffles and
//                  stored as 32-bit words.
// Arithmetic follows the render spec of DESIGN.md (the CPU checker implements the same spec) bit for bit
// (compiled with -fmad=false; fmaf() is spelled out where the spec has one).
//
// HBM traffic per env-frame: obs store W*H*3 B (compulsory) + PrimRec slab / BinRec lists / lattice table
// (tens of KB per env, written by k_geometry / k_bin and read once by k_raster) + texels (shared, L2-resident).
#include <cstddef>

#include "dts_camera.cuh"
#include "dts_kernels.h"

namespace dts {

namespace {

#ifndef DTS_STATS
#define DTS_STATS 0         // 1: k_raster counts bins / prim visits / shading rounds into the diagnostic counters (tools/raster_stats.py)
#endif
#if DTS_STATS
#define DTS_COUNT(slot, n) do { if (lane == 0) atomicAdd(err + (slot), (n)); } while (0)
#else
#define DTS_COUNT(slot, n) do { } while (0)
#endif
constexpr int kThreads = 256;       // k_raster CTA
constexpr int kRenderMinCtas = 3;   // resident CTAs per SM of k_raster (register budget 65536 / (kThreads * this))
constexpr int kSoloMinCtas = 3;     // resident CTAs per SM of k_raster_solo (register budget 65536 / (256 * this))
constexpr int kWarps = kThreads / 32;
constexpr int kBinW = 8, kBinH = 4;   // fine bin = one warp's pixel block (one pixel per lane)
constexpr int kCFX = 4, kCFY = 2;     // coarse bin = 4 x 2 fine bins = 32 x 8 px: unit of binning and staging
constexpr int kCoarseW = kBinW * kCFX, kCoarseH = kBinH * kCFY;
constexpr int kStage = 32;        // prims staged per pass and warp
constexpr float kGuard = 4.0f;
constexpr int kSub = 64;          // sub-pixel units per pixel
// MSAA sample offsets in 1/64 px, (.375,.125)(.875,.375)(.125,.625)(.625,.875); constexpr so that the
// unrolled sample loops fold them into immediates
__host__ __device__ constexpr int sample_x(int s) { return s == 0 ? 24 : (s == 1 ? 56 : (s == 2 ? 8 : 40)); }
__host__ __device__ constexpr int sample_y(int s) { return s == 0 ? 8 : (s == 1 ? 24 : (s == 2 ? 40 : 56)); }

// Fine bins of coarse bin (cbx, cby) that lie inside a W x H image: all 4 x 2 except on the right / bottom border.
// k_bin hands a bin to k_raster_solo only if its prim covers every one of them; k_raster then skips the bin and
// k_raster_solo draws exactly these fine bins, so all three take them from here.  As bit masks, bit f = fine bin
// (f & 3, f >> 2): fine_bins_inside = row mask & column mask (k_raster keeps the row mask for a whole row of bins).
__device__ __forceinline__ int fine_cols_in_image(int cbx, int W) { return min(kCFX, (W - cbx * kCoarseW + kBinW - 1) / kBinW); }   // 1..4
__device__ __forceinline__ unsigned fine_col_mask(int cbx, int W) {
  const unsigned cols = (1u << fine_cols_in_image(cbx, W)) - 1u;
  return cols | (cols << 4);
}
__device__ __forceinline__ unsigned fine_row_mask(int cby, int H) { return ((cby * kCFY + 1) * kBinH < H) ? 0xffu : 0x0fu; }
__device__ __forceinline__ unsigned fine_bins_inside(int cbx, int cby, int W, int H) { return fine_row_mask(cby, H) & fine_col_mask(cbx, W); }

// The fisheye LUT entry of output pixel (x, y) (FishTab::src_xy, built by dts_set_fisheye_lut): the source pixel, in
// sub-pixels, and whether it lies inside the image (cv2.remap BORDER_CONSTANT: black if not).  x, y are clamped to the
// image, so lanes past its edge read an edge entry; their pixels are not stored.
struct FishSrc { int x, y; bool valid; };
__device__ __forceinline__ FishSrc fish_src(const FishTab& ft, int x, int y, int W, int H) {
  const int gx = min(x, W - 1), gy = min(y, H - 1);
  const int sxy = __ldg(ft.src_xy + gy * W + gx);
  const int sx = (int)(short)(sxy & 0xffff), sy = sxy >> 16;
  return {sx * kSub, sy * kSub, sx != -32768};
}

struct Vtx { float cx, cy, cz, cw, r, g, b, u, v; };

struct __align__(16) PrimRec {   // 128 B in the env's slab, words grouped for 128-bit loads
  int32_t X0, Y0, X1, Y1;        // w0  snapped vertices in cyclic order, orientation normalised (area > 0)
  int32_t X2, Y2, X3, Y3;        // w1  vertex 3: 4th corner of a quad, else a copy of vertex 0
  float z0, zx, zy;              // w2  depth plane anchored at vertex 0 (f0, d/dx, d/dy per pixel)
  int32_t id;                    //     draw id (GL_LESS ties go to the earlier draw)
  float q0, qx, qy, u0;          // w3  q = 1/w, then u*q, v*q, r*q, g*q, b*q
  float ux, uy, v0, vx;          // w4
  float vy;                      // w5
  int32_t ltq;                   //     (lattice slot + 1) | (texture index + 1) << 16 | quad << 24
  uint32_t tex;                  //     DTexture::info of the prim's texture (pool offset >> 8 | log2 w << 24 | log2 h << 28)
  float r0;
  float rx, ry, g0, gx;          // w6
  float gy, b0, bx, by;          // w7
};
static_assert(sizeof(PrimRec) == 128, "PrimRec must be 128 bytes");
static_assert(offsetof(PrimRec, q0) == 48 && offsetof(PrimRec, vy) == 80 && offsetof(PrimRec, rx) == 96, "PrimRec word groups");

struct __align__(16) BinRec {    // 80 B per (prim, coarse bin) pair: what visibility needs, re-based to the bin corner
  int32_t E0[4], A[4], B[4];     // E_k(x,y) = E0_k + A_k*x + B_k*y, x,y in 1/64 px from the bin corner (triangles: E_3 = 0)
  float z0, zx, zy;              // depth plane
  int32_t id;                    // draw id
  int32_t x0, y0;                // anchor vertex relative to the bin corner (sub-pixels)
  uint32_t prim_flags;           // prim index | per fine bin f of the coarse bin: bit 16+f = may touch, bit 24+f = every sample inside
  int32_t kind;                  // bit 0: quad (4 edges), bit 1: ground quad (draw id < 2), bit 2: tiny triangle — its pixel box
                                 // inside the coarse bin is at most 4x4 and sits in the unused 4th-edge slots:
                                 // E0[3] = x0 | y0 << 16, A[3] = x1 | y1 << 16 (pixels from the bin corner, inclusive)
};
static_assert(sizeof(BinRec) == 80, "BinRec layout");
constexpr unsigned kNoPrim = 0xffffu;   // sample not covered by any prim: clear colour

struct Xform { float MV[12], N[9]; };

struct __align__(16) FrameCtx {   // per env, global memory
  double V[12];                  // agent camera modelview (S:1780-1803)
  float P00, P11, P22, P23;      // gluPerspective (S:1761)
  int32_t n_prims, n_lat, overflow, pad;
};

struct __align__(16) GeoWarp {    // per warp of k_geometry, shared memory
  int32_t unlit, pad_[3];        // segment=True: GL_LIGHTING off, the vertex colour is the material colour (S:1730-1733)
  RenderEp ep;
  double V[12];
  float P00, P11, P22, P23;
  Xform x;                       // model-view / normal matrix of the warp's draw item (warp-uniform)
  Vtx corners[4];
  Vtx poly[2][12];               // ping-pong polygon of the warp-parallel clipper
};
using Shared = GeoWarp;           // shade_vertex reads ep and P from it

// MV = V * T(t) * S(sc) * Ry(c,s), N = rot(V) * Ry / sc — float64 then rounded (spec).  Lanes 0..11 each produce
// one entry of the 3x4 matrix (and of N for the rotation part) into the warp's shared Xform.
__device__ __forceinline__ void model_view(const double* V, double tx, double ty, double tz, double sc, double c,
                                           double s, Xform& x, int lane) {
  __syncwarp();
  if (lane < 12) {
    const int r = lane >> 2, k = lane & 3;
    if (k < 3) {
      const double R0 = k == 0 ? c : (k == 1 ? 0.0 : s), R1 = k == 1 ? 1.0 : 0.0, R2 = k == 0 ? -s : (k == 1 ? 0.0 : c);
      const double a = V[4 * r + 0] * R0 + V[4 * r + 1] * R1 + V[4 * r + 2] * R2;
      x.MV[4 * r + k] = (float)(a * sc);
      x.N[3 * r + k] = (float)(sc == 1.0 ? a : a / sc);   // x / 1.0 == x exactly
    } else {
      x.MV[4 * r + 3] = (float)(V[4 * r + 0] * tx + V[4 * r + 1] * ty + V[4 * r + 2] * tz + V[4 * r + 3]);
    }
  }
  __syncwarp();
}

// fixed-function transform & lighting of one vertex (float32, operation order = spec)
__device__ __forceinline__ Vtx shade_vertex(const Xform& x, const Shared& sh, float px, float py, float pz, float nx,
                                           float ny, float nz, float cr, float cg, float cb, float u, float v) {
  float e[3], ne[3];
#pragma unroll
  for (int r = 0; r < 3; r++) {
    float t = x.MV[4 * r] * px;
    t = t + x.MV[4 * r + 1] * py;
    t = t + x.MV[4 * r + 2] * pz;
    e[r] = t + x.MV[4 * r + 3];
    float q = x.N[3 * r] * nx;
    q = q + x.N[3 * r + 1] * ny;
    ne[r] = q + x.N[3 * r + 2] * nz;
  }
  const float* lp = sh.ep.light_eye;
  float lx, ly, lz;
  if (lp[3] == 0.0f) { lx = lp[0]; ly = lp[1]; lz = lp[2]; }
  else { lx = lp[0] - e[0]; ly = lp[1] - e[1]; lz = lp[2] - e[2]; }
  float len = lx * lx;
  len = len + ly * ly;
  len = len + lz * lz;
  len = sqrtf(len);
  float ndl = 0.0f;
  if (len > 0.0f) {
    lx = lx / len; ly = ly / len; lz = lz / len;
    ndl = ne[0] * lx;
    ndl = ndl + ne[1] * ly;
    ndl = ndl + ne[2] * lz;
    if (!(ndl > 0.0f)) ndl = 0.0f;
  }
  Vtx o;
  const float col[3] = {cr, cg, cb};
  float lit[3];
#pragma unroll
  for (int k = 0; k < 3; k++) {
    float s = 0.3f + sh.ep.ambient[k];
    s = s + ndl * sh.ep.diffuse[k];
    const float c = sh.unlit ? col[k] : col[k] * s;
    lit[k] = c < 0.0f ? 0.0f : (c > 1.0f ? 1.0f : c);
  }
  o.r = lit[0]; o.g = lit[1]; o.b = lit[2];
  o.u = u; o.v = v;
  o.cx = sh.P00 * e[0];
  o.cy = sh.P11 * e[1];
  o.cz = sh.P22 * e[2] + sh.P23;
  o.cw = -e[2];
  return o;
}

__device__ __forceinline__ float plane_dist(const Vtx& a, int pl) {
  switch (pl) {
    case 0: return a.cz + a.cw;
    case 1: return a.cw - a.cz;
    case 2: return a.cx + kGuard * a.cw;
    case 3: return kGuard * a.cw - a.cx;
    case 4: return a.cy + kGuard * a.cw;
    default: return kGuard * a.cw - a.cy;
  }
}

// 0 = visible without clipping, 1 = needs the clipper, 2 = invisible (outside one true-frustum plane)
__device__ __forceinline__ int classify(const Vtx& a, const Vtx& b, const Vtx& c) {
  const Vtx* v[3] = {&a, &b, &c};
  int out[6] = {0, 0, 0, 0, 0, 0}, need = 0;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const float x = v[k]->cx, y = v[k]->cy, z = v[k]->cz, w = v[k]->cw;
    out[0] += !(z + w >= 0.0f); out[1] += !(w - z >= 0.0f);
    out[2] += x < -w; out[3] += x > w; out[4] += y < -w; out[5] += y > w;
    need |= !(x + kGuard * w >= 0.0f) | !(kGuard * w - x >= 0.0f) | !(y + kGuard * w >= 0.0f) |
            !(kGuard * w - y >= 0.0f);
  }
  need |= out[0] | out[1];
#pragma unroll
  for (int p = 0; p < 6; p++) if (out[p] == 3) return 2;
  return need ? 1 : 0;
}

struct EmitCtx {
  const DTexture* textures;
  GeoWarp* gw;
  FrameCtx* ctx;
  PrimRec* prims;          // this env's slab
  int max_prims, W, H;
};

// screen mapping + triangle setup (spec steps 5-7) and append to the slab
// With `d` the prim is the QUAD a,b,c,d (spec tile mode 1: an unclipped road tile): planes of triangle (a,b,c),
// coverage by four edges.  Returns false — nothing emitted — if the snapped quad is not strictly convex; the
// caller then draws the two triangles (a,b,c)(a,c,d) instead.
// Out of line, while shade_vertex and the clipper are inlined: k_geometry is instruction-fetch bound (ncu: 6.9
// stall_no_instruction cycles per issue, 174 KB of SASS against a 32 KB L1.5 I-cache), and inlined, setup_and_emit alone
// is 107 KB in a dozen copies.  Measured k_geometry at c2 / c3 for each choice of inlined functions: all three 198 / 466 us,
// shade_vertex + clipper (this) 177 / 424 us, shade_vertex 188 / 435, shade_vertex + setup_and_emit 220 / 493, none 221 / 447.
__device__ __noinline__ bool setup_and_emit(const EmitCtx& ec, const Vtx& a, const Vtx& b, const Vtx& c, int id,
                                            int tex, int lat, const Vtx* d = nullptr) {
  const Vtx* vs[3] = {&a, &b, &c};
  int X[3], Y[3];
  float zw[3], q[3];
  const float Wf = (float)ec.W, Hf = (float)ec.H;
#pragma unroll
  for (int k = 0; k < 3; k++) {
    const float iw = 1.0f / vs[k]->cw;
    const float nx = vs[k]->cx * iw, ny = vs[k]->cy * iw, nz = vs[k]->cz * iw;
    const float sx = (nx * 0.5f + 0.5f) * Wf;
    const float sy = (0.5f - ny * 0.5f) * Hf;
    X[k] = (int)rintf(sx * 64.0f);
    Y[k] = (int)rintf(sy * 64.0f);
    zw[k] = nz * 0.5f + 0.5f;
    q[k] = iw;
  }
  const long long area2 = (long long)(X[1] - X[0]) * (Y[2] - Y[0]) - (long long)(X[2] - X[0]) * (Y[1] - Y[0]);
  if (area2 == 0) return false;
  const int i1 = area2 < 0 ? 2 : 1, i2 = area2 < 0 ? 1 : 2;
  const int x0 = X[0], y0 = Y[0], x1 = X[i1], y1 = Y[i1], x2 = X[i2], y2 = Y[i2];
  int minx = min(x0, min(x1, x2)), maxx = max(x0, max(x1, x2));
  int miny = min(y0, min(y1, y2)), maxy = max(y0, max(y1, y2));
  int qx[4] = {x0, x1, x2, 0}, qy[4] = {y0, y1, y2, 0};   // quad: cyclic order with positive orientation
  if (d) {
    const float iw = 1.0f / d->cw;
    const float sx = ((d->cx * iw) * 0.5f + 0.5f) * Wf, sy = (0.5f - (d->cy * iw) * 0.5f) * Hf;
    const int X3 = (int)rintf(sx * 64.0f), Y3 = (int)rintf(sy * 64.0f);
    if (area2 > 0) { qx[1] = X[1]; qy[1] = Y[1]; qx[2] = X[2]; qy[2] = Y[2]; qx[3] = X3; qy[3] = Y3; }       // a b c d
    else { qx[1] = X3; qy[1] = Y3; qx[2] = X[2]; qy[2] = Y[2]; qx[3] = X[1]; qy[3] = Y[1]; }                 // a d c b
#pragma unroll
    for (int k = 0; k < 4; k++) {   // strictly convex: every corner turns the same (positive) way
      const int k1 = (k + 1) & 3, k2 = (k + 2) & 3;
      const long long cr = (long long)(qx[k1] - qx[k]) * (qy[k2] - qy[k1]) - (long long)(qx[k2] - qx[k1]) * (qy[k1] - qy[k]);
      if (cr <= 0) return false;
    }
    minx = min(minx, X3); maxx = max(maxx, X3); miny = min(miny, Y3); maxy = max(maxy, Y3);
  }
  const int px0 = max(minx >> 6, 0), px1 = min(maxx >> 6, ec.W - 1);
  const int py0 = max(miny >> 6, 0), py1 = min(maxy >> 6, ec.H - 1);
  if (px0 > px1 || py0 > py1) return true;   // off screen: emitted nothing, and nothing is what it covers
  if (!d && (maxx >> 6) - (minx >> 6) < 3 && (maxy >> 6) - (miny >> 6) < 3) {   // (the unclamped box: everything below stays small)
    // A small triangle that covers NO sample position draws nothing — half the triangles of a distant mesh at
    // 160x120 — so it needs no record, no bin pair and no visit by the rasteriser.  Same integer edge functions and
    // fill rule as the coverage test proper (build_binrec / k_raster); coordinates relative to vertex 0 stay in int32.
    const int ex[3] = {x1 - x0, x2 - x1, x0 - x2}, ey[3] = {y1 - y0, y2 - y1, y0 - y2};
    const int ax[3] = {0, x1 - x0, x2 - x0}, ay[3] = {0, y1 - y0, y2 - y0};
    int e00[3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
      const int bias = (ey[k] > 0 || (ey[k] == 0 && ex[k] < 0)) ? 0 : 1;
      e00[k] = ex[k] * (py0 * kSub - y0 - ay[k]) - ey[k] * (px0 * kSub - x0 - ax[k]) - bias;
    }
    bool any = false;
    for (int py = 0; py <= py1 - py0; py++)
      for (int px = 0; px <= px1 - px0; px++) {
#pragma unroll
        for (int s = 0; s < 4; s++) {
          const int sx = px * kSub + sample_x(s), sy = py * kSub + sample_y(s);
          const int e0 = e00[0] + ex[0] * sy - ey[0] * sx, e1 = e00[1] + ex[1] * sy - ey[1] * sx, e2 = e00[2] + ex[2] * sy - ey[2] * sx;
          any |= (e0 | e1 | e2) >= 0;
        }
      }
    if (!any) return true;
  }
  PrimRec r;
  r.X0 = x0; r.Y0 = y0; r.X1 = x1; r.Y1 = y1; r.X2 = x2; r.Y2 = y2; r.X3 = x0; r.Y3 = y0;
  const float dx1 = (float)(x1 - x0) * 0.015625f, dy1 = (float)(y1 - y0) * 0.015625f;
  const float dx2 = (float)(x2 - x0) * 0.015625f, dy2 = (float)(y2 - y0) * 0.015625f;
  const float areaf = dx1 * dy2 - dx2 * dy1;
  const float ia = 1.0f / areaf;
  const Vtx* p0 = vs[0]; const Vtx* p1 = vs[i1]; const Vtx* p2 = vs[i2];
  const float q0 = q[0], q1 = q[i1], q2 = q[i2];
  const float v0[7] = {zw[0], q0, p0->u * q0, p0->v * q0, p0->r * q0, p0->g * q0, p0->b * q0};
  const float v1[7] = {zw[i1], q1, p1->u * q1, p1->v * q1, p1->r * q1, p1->g * q1, p1->b * q1};
  const float v2[7] = {zw[i2], q2, p2->u * q2, p2->v * q2, p2->r * q2, p2->g * q2, p2->b * q2};
  float f0[7], fx[7], fy[7];
#pragma unroll
  for (int at = 0; at < 7; at++) {
    const float d1 = v1[at] - v0[at], d2 = v2[at] - v0[at];
    f0[at] = v0[at];
    fx[at] = (d1 * dy2 - d2 * dy1) * ia;
    fy[at] = (d2 * dx1 - d1 * dx2) * ia;
  }
  r.z0 = f0[0]; r.zx = fx[0]; r.zy = fy[0];
  r.q0 = f0[1]; r.qx = fx[1]; r.qy = fy[1];
  r.u0 = f0[2]; r.ux = fx[2]; r.uy = fy[2];
  r.v0 = f0[3]; r.vx = fx[3]; r.vy = fy[3];
  r.r0 = f0[4]; r.rx = fx[4]; r.ry = fy[4];
  r.g0 = f0[5]; r.gx = fx[5]; r.gy = fy[5];
  r.b0 = f0[6]; r.bx = fx[6]; r.by = fy[6];
  r.id = id;
  r.ltq = (lat + 1) | ((tex + 1) << 16);
  r.tex = tex >= 0 ? ec.textures[tex].info : 0u;
  (void)px0; (void)py0; (void)px1; (void)py1;
  if (d) {   // vertices in cyclic order; planes stay those of triangle (a,b,c) anchored at a
    r.ltq |= 1 << 24;
    r.X1 = qx[1]; r.Y1 = qy[1]; r.X2 = qx[2]; r.Y2 = qy[2]; r.X3 = qx[3]; r.Y3 = qy[3];
  }
  const int slot = atomicAdd(&ec.ctx->n_prims, 1);
  if (slot >= ec.max_prims) { ec.ctx->overflow = 1; return true; }
  const int4* src = reinterpret_cast<const int4*>(&r);
  int4* dst = reinterpret_cast<int4*>(ec.prims + slot);
#pragma unroll
  for (int k = 0; k < 8; k++) dst[k] = src[k];
  return true;
}

__device__ __forceinline__ Vtx clip_lerp(const Vtx& in, const Vtx& out, float din, float dout) {
  const float t = din / (din - dout);
  Vtx o;
  const float* a = reinterpret_cast<const float*>(&in);
  const float* b = reinterpret_cast<const float*>(&out);
  float* c = reinterpret_cast<float*>(&o);
#pragma unroll
  for (int k = 0; k < 9; k++) { const float d = b[k] - a[k]; c[k] = a[k] + t * d; }
  return o;
}

// Sutherland-Hodgman against near, far and the guard band (spec step 4), then a triangle fan — executed by the
// WHOLE warp for one triangle: lane k owns polygon vertex k, neighbours' plane distances come by shuffle, output
// slots by ballot prefix sums, so a plane costs a few dozen instructions instead of a serial loop over vertices.
// Same arithmetic, same vertex order (hence the same fan) as the serial formulation of the spec.
__device__ __forceinline__ void clip_and_emit_warp(const EmitCtx& ec, const Vtx& a, const Vtx& b, const Vtx& c, int id,
                                                   int tex, int lat, int lane) {
  for (int p2 = 0; p2 < 6; p2++) {   // the spec's trivial reject looks at the ORIGINAL triangle, guard planes
    const int cnt = !(plane_dist(a, p2) >= 0.0f) + !(plane_dist(b, p2) >= 0.0f) + !(plane_dist(c, p2) >= 0.0f);
    if (cnt == 3) return;
  }
  GeoWarp& g = *ec.gw;
  __syncwarp();
  if (lane == 0) { g.poly[0][0] = a; g.poly[0][1] = b; g.poly[0][2] = c; }
  __syncwarp();
  int n = 3, cur = 0;
  for (int pl = 0; pl < 6; pl++) {
    const Vtx* P = g.poly[cur];
    const float dk = lane < n ? plane_dist(P[lane], pl) : 0.0f;
    const bool in1 = dk >= 0.0f;
    const unsigned valid = (1u << n) - 1u;
    const unsigned out_mask = __ballot_sync(0xffffffffu, lane < n && !in1);
    if (!out_mask) continue;
    const int k2 = (lane + 1 == n) ? 0 : lane + 1;
    const float dn = __shfl_sync(0xffffffffu, dk, k2 & 31);
    const bool in2 = dn >= 0.0f;
    const bool cross = lane < n && (in1 != in2);
    const unsigned keep_mask = __ballot_sync(0xffffffffu, lane < n && in1) & valid;
    const unsigned cross_mask = __ballot_sync(0xffffffffu, cross) & valid;
    const unsigned below = (1u << lane) - 1u;
    int pos = __popc(keep_mask & below) + __popc(cross_mask & below);
    Vtx* T = g.poly[cur ^ 1];
    if (lane < n) {
      if (in1) T[pos++] = P[lane];
      if (in1 && !in2) T[pos] = clip_lerp(P[lane], P[k2], dk, dn);
      else if (!in1 && in2) T[pos] = clip_lerp(P[k2], P[lane], dn, dk);
    }
    n = __popc(keep_mask) + __popc(cross_mask);
    cur ^= 1;
    __syncwarp();
    if (n < 3) return;
  }
  const Vtx* P = g.poly[cur];
  if (lane + 2 < n) setup_and_emit(ec, P[0], P[lane + 1], P[lane + 2], id, tex, lat);
  __syncwarp();
}

// one warp-uniform triangle (ground, analytic tile): classify once, lane 0 emits or the warp clips
__device__ __forceinline__ void process_triangle_uniform(const EmitCtx& ec, const Vtx& a, const Vtx& b, const Vtx& c,
                                                         int id, int tex, int lat, int lane) {
  const int cls = classify(a, b, c);
  if (cls == 2) return;
  if (cls == 0) { if (lane == 0) setup_and_emit(ec, a, b, c, id, tex, lat); }
  else clip_and_emit_warp(ec, a, b, c, id, tex, lat, lane);
}

// one triangle per lane (meshes, tessellated tiles): unclipped ones are emitted in place, the rare ones that
// need clipping are broadcast lane by lane to the warp-parallel clipper
__device__ __forceinline__ void process_triangle_lanes(const EmitCtx& ec, bool have, const Vtx& a, const Vtx& b,
                                                       const Vtx& c, int id, int tex, int lat, int lane) {
  const int cls = have ? classify(a, b, c) : 2;
  if (cls == 0) setup_and_emit(ec, a, b, c, id, tex, lat);
  unsigned need = __ballot_sync(0xffffffffu, cls == 1);
  while (need) {
    const int src = __ffs(need) - 1;
    need &= need - 1;
    Vtx va, vb, vc;
    const float* fa = reinterpret_cast<const float*>(&a);
    const float* fb = reinterpret_cast<const float*>(&b);
    const float* fc = reinterpret_cast<const float*>(&c);
#pragma unroll
    for (int k = 0; k < 9; k++) {
      reinterpret_cast<float*>(&va)[k] = __shfl_sync(0xffffffffu, fa[k], src);
      reinterpret_cast<float*>(&vb)[k] = __shfl_sync(0xffffffffu, fb[k], src);
      reinterpret_cast<float*>(&vc)[k] = __shfl_sync(0xffffffffu, fc[k], src);
    }
    const int sid = __shfl_sync(0xffffffffu, id, src), stex = __shfl_sync(0xffffffffu, tex, src);
    clip_and_emit_warp(ec, va, vb, vc, sid, stex, lat, lane);
  }
}

// conservative prim / box overlap: false only if one edge has every sample position of the box
// [x_lo, x_hi] x [y_lo, y_hi] (sub-pixels) on its outside
__device__ __forceinline__ bool box_overlaps(const int qx[4], const int qy[4], int n, int x_lo, int x_hi, int y_lo, int y_hi) {
#pragma unroll
  for (int k = 0; k < 4; k++) {
    if (k >= n) break;
    const int k1 = (k + 1) & 3;   // a triangle's vertex 3 aliases vertex 0
    const int dx = qx[k1] - qx[k], dy = qy[k1] - qy[k];
    // E(x,y) = dx*(y-ay) - dy*(x-ax); maximise over the box
    const int xs = (-dy > 0) ? x_hi : x_lo;
    const int ys = (dx > 0) ? y_hi : y_lo;
    const long long e = (long long)dx * (ys - qy[k]) - (long long)dy * (xs - qx[k]);
    if (e < 0) return false;
  }
  return true;
}
__device__ __forceinline__ bool bin_overlaps(const int qx[4], const int qy[4], int n, int ox, int oy) {
  return box_overlaps(qx, qy, n, ox + 8, ox + (kCoarseW - 1) * kSub + 56, oy + 8, oy + (kCoarseH - 1) * kSub + 56);
}

// The visibility record of prim `p` for the coarse bin whose corner is (ox, oy) sub-pixels: edge functions re-based
// to the corner (exact in 64 bits, then int32: inside the coarse bin |A*x + B*y| < 2^30), exact reject /
// trivial-accept bits for each of the bin's 8 fine bins, depth plane, draw id.
// With `fb` (fused fisheye) the bin's pixels are wherever the LUT sends its output pixels: (ox, oy) is the corner of
// their source bounding box and fb[f] the source box of fine bin f; the bits then speak about every pixel of that box.
// Returns the fine bins every sample of which the prim covers (bits 0-7) | ground quad << 8.
__device__ __forceinline__ unsigned build_binrec(const PrimRec* __restrict__ pr, int p, int ox, int oy, BinRec* __restrict__ out,
                                                 const short4* __restrict__ fb = nullptr) {
  const int4 w0 = __ldg(reinterpret_cast<const int4*>(pr));
  const int4 w1 = __ldg(reinterpret_cast<const int4*>(pr) + 1);
  const float4 w2 = __ldg(reinterpret_cast<const float4*>(pr) + 2);
  const int ltq = __ldg(&pr->ltq);
  const int quad = (ltq >> 24) & 1;
  const int flat = (ltq & 0xffff) ? 8 : 0;   // a road tile of tile mode 1 (it carries a lattice): lies in the plane y = 0
  const int qx[4] = {w0.x, w0.z, w1.x, w1.z}, qy[4] = {w0.y, w0.w, w1.y, w1.w};
  const int nv = quad ? 4 : 3;
  unsigned live = 0xffu, inside = 0xffu;
  int E0[4] = {0, 0, 0, 0}, A[4] = {0, 0, 0, 0}, B[4] = {0, 0, 0, 0};   // triangles: a fourth edge that every sample passes
#pragma unroll
  for (int k = 0; k < 4; k++) {
    if (k >= nv) break;
    const int ka = k, kb = (k + 1) & 3;   // edge k: vertex k -> k+1 (a triangle's vertex 3 is a copy of vertex 0)
    const int dx = qx[kb] - qx[ka], dy = qy[kb] - qy[ka];
    const int bias = (dy > 0 || (dy == 0 && dx < 0)) ? 0 : 1;
    long long e0 = (long long)dx * (oy - qy[ka]) - (long long)dy * (ox - qx[ka]) - bias;
    if (e0 < -(1LL << 30)) live = 0;          // negative for every sample of the coarse bin
    if (e0 > (1LL << 30)) e0 = (1LL << 30);   // positive for every sample: keep the sign, stay in int32
    if (e0 < -(1LL << 30)) e0 = -(1LL << 30);
    const int a = -dy, b = dx, e = (int)e0;
    E0[k] = e; A[k] = a; B[k] = b;
    if (fb) {
      // (fisheye: the fine bins' source boxes are handled after the edge loop, one box load per fine bin)
    } else {
      // extremes of A*x + B*y over one fine bin's sample span x in [8, 504], y in [8, 248]
      const int hi = (a > 0 ? a * 504 : a * 8) + (b > 0 ? b * 248 : b * 8);
      const int lo = (a > 0 ? a * 8 : a * 504) + (b > 0 ? b * 8 : b * 248);
#pragma unroll
      for (int f = 0; f < 8; f++) {
        const int ef = e + a * ((f & 3) * kBinW * kSub) + b * ((f >> 2) * kBinH * kSub);
        if (ef + hi < 0) live &= ~(1u << f);
        if (ef + lo < 0) inside &= ~(1u << f);
      }
    }
  }
  if (fb) {
#pragma unroll 1
    for (int f = 0; f < 8; f++) {
      const short4 q = fb[f];
      if (q.z < q.x) { live &= ~(1u << f); continue; }   // no pixel of this fine bin has a source inside the image
      const int X0 = q.x * kSub - ox + 8, X1 = q.z * kSub - ox + 56, Y0 = q.y * kSub - oy + 8, Y1 = q.w * kSub - oy + 56;
#pragma unroll
      for (int k = 0; k < 4; k++) {
        if (k >= nv) break;
        const int a = A[k], b = B[k], e = E0[k];
        const int hi = (a > 0 ? a * X1 : a * X0) + (b > 0 ? b * Y1 : b * Y0);
        const int lo = (a > 0 ? a * X0 : a * X1) + (b > 0 ? b * Y0 : b * Y1);
        if (e + hi < 0) live &= ~(1u << f);
        if (e + lo < 0) inside &= ~(1u << f);
      }
    }
  }
  int tiny = 0;
  if (!fb && !quad && live) {
    // small triangles (a 6 cm duckie is 148 triangles in a dozen pixels) are rasterised one per LANE in k_raster instead
    // of one per warp: they carry their pixel box
    const int minx = min(qx[0], min(qx[1], qx[2])) - ox, maxx = max(qx[0], max(qx[1], qx[2])) - ox;
    const int miny = min(qy[0], min(qy[1], qy[2])) - oy, maxy = max(qy[0], max(qy[1], qy[2])) - oy;
    const int x0 = max(minx >> 6, 0), x1 = min(maxx >> 6, kCoarseW - 1), y0 = max(miny >> 6, 0), y1 = min(maxy >> 6, kCoarseH - 1);
    if (x1 - x0 < 4 && y1 - y0 < 4 && x1 >= x0 && y1 >= y0) {
      tiny = 4;
      E0[3] = x0 | (y0 << 16); A[3] = x1 | (y1 << 16);
    }
  }
  const int id = __float_as_int(w2.w);
  int4* o = reinterpret_cast<int4*>(out);
  o[0] = make_int4(E0[0], E0[1], E0[2], E0[3]);
  o[1] = make_int4(A[0], A[1], A[2], A[3]);
  o[2] = make_int4(B[0], B[1], B[2], B[3]);
  o[3] = make_int4(__float_as_int(w2.x), __float_as_int(w2.y), __float_as_int(w2.z), id);
  o[4] = make_int4(qx[0] - ox, qy[0] - oy, (int)((unsigned)p | (live << 16) | ((inside & live) << 24)), quad | (id < 2 ? 2 : 0) | tiny | flat);
  return (inside & live) | (id < 2 ? 0x100u : 0u);
}

// Fragment colour of prim `w` of the env's slab at the pixel whose centre is (pxa + 32, pya + 32) sub-pixels (spec steps
// 5-6 and 8): perspective-correct u,v (+ rgb for meshes / ground), analytic lattice lighting for road tiles,
// bilinear REPEAT texel, MODULATE.  Deferred shading: each lane may shade a different prim.  Split in two so that a
// coarse bin lying inside ONE prim fetches the prim's planes once for its 256 pixels.
struct ShadeIn {
  const PrimRec* pr;
  int x0, y0;
  float q0, qx, qy, u0, ux, uy, v0, vx, vy, r0;
  int ltq;
  unsigned tex;
};
__device__ __forceinline__ ShadeIn load_shade(const PrimRec* __restrict__ prims, unsigned w) {
  const PrimRec* pr = prims + w;
  const int2 xy0 = __ldg(reinterpret_cast<const int2*>(pr));
  const float4 w3 = __ldg(reinterpret_cast<const float4*>(pr) + 3);   // q0 qx qy u0
  const float4 w4 = __ldg(reinterpret_cast<const float4*>(pr) + 4);   // ux uy v0 vx
  const float4 w5 = __ldg(reinterpret_cast<const float4*>(pr) + 5);   // vy ltq tex r0
  ShadeIn si;
  si.pr = pr; si.x0 = xy0.x; si.y0 = xy0.y;
  si.q0 = w3.x; si.qx = w3.y; si.qy = w3.z; si.u0 = w3.w;
  si.ux = w4.x; si.uy = w4.y; si.v0 = w4.z; si.vx = w4.w;
  si.vy = w5.x; si.ltq = __float_as_int(w5.y); si.tex = __float_as_uint(w5.z); si.r0 = w5.w;
  return si;
}
__device__ __forceinline__ void shade_eval(const ShadeIn& si, const uint8_t* __restrict__ tex_pool, const float4* __restrict__ lat_tab,
                                           int pxa, int pya, float c3[3]) {
  const float cdx = (float)(pxa + 32 - si.x0) * 0.015625f, cdy = (float)(pya + 32 - si.y0) * 0.015625f;
  float qq = fmaf(si.qy, cdy, fmaf(si.qx, cdx, si.q0));
  if (!(qq > 1e-20f)) qq = 1e-20f;
  const float rq = 1.0f / qq;
  const float u = fmaf(si.uy, cdy, fmaf(si.ux, cdx, si.u0)) * rq;
  const float v = fmaf(si.vy, cdy, fmaf(si.vx, cdx, si.v0)) * rq;
  const int ltq = si.ltq;
  const int lat = (ltq & 0xffff) - 1;
  if (lat >= 0) {
    // analytic road tile: Gouraud interpolant of the lit 8x8 lattice at (u,v)
    const float fa_ = u * 7.0f, fb_ = (1.0f - v) * 7.0f;
    int ia = __float2int_rd(fa_), ib = __float2int_rd(fb_);   // (int)floorf(.)
    ia = ia < 0 ? 0 : (ia > 6 ? 6 : ia);
    ib = ib < 0 ? 0 : (ib > 6 ? 6 : ib);
    const float fa = fa_ - (float)ia, fb = fb_ - (float)ib;
    const float4* L = lat_tab + lat * 64 + ia * 8 + ib;
    // the cell's two triangles share c00 and c11; pick the third corner and the order of the two weights
    // instead of branching (same arithmetic, three loads instead of four)
    const bool lower = fb <= fa;
    const float4 c00 = L[0], c11 = L[9], cm = L[lower ? 8 : 1];
    const float t1 = lower ? fa : fb, t2 = lower ? fb : fa;
    c3[0] = fmaf(t2, c11.x - cm.x, fmaf(t1, cm.x - c00.x, c00.x));
    c3[1] = fmaf(t2, c11.y - cm.y, fmaf(t1, cm.y - c00.y, c00.y));
    c3[2] = fmaf(t2, c11.z - cm.z, fmaf(t1, cm.z - c00.z, c00.z));
  } else {
    const float4 w6 = __ldg(reinterpret_cast<const float4*>(si.pr) + 6);    // rx ry g0 gx
    const float4 w7 = __ldg(reinterpret_cast<const float4*>(si.pr) + 7);    // gy b0 bx by
    c3[0] = fmaf(w6.y, cdy, fmaf(w6.x, cdx, si.r0)) * rq;
    c3[1] = fmaf(w7.x, cdy, fmaf(w6.w, cdx, w6.z)) * rq;
    c3[2] = fmaf(w7.w, cdy, fmaf(w7.z, cdx, w7.y)) * rq;
  }
  if (ltq & 0x00ff0000) {
    const unsigned ti = si.tex;
    const int lw = (ti >> 24) & 15, lh = ti >> 28;
    const int tw = 1 << lw, th = 1 << lh;
    const float twf = __int_as_float((127 + lw) << 23), thf = __int_as_float((127 + lh) << 23);   // (float)tw: a power of two
    const float tx = u * twf - 0.5f, ty = v * thf - 0.5f;
    const int txi = __float2int_rd(tx), tyi = __float2int_rd(ty);   // floorf(.) as the int the wrap needs; exact back in float
    const float ffx = tx - (float)txi, ffy = ty - (float)tyi;
    const int ti0 = txi & (tw - 1), ti1 = (ti0 + 1) & (tw - 1);
    const int tj0 = tyi & (th - 1), tj1 = (tj0 + 1) & (th - 1);
    const uchar4* tp = reinterpret_cast<const uchar4*>(tex_pool + ((size_t)(ti & 0xffffffu) << 8));
    const uchar4 t00 = __ldg(tp + (tj0 << lw) + ti0), t10 = __ldg(tp + (tj0 << lw) + ti1);
    const uchar4 t01 = __ldg(tp + (tj1 << lw) + ti0), t11 = __ldg(tp + (tj1 << lw) + ti1);
    const float a0[3] = {(float)t00.x, (float)t00.y, (float)t00.z}, a1[3] = {(float)t10.x, (float)t10.y, (float)t10.z};
    const float b0[3] = {(float)t01.x, (float)t01.y, (float)t01.z}, b1[3] = {(float)t11.x, (float)t11.y, (float)t11.z};
#pragma unroll
    for (int ch = 0; ch < 3; ch++) {
      const float ta = fmaf(ffx, a1[ch] - a0[ch], a0[ch]);
      const float tb = fmaf(ffx, b1[ch] - b0[ch], b0[ch]);
      const float tc = fmaf(ffy, tb - ta, ta);
      c3[ch] = tc * (c3[ch] * 0.00392156862745098f);
    }
  }
}
__device__ __forceinline__ void shade_prim(const PrimRec* __restrict__ prims, unsigned w, const uint8_t* __restrict__ tex_pool,
                                           const float4* __restrict__ lat_tab, int pxa, int pya, float c3[3]) {
  const ShadeIn si = load_shade(prims, w);
  shade_eval(si, tex_pool, lat_tab, pxa, pya, c3);
}

// ---- bulk-async copy (TMA, 1-D) + mbarrier: global -> shared without register staging
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok)
                 : "r"(smem_u32(bar)), "r"(parity)
                 : "memory");
  } while (!ok);
}

// u8 = rint(255 * clamp(c)) packed r | g<<8 | b<<16 (resolve of 4 equal samples is the value itself).  The
// float->unsigned conversion rounds to nearest-even and saturates below at 0 (NaN -> 0), min() saturates above:
// identical to clamping c to [0, 1] first.
__device__ __forceinline__ unsigned pack_rgb(float r, float g, float b) {
  const unsigned ur = min(__float2uint_rn(r * 255.0f), 255u);
  const unsigned ug = min(__float2uint_rn(g * 255.0f), 255u);
  const unsigned ub = min(__float2uint_rn(b * 255.0f), 255u);
  return ur | (ug << 8) | (ub << 16);
}

// one 8x4 bin of packed pixels -> global memory: rows of 24 bytes as 6 aligned words built with shuffles.
// The lane-constant parts (shuffle sources, shift, byte offset inside a bin) are computed once per kernel (StoreLane).
struct StoreLane {
  int src_lo, src_hi;   // lanes holding the two pixels this lane's output word straddles
  int sh8;              // bit offset of the word inside lo | hi << 24
  int off;              // byte offset of the word from the bin's first byte: (lane >> 3) * W * 3 + 4 * (lane & 7)
  int j, row;           // word index in the row (only 0..5 store), row inside the bin
};
__device__ __forceinline__ StoreLane make_store_lane(int lane, int W) {
  StoreLane sl;
  const int j = lane & 7, rowbase = lane & ~7;
  const int p0 = (4 * j) / 3;
  sl.sh8 = (4 * j - 3 * p0) * 8;
  sl.src_lo = rowbase + min(p0, 7);
  sl.src_hi = rowbase + min(p0 + 1, 7);
  sl.off = (lane >> 3) * W * 3 + 4 * j;
  sl.j = j; sl.row = lane >> 3;
  return sl;
}
// `bin0` = address of the bin's first byte (warp-uniform); rows_ok = how many of the bin's 4 rows are inside the image
__device__ __forceinline__ void store_bin_fast(uint8_t* __restrict__ bin0, const StoreLane& sl, unsigned rgb, int rows_ok) {
  const unsigned lo = __shfl_sync(0xffffffffu, rgb, sl.src_lo);
  const unsigned hi = __shfl_sync(0xffffffffu, rgb, sl.src_hi);
  const unsigned word = __funnelshift_r(lo | (hi << 24), hi >> 8, sl.sh8);   // (lo | hi << 24) >> sh8, low 32 bits
  if (sl.j < 6 && sl.row < rows_ok) *reinterpret_cast<unsigned*>(bin0 + sl.off) = word;
}
// general form (any width, bins cut by the right border)
__device__ __forceinline__ void store_bin(uint8_t* __restrict__ out, unsigned rgb, int lane, int bx, int by, int W, int H) {
  const int gx = bx * kBinW + (lane & 7), gy = by * kBinH + (lane >> 3);
  if ((W & 3) == 0 && bx * kBinW + kBinW <= W) {
    const int j = lane & 7, rowbase = lane & ~7;
    const int p0 = (4 * j) / 3, sh8 = (4 * j - 3 * p0) * 8;
    const unsigned lo = __shfl_sync(0xffffffffu, rgb, rowbase + min(p0, 7));
    const unsigned hi = __shfl_sync(0xffffffffu, rgb, rowbase + min(p0 + 1, 7));
    const unsigned long long both = (unsigned long long)lo | ((unsigned long long)hi << 24);
    if (j < 6 && gy < H)
      *reinterpret_cast<unsigned*>(out + ((size_t)gy * W + bx * kBinW) * 3 + 4 * j) = (unsigned)(both >> sh8);
  } else if (gx < W && gy < H) {
    uint8_t* d = out + ((size_t)gy * W + gx) * 3;
    d[0] = (uint8_t)(rgb & 255); d[1] = (uint8_t)((rgb >> 8) & 255); d[2] = (uint8_t)(rgb >> 16);
  }
}

// One pixel in a wrapper layout / dtype (dts_output_format): element index of channel c at (x, y)
__device__ __forceinline__ size_t fmt_index(int layout, int x, int y, int c, int W, int H) {
  return layout == DTS_OBS_CHW ? ((size_t)c * H + y) * W + x
       : layout == DTS_OBS_CWH ? ((size_t)c * W + x) * H + y
                               : ((size_t)y * W + x) * 3 + c;
}
__device__ __forceinline__ void store_px_fmt(void* frame, int layout, int dtype, int x, int y, int W, int H, unsigned rgb) {
#pragma unroll
  for (int c = 0; c < 3; c++) {
    const unsigned v = (rgb >> (8 * c)) & 255u;
    const size_t i = fmt_index(layout, x, y, c, W, H);
    if (dtype == DTS_OBS_F32_UNIT) reinterpret_cast<float*>(frame)[i] = (float)v / 255.0f;   // NormalizeWrapper LW:66-70
    else reinterpret_cast<uint8_t*>(frame)[i] = (uint8_t)v;
  }
}
// One whole 8x4 bin in a PLANAR u8 layout (ImgWrapper's CHW, PyTorchObsWrapper's CWH) as 24 aligned 32-bit words, one per
// lane: a word is four horizontally (CHW) or vertically (CWH) adjacent pixels of one channel plane, collected from the
// four lanes holding them by shuffles and two byte permutes — instead of three scattered byte stores per lane.
// Needs the bin inside the image and W % 4 == 0 (CHW) / H % 4 == 0 (CWH).
__device__ __forceinline__ void store_bin_planar_u8(uint8_t* __restrict__ out, int layout, unsigned rgb, int lane, int bx, int by,
                                                    int W, int H) {
  const int j = lane < 24 ? lane : 0, c = j >> 3;
  int s0, step;
  size_t addr;
  if (layout == DTS_OBS_CHW) {
    const int r = (j & 7) >> 1, h = j & 1;
    s0 = r * 8 + 4 * h; step = 1;
    addr = ((size_t)c * H + by * kBinH + r) * W + bx * kBinW + 4 * h;
  } else {
    const int xi = j & 7;
    s0 = xi; step = 8;
    addr = ((size_t)c * W + bx * kBinW + xi) * H + by * kBinH;
  }
  const unsigned p0 = __shfl_sync(0xffffffffu, rgb, s0), p1 = __shfl_sync(0xffffffffu, rgb, s0 + step);
  const unsigned p2 = __shfl_sync(0xffffffffu, rgb, s0 + 2 * step), p3 = __shfl_sync(0xffffffffu, rgb, s0 + 3 * step);
  const unsigned sel = (unsigned)c | ((unsigned)(4 + c) << 4);   // byte c of the first operand, byte c of the second
  const unsigned word = __byte_perm(__byte_perm(p0, p1, sel), __byte_perm(p2, p3, sel), 0x5410);
  if (lane < 24) *reinterpret_cast<unsigned*>(out + addr) = word;
}

// Fine-bin store: the packed u8 HWC fast path, or the wrapper format straight from the resolve registers.
__device__ __forceinline__ void store_bin_any(uint8_t* __restrict__ out, int fmt, unsigned rgb, int lane, int bx, int by,
                                              int W, int H) {
  if (fmt == 0) { store_bin(out, rgb, lane, bx, by, W, H); return; }
  const int gx = bx * kBinW + (lane & 7), gy = by * kBinH + (lane >> 3);
  if (gx < W && gy < H) store_px_fmt(out, fmt & 3, fmt >> 2, gx, gy, W, H, rgb);
}

}  // namespace


int render_ctas_per_sm() { return kRenderMinCtas; }

// ------------------------------------------------------------------------------------------------ frame memory
struct FrameMem {
  FrameCtx* ctx;        // [N]
  PrimRec* prims;       // [N][max_prims]
  uint32_t* pairs;      // [pool]  prim | coarse bin << 16, grouped by env and coarse bin (k_bin pass 1).  One pool for the
  BinRec* recs;         // [pool]  batch: an env takes exactly the entries it needs (atomic cursor work[1]), densely packed
  int* bin_count;       // [N][cbins]
  int* bin_start;       // [N][cbins]  pool index of the bin's first pair / record
  float4* lat;          // [N][max_lat][64]
  uint2* geo_list;      // [N * items_max] (env, draw item) pairs that passed k_cull
  uint2* solo;          // [N * cbins] (env, coarse bin | prim << 16): coarse bins lying inside one prim (k_bin -> k_raster_solo)
  int* work;            // global counters: [0] k_raster work items, [1] pair-pool cursor, [2] geo_list length, [3] solo list length
  int32_t* status;      // mapped host word (dts_status): bit 0 = a frame ran out of frame memory
};

__host__ __device__ inline size_t align256(size_t b) { return (b + 255) & ~size_t(255); }

__host__ FrameMem carve(void* scratch, int n, int max_prims, int cbins, int max_pairs, int max_lat, size_t geo_items) {
  uint8_t* p = reinterpret_cast<uint8_t*>(scratch);
  FrameMem f;
  f.work = reinterpret_cast<int*>(p); p += 256;
  f.ctx = reinterpret_cast<FrameCtx*>(p); p += align256((size_t)n * sizeof(FrameCtx));
  f.bin_count = reinterpret_cast<int*>(p); p += align256((size_t)n * cbins * sizeof(int));
  f.bin_start = reinterpret_cast<int*>(p); p += align256((size_t)n * cbins * sizeof(int));
  f.prims = reinterpret_cast<PrimRec*>(p); p += align256((size_t)n * max_prims * sizeof(PrimRec));
  f.pairs = reinterpret_cast<uint32_t*>(p); p += align256((size_t)max_pairs * sizeof(uint32_t));   // max_pairs = pool entries
  f.recs = reinterpret_cast<BinRec*>(p); p += align256((size_t)max_pairs * sizeof(BinRec));
  f.lat = reinterpret_cast<float4*>(p); p += align256((size_t)n * max_lat * 64 * sizeof(float4));
  f.geo_list = reinterpret_cast<uint2*>(p); p += align256((size_t)n * geo_items * sizeof(uint2));
  f.solo = reinterpret_cast<uint2*>(p); p += align256((size_t)n * cbins * sizeof(uint2));
  f.status = nullptr;
  return f;
}

size_t render_scratch_bytes(int n, int max_prims, int cbins, int max_pairs, int max_lat, size_t geo_items) {
  return 256 + align256((size_t)n * sizeof(FrameCtx)) + 2 * align256((size_t)n * cbins * sizeof(int)) +
         align256((size_t)n * max_prims * sizeof(PrimRec)) + align256((size_t)max_pairs * sizeof(uint32_t)) +
         align256((size_t)max_pairs * sizeof(BinRec)) +
         align256((size_t)n * max_lat * 64 * sizeof(float4)) + align256((size_t)n * geo_items * sizeof(uint2)) +
         align256((size_t)n * cbins * sizeof(uint2)) + 256;
}

// ------------------------------------------------------------------------------------------------ k_frame_setup
__global__ void __launch_bounds__(128) k_frame_setup(const DState S, const DMap* __restrict__ maps, RenderCfg rc, FrameMem fm) {
  const int env = blockIdx.x * blockDim.x + threadIdx.x;
  if (env >= rc.n_envs) return;
  FrameCtx& c = fm.ctx[env];
  const RenderEp ep = S.rep[env];
  double V[12];
  if (rc.mode & DTS_RENDER_TOP_DOWN) {
    const DMap& m = maps[S.map_id[env]];
    top_down_view((double)m.grid_w, (double)m.grid_h, m.tile_size, (double)ep.cam_fov_y_deg, V);
  } else {
    camera_view(S.pos_x[env], S.pos_z[env], S.angle[env], ep, (rc.flags & DTS_FLAG_DOMAIN_RAND) != 0, V);
  }
#pragma unroll
  for (int k = 0; k < 12; k++) c.V[k] = V[k];
  const double f = 1.0 / tan((double)ep.cam_fov_y_deg * kDeg2Rad / 2.0), aspect = (double)rc.width / (double)rc.height;
  const double zn = 0.04, zf = 100.0;                                     // gluPerspective S:1761
  c.P00 = (float)(f / aspect); c.P11 = (float)f;
  c.P22 = (float)((zf + zn) / (zn - zf)); c.P23 = (float)(2.0 * zf * zn / (zn - zf));
  c.n_prims = 0; c.n_lat = 0; c.overflow = 0; c.pad = 0;
}

// Conservative bounding-sphere cull in eye space against the four side planes and near: true only if the sphere
// — hence everything inside it — lies outside one plane (margins cover the f32 rounding of the test itself).
__device__ __forceinline__ bool sphere_outside(float P00, float P11, float cx_, float cy_, float cz_, float rad) {
  const float hx = rsqrtf(P00 * P00 + 1.0f), hy = rsqrtf(P11 * P11 + 1.0f);
  bool out = cz_ - rad > -0.04f;                                  // entirely behind the near plane
  out |= (P00 * cx_ + cz_) * hx > rad * 1.01f;                    // right plane: P00*x <= -z
  out |= (-P00 * cx_ + cz_) * hx > rad * 1.01f;
  out |= (P11 * cy_ + cz_) * hy > rad * 1.01f;
  out |= (-P11 * cy_ + cz_) * hy > rad * 1.01f;
  return out;
}
// world point -> eye space with the f64 camera matrix (row-major 3x4)
__device__ __forceinline__ void eye_point(const double* V, double wx, double wy, double wz, float& ex, float& ey, float& ez) {
  ex = (float)(V[0] * wx + V[1] * wy + V[2] * wz + V[3]);
  ey = (float)(V[4] * wx + V[5] * wy + V[6] * wz + V[7]);
  ez = (float)(V[8] * wx + V[9] * wy + V[10] * wz + V[11]);
}

// Does draw item `item` of env `env` need any work this frame?  Conservative bounding-sphere test against the view
// frustum before anything is transformed (most (env, item) pairs end here), plus the values the mesh path needs later:
// the obstacle's per-env pose.  Run once per pair by k_cull (one thread each) and again by the warp that draws the item.
struct ItemPose { int dyn_kind; float opx, opz, orot; bool agent_item; };
__device__ __forceinline__ bool item_visible(const DState& S, const DMap& m, const RenderCfg& rc, const FrameCtx& ctx, int env,
                                             int item, ItemPose& ip) {
  const int n_tiles = m.grid_w * m.grid_h;
  ip.dyn_kind = 0; ip.opx = 0.f; ip.opz = 0.f; ip.orot = 0.f;
  ip.agent_item = item == 1 + n_tiles + m.n_objects;   // top-down views draw the agent's own mesh last (S:1923-1929)
  if (item > 1 + n_tiles + m.n_objects) return false;
  if (ip.agent_item && (!(rc.mode & DTS_RENDER_TOP_DOWN) || m.agent.tri_count == 0)) return false;
  if (item >= 1 && item <= n_tiles) {
    const int t = item - 1, ti = t / m.grid_h, tj = t - ti * m.grid_h;
    if (m.tile_kind[tj * m.grid_w + ti] < 0) return false;
    const double ts = m.tile_size;
    float ex, ey, ez;
    eye_point(ctx.V, (ti + 0.5) * ts, 0.0, (tj + 0.5) * ts, ex, ey, ez);
    if (sphere_outside(ctx.P00, ctx.P11, ex, ey, ez, (float)(ts * 0.7071067811865476) * 1.001f + 1e-4f)) return false;
  } else if (item > n_tiles) {
    const int o = item - 1 - n_tiles;
    if (!ip.agent_item && (S.rep[env].hidden[o >> 5] >> (o & 31) & 1u)) return false;
    const DObject& ob = ip.agent_item ? m.agent : m.objects[o];
    ip.opx = ob.pos[0]; ip.opz = ob.pos[2]; ip.orot = ob.y_rot_deg;
    if (ip.agent_item) {   // glTranslatef(*cur_pos); glRotatef(cur_angle * 180 / pi, 0, 1, 0): GLfloat arguments
      ip.opx = (float)S.pos_x[env]; ip.opz = (float)S.pos_z[env];
      ip.orot = (float)(S.angle[env] * 180.0 / 3.141592653589793);
    }
    if (ob.dyn_slot >= 0) {
      ip.dyn_kind = m.dyn[ob.dyn_slot].kind;
      if (ip.dyn_kind != DTS_DYN_TRAFFICLIGHT) {   // a moving obstacle: this env's pos / y_rot, rounded to float like glTranslatef / glRotatef
        const size_t nd = m.n_dyn, ne = rc.n_envs;
        ip.opx = (float)m.dyn_state[((size_t)DTS_DYN_PX * nd + ob.dyn_slot) * ne + env];
        ip.opz = (float)m.dyn_state[((size_t)DTS_DYN_PZ * nd + ob.dyn_slot) * ne + env];
        ip.orot = (float)m.dyn_state[((size_t)DTS_DYN_YROT * nd + ob.dyn_slot) * ne + env];
      }
    }
    double sn, cs;
    sincos((double)ip.orot * kDeg2Rad, &sn, &cs);
    const double sc = (double)ob.scale, ccx = ob.centre[0], ccy = ob.centre[1], ccz = ob.centre[2];
    float ex, ey, ez;   // T(pos) S(scale) Ry(rot) applied to the bounding-sphere centre
    eye_point(ctx.V, (double)ip.opx + sc * (cs * ccx + sn * ccz), (double)ob.pos[1] + sc * ccy, (double)ip.opz + sc * (-sn * ccx + cs * ccz), ex, ey, ez);
    if (sphere_outside(ctx.P00, ctx.P11, ex, ey, ez, ob.bound_rad * ob.scale * 1.002f + 2e-4f)) return false;
  }
  return true;
}

// ------------------------------------------------------------------------------------------------ k_cull
// thread per (env, draw item), item-major: the pairs that survive item_visible() go to a compact work list (warp-
// aggregated atomic append), so that k_geometry spends warps only on items that will emit something.
__global__ void __launch_bounds__(256) k_cull(const DState S, const DMap* __restrict__ maps, RenderCfg rc, FrameMem fm, int items_max) {
  const size_t g = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  const int item = (int)(g / rc.n_envs), env = (int)(g - (size_t)item * rc.n_envs);
  bool vis = false;
  if (item < items_max) {
    ItemPose ip;
    vis = item_visible(S, maps[S.map_id[env]], rc, fm.ctx[env], env, item, ip);
  }
  const unsigned m = __ballot_sync(0xffffffffu, vis);
  if (!m) return;
  const int lane = threadIdx.x & 31;
  int base = 0;
  if (lane == __ffs(m) - 1) base = atomicAdd(fm.work + 2, __popc(m));
  base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
  if (vis) fm.geo_list[base + __popc(m & ((1u << lane) - 1u))] = make_uint2((unsigned)env, (unsigned)item);
}

// ------------------------------------------------------------------------------------------------ k_geometry
// One warp per CTA, 64 registers, 32 CTAs per SM: the kernel is latency-bound (short dependent chains), so resident warps
// matter more than spills.  Each warp draws the (env, item) pairs of k_cull's work list, grid-strided.
constexpr int kGeoWarps = 1, kGeoMinCtas = 32;
template <bool kTess>   // true: spec tile mode 0 (DTS_FLAG_TESSELLATE), the literal 98 triangles per road tile
__device__ __forceinline__ void geometry_item(const DState& S, const DMap* __restrict__ maps, const RenderCfg& rc, const FrameMem& fm,
                                              int max_prims, int max_lat, int32_t* __restrict__ err, int env, int item, int lane,
                                              GeoWarp& sh) {
  const DMap& m = maps[S.map_id[env]];
  const int n_tiles = m.grid_w * m.grid_h;
  const bool seg = (rc.mode & DTS_RENDER_SEGMENT) != 0;
  const int W = rc.width, H = rc.height;
  FrameCtx& ctx = fm.ctx[env];
  ItemPose ip;
  if (!item_visible(S, m, rc, ctx, env, item, ip)) return;
  const bool agent_item = ip.agent_item;
  const int dyn_kind = ip.dyn_kind;
  const float opx = ip.opx, opz = ip.opz, orot = ip.orot;
  __syncwarp();   // the previous item of this warp is done with the shared GeoWarp
  for (int k = lane; k < (int)(sizeof(RenderEp) / 4); k += 32)
    reinterpret_cast<uint32_t*>(&sh.ep)[k] = reinterpret_cast<const uint32_t*>(&S.rep[env])[k];
  if (lane < 12) sh.V[lane] = ctx.V[lane];
  if (lane == 12) { sh.P00 = ctx.P00; sh.P11 = ctx.P11; sh.P22 = ctx.P22; sh.P23 = ctx.P23; sh.unlit = seg ? 1 : 0; }
  __syncwarp();
  EmitCtx ec{m.textures, &sh, &ctx, fm.prims + (size_t)env * max_prims, max_prims, W, H};
  float4* lat_tab = fm.lat + (size_t)env * max_lat * 64;
  const int tris_per_tile = kTess ? 98 : 2;
  Xform& x = sh.x;
  if (item == 0) {
    // ground quad S:1805-1812: glScalef(50,0.01,50) applied to (+-1,-0.8,+-1), world-space +y normal
    model_view(sh.V, 0.0, 0.0, 0.0, 1.0, 1.0, 0.0, x, lane);
    const float gy = (float)(-0.8 * 0.01);
    const float P[4][3] = {{-50.f, gy, 50.f}, {-50.f, gy, -50.f}, {50.f, gy, -50.f}, {50.f, gy, 50.f}};
    const float magenta[3] = {255.f, 0.f, 255.f};   // glColor3f(255, 0, 255) S:1808: clamped to (1, 0, 1) as a vertex colour
    const float* g = seg ? magenta : sh.ep.ground;
    const int pl_ = lane & 3;   // lanes 0..3 light the four corners, the two triangles (0,1,2)(0,2,3) are then warp-uniform
    const Vtx mine = shade_vertex(x, sh, P[pl_][0], P[pl_][1], P[pl_][2], 0.f, 1.f, 0.f, g[0], g[1], g[2], 0.f, 0.f);
    if (lane < 4) sh.corners[lane] = mine;
    __syncwarp();
    process_triangle_uniform(ec, sh.corners[0], sh.corners[1], sh.corners[2], 0, -1, -1, lane);
    process_triangle_uniform(ec, sh.corners[0], sh.corners[2], sh.corners[3], 1, -1, -1, lane);
  } else if (item <= n_tiles) {
    // road tile S:1852-1884: draw order i outer, j inner
    const int t = item - 1, ti = t / m.grid_h, tj = t - ti * m.grid_h;
    const int idx = tj * m.grid_w + ti;
    const int quarter = (m.tile_angle[idx] + 2) & 3;                     // glRotatef(angle*90+180) S:1873
    const double cs = quarter == 0 ? 1.0 : (quarter == 2 ? -1.0 : 0.0), sn = quarter == 1 ? 1.0 : (quarter == 3 ? -1.0 : 0.0);
    const double ts = m.tile_size;
    // glTranslatef((i + 0.5) * TS, 0, (j + 0.5) * TS) S:1870 takes GLfloat arguments
    model_view(sh.V, (double)(float)((ti + 0.5) * ts), 0.0, (double)(float)((tj + 0.5) * ts), 1.0, cs, sn, x, lane);
    int tex = m.tile_tex[idx];
    if (seg && tex >= 0) tex = m.tex_segment[tex];   // Texture.bind(segment=True) G:52-56
    const int base_id = 2 + tris_per_tile * t;
    if (!kTess) {
      // analytic tile: the prim is the quad of the 4 corners — cull on those before lighting the lattice
      const int ca = (lane == 1 || lane == 2) ? 7 : 0, cb = (lane >= 2) ? 7 : 0;   // lanes 0..3: (0,0) (7,0) (7,7) (0,7)
      const float lx = (float)(-ts / 2 + ((double)ca / 7.0) * ts), lz = (float)(-ts / 2 + ((double)cb / 7.0) * ts);
      const Vtx v = shade_vertex(x, sh, lx, 0.0f, lz, 0.f, 1.f, 0.f, 1.f, 1.f, 1.f, (float)((double)ca / 7.0),
                                 (float)(1.0 - (double)cb / 7.0));
      const unsigned four = 0xFu;
      bool culled4 = false;
      culled4 |= (__ballot_sync(0xffffffffu, !(v.cz + v.cw >= 0.0f)) & four) == four;
      culled4 |= (__ballot_sync(0xffffffffu, !(v.cw - v.cz >= 0.0f)) & four) == four;
      culled4 |= (__ballot_sync(0xffffffffu, v.cx < -v.cw) & four) == four;
      culled4 |= (__ballot_sync(0xffffffffu, v.cx > v.cw) & four) == four;
      culled4 |= (__ballot_sync(0xffffffffu, v.cy < -v.cw) & four) == four;
      culled4 |= (__ballot_sync(0xffffffffu, v.cy > v.cw) & four) == four;
      if (culled4) return;
    }
    // the tile's 8x8 lattice, two vertices per lane (tessellated mode: also frustum-culls the whole tile)
    Vtx lv[2];
    int outside[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int h = 0; h < 2; h++) {
      const int vi = lane + 32 * h, a = vi >> 3, b = vi & 7;             // a: u index (x), b: v index (z)
      const float lx = (float)(-ts / 2 + ((double)a / 7.0) * ts), lz = (float)(-ts / 2 + ((double)b / 7.0) * ts);
      lv[h] = shade_vertex(x, sh, lx, 0.0f, lz, 0.f, 1.f, 0.f, 1.f, 1.f, 1.f, (float)((double)a / 7.0),
                           (float)(1.0 - (double)b / 7.0));
      const Vtx& v = lv[h];
      outside[0] += !(v.cz + v.cw >= 0.0f); outside[1] += !(v.cw - v.cz >= 0.0f);
      outside[2] += v.cx < -v.cw; outside[3] += v.cx > v.cw; outside[4] += v.cy < -v.cw; outside[5] += v.cy > v.cw;
    }
    if (kTess) {
      bool culled = false;
#pragma unroll
      for (int p = 0; p < 6; p++) culled |= __all_sync(0xffffffffu, outside[p] == 2);
      if (culled) return;
    }
    if (!kTess) {
      // analytic tile (spec tile mode 1): lattice colours -> table, one quad (0,1,2)(0,2,3) of the corners
      int slot = 0;
      if (lane == 0) slot = atomicAdd(&ctx.n_lat, 1);
      slot = __shfl_sync(0xffffffffu, slot, 0);
      if (slot >= max_lat) { if (lane == 0) ctx.overflow = 1; return; }
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const int vi = lane + 32 * h;
        lat_tab[slot * 64 + vi] = make_float4(lv[h].r, lv[h].g, lv[h].b, 0.0f);
        int corner = -1;
        if (vi == 0) corner = 0; else if (vi == 56) corner = 1; else if (vi == 63) corner = 2; else if (vi == 7) corner = 3;
        if (corner >= 0) { Vtx c = lv[h]; c.r = 0.f; c.g = 0.f; c.b = 0.f; sh.corners[corner] = c; }
      }
      __syncwarp();
      // a tile that needs no clipping is ONE quad prim (its diagonal then splits no bin); otherwise two triangles
      bool as_quad = false;
      if (classify(sh.corners[0], sh.corners[1], sh.corners[2]) == 0 && classify(sh.corners[0], sh.corners[2], sh.corners[3]) == 0) {
        if (lane == 0) as_quad = setup_and_emit(ec, sh.corners[0], sh.corners[1], sh.corners[2], base_id, tex, slot, &sh.corners[3]);
        as_quad = __shfl_sync(0xffffffffu, (int)as_quad, 0) != 0;
      }
      if (!as_quad) {
        process_triangle_uniform(ec, sh.corners[0], sh.corners[1], sh.corners[2], base_id, tex, slot, lane);
        process_triangle_uniform(ec, sh.corners[0], sh.corners[2], sh.corners[3], base_id + 1, tex, slot, lane);
      }
      } else {
      // literal vertex list S:407-433 (spec tile mode 0): 7x7 quads, (0,1,2)(0,2,3) split, 3 shades / triangle
      for (int k0 = 0; k0 < 98; k0 += 32) {
        const int k = k0 + lane;
        Vtx v[3];
        if (k < 98) {
          const int quad = k >> 1, half = k & 1, a = quad / 7, b = quad - 7 * a;
#pragma unroll
          for (int j = 0; j < 3; j++) {
            const int aa = j == 0 ? a : (j == 1 ? a + 1 : (half == 0 ? a + 1 : a));
            const int bb = j == 0 ? b : (j == 1 ? (half == 0 ? b : b + 1) : b + 1);
            const float lx = (float)(-ts / 2 + ((double)aa / 7.0) * ts), lz = (float)(-ts / 2 + ((double)bb / 7.0) * ts);
            v[j] = shade_vertex(x, sh, lx, 0.0f, lz, 0.f, 1.f, 0.f, 1.f, 1.f, 1.f, (float)((double)aa / 7.0),
                                (float)(1.0 - (double)bb / 7.0));
          }
        }
        process_triangle_lanes(ec, k < 98, v[0], v[1], v[2], base_id + k, tex, -1, lane);
          }
    }
  } else {
    // placed mesh S:1905-1907, O:123-148: T(pos) S(scale) Ry(y_rot)
    const int o = item - 1 - n_tiles;
    const DObject& ob = agent_item ? m.agent : m.objects[o];
    int alt_from = -2;        // traffic-light card on pattern 1: swap this texture id for ob.alt_to
    if (dyn_kind == DTS_DYN_TRAFFICLIGHT) {
      const size_t nd = m.n_dyn, ne = rc.n_envs;
      if (m.dyn_state[((size_t)DTS_DYN_SHOWN * nd + m.dyn[ob.dyn_slot].tl_first) * ne + env] != 0.0) alt_from = ob.alt_from;
    }
    double sn, cs;
    sincos((double)orot * kDeg2Rad, &sn, &cs);
    model_view(sh.V, (double)opx, (double)ob.pos[1], (double)opz, (double)ob.scale, cs, sn, x, lane);
    int base_id = 2 + tris_per_tile * n_tiles;
    for (int q = 0; q < o; q++) base_id += m.objects[q].tri_count;   // (the agent item follows every object)
    for (int k0 = 0; k0 < ob.tri_count; k0 += 32) {
      const int k = k0 + lane;
      Vtx v[3];
      int ttex = -1;
      if (k < ob.tri_count) {
        const size_t ti = (size_t)ob.tri_offset + k;
        const float* p = m.tri_pos + ti * 9;
        const float* n = m.tri_nrm + ti * 9;
        const float* uv = m.tri_uv + ti * 6;
        const float* c = m.tri_col + ti * 9;
#pragma unroll
        for (int j = 0; j < 3; j++)
          v[j] = shade_vertex(x, sh, p[3 * j], p[3 * j + 1], p[3 * j + 2], n[3 * j], n[3 * j + 1], n[3 * j + 2],
                              c[3 * j], c[3 * j + 1], c[3 * j + 2], uv[2 * j], uv[2 * j + 1]);
        ttex = m.tri_tex[ti];
        if (ttex == alt_from) ttex = ob.alt_to;
        if (seg) ttex = ob.seg_tex;   // get_mesh(name, segment=True): every chunk shows the flat class colour (M:268-290)
      }
      process_triangle_lanes(ec, k < ob.tri_count, v[0], v[1], v[2], base_id + k, ttex, -1, lane);
      }
  }
  if (lane == 0 && ctx.overflow) { atomicOr(err, 1); *reinterpret_cast<volatile int32_t*>(fm.status) = 1; }
}

template <bool kTess>
__global__ void __launch_bounds__(kGeoWarps * 32, kGeoMinCtas)
k_geometry(const DState S, const DMap* __restrict__ maps, RenderCfg rc, FrameMem fm, int max_prims, int max_lat,
           int32_t* __restrict__ err) {
  __shared__ GeoWarp gws[kGeoWarps];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int n_list = fm.work[2];   // written by k_cull
  for (int wi = blockIdx.x * kGeoWarps + wib; wi < n_list; wi += gridDim.x * kGeoWarps) {
    const uint2 e = fm.geo_list[wi];
    geometry_item<kTess>(S, maps, rc, fm, max_prims, max_lat, err, (int)e.x, (int)e.y, lane, gws[wib]);
  }
}

// ------------------------------------------------------------------------------------------------ k_bin
// CTA (1 or 4 warps) per env, the env's prims striped over the warps.  Pass 1: exact-size lists of (prim, 32x8-px coarse bin)
// pairs — count (shared-memory atomics), scan, scatter; prims with a small bounding box are binned by it, larger ones
// test each bin of the box against their edges, one bin per lane.  Pass 2, dense over the pairs (one per thread, so a
// screen-filling prim costs no more lanes than a sliver): the pair's BinRec.
constexpr int kBinWarps = 4;
constexpr int kCountMask = 0xfffff, kGroundInc = 1 << 20;   // a bin's counter: records | ground-quad records << 20
template <bool kFish>   // true: bins are the LUT's source boxes of the output bins (fused fisheye gather)
__global__ void __launch_bounds__(kBinWarps * 32)
k_bin(RenderCfg rc, FrameMem fm, FishTab ft, int max_prims, int max_pairs, int32_t* __restrict__ err) {
  extern __shared__ int bin_smem[];
  __shared__ int s_total, s_base, s_ok;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, tid = threadIdx.x;
  const int env = blockIdx.x, nthr = blockDim.x;   // 1 warp per env for small cameras, 4 for large ones (launch_render)
  const int W = rc.width, H = rc.height;
  const int cbins_x = (W + kCoarseW - 1) / kCoarseW, cbins_y = (H + kCoarseH - 1) / kCoarseH, cbins = cbins_x * cbins_y;
  int* cnt = bin_smem;
  int* start = cnt + cbins;
  const PrimRec* prims = fm.prims + (size_t)env * max_prims;
  uint32_t* pairs = fm.pairs;
  const int n = min(fm.ctx[env].n_prims, max_prims);
  for (int pass = 0; pass < 2; pass++) {
    for (int b = tid; b < cbins; b += nthr) cnt[b] = 0;
    __syncthreads();
    for (int p0 = wib * 32; p0 < n; p0 += nthr) {
      const int p = p0 + lane;
      const bool have = p < n;
      int qx[4] = {0, 0, 0, 0}, qy[4] = {0, 0, 0, 0}, nv = 3, ginc = 1;
      if (have) {
        const int4 w0 = __ldg(reinterpret_cast<const int4*>(prims + p));
        const int4 w1 = __ldg(reinterpret_cast<const int4*>(prims + p) + 1);
        qx[0] = w0.x; qx[1] = w0.z; qx[2] = w1.x; qx[3] = w1.z;
        qy[0] = w0.y; qy[1] = w0.w; qy[2] = w1.y; qy[3] = w1.w;
        nv = ((__ldg(&prims[p].ltq) >> 24) & 1) ? 4 : 3;   // vertex 3 of a triangle repeats vertex 0
        if (__ldg(&prims[p].id) < 2) ginc = 1 + kGroundInc;   // the ground quad's records are counted in the upper bits too
      }
      const int minx = min(min(qx[0], qx[1]), min(qx[2], qx[3])), maxx = max(max(qx[0], qx[1]), max(qx[2], qx[3]));
      const int miny = min(min(qy[0], qy[1]), min(qy[2], qy[3])), maxy = max(max(qy[0], qy[1]), max(qy[2], qy[3]));
      // pixel bounding box, and (identity bins) the range of coarse bins it meets
      const int pminx = max(minx >> 6, 0), pmaxx = min(maxx >> 6, W - 1), pminy = max(miny >> 6, 0), pmaxy = min(maxy >> 6, H - 1);
      const int bx0 = pminx / kCoarseW, by0 = pminy / kCoarseH, bx1 = pmaxx / kCoarseW, by1 = pmaxy / kCoarseH;
      // A prim that may meet many bins is handed to the whole warp (one bin per lane and round) instead of one lane
      // walking all of them while 31 wait: the ground quad and the near tiles span hundreds of bins.
      const bool big = have && (bx1 - bx0 + 1) * (by1 - by0 + 1) > 8;   // (fisheye: source cells under the prim's box)
      if (have && !big) {
        if (kFish) {
          // the output bins whose SOURCE box meets the prim, through the inverse index: the source cells under the prim's
          // pixel box (the same 32x8 grid), each with its list of output bins.  A bin listed by several of those cells
          // is taken from the first one only (the cell holding the top-left corner of box ∩ prim-cell-range).
          for (int cy = by0; cy <= by1; cy++)
            for (int cx = bx0; cx <= bx1; cx++) {
              const int c = cy * cbins_x + cx;
              for (int q = ft.cell_start[c]; q < ft.cell_start[c + 1]; q++) {
                const int b = ft.cell_bins[q];
                const short4 cb = ft.cbox[b];
                if (pmaxx < cb.x || pminx > cb.z || pmaxy < cb.y || pminy > cb.w) continue;
                if (cx != max(bx0, cb.x / kCoarseW) || cy != max(by0, cb.y / kCoarseH)) continue;   // counted from another cell
                const int pos = atomicAdd(&cnt[b], ginc) & kCountMask;
                if (pass == 1) pairs[start[b] + pos] = (uint32_t)p | ((uint32_t)b << 16);
              }
            }
        } else {
          const bool large = (bx1 - bx0 + 1) * (by1 - by0 + 1) > 4;
          for (int by = by0; by <= by1; by++)
            for (int bx = bx0; bx <= bx1; bx++) {
              if (large && !bin_overlaps(qx, qy, nv, bx * kCoarseW * kSub, by * kCoarseH * kSub)) continue;
              const int b = by * cbins_x + bx;
              const int pos = atomicAdd(&cnt[b], ginc) & kCountMask;
              if (pass == 1) pairs[start[b] + pos] = (uint32_t)p | ((uint32_t)b << 16);
            }
        }
      }
      unsigned bigs = __ballot_sync(0xffffffffu, big);
      while (bigs) {
        const int src = __ffs(bigs) - 1;
        bigs &= bigs - 1;
        int vx[4], vy[4];
#pragma unroll
        for (int k = 0; k < 4; k++) { vx[k] = __shfl_sync(0xffffffffu, qx[k], src); vy[k] = __shfl_sync(0xffffffffu, qy[k], src); }
        const int snv = __shfl_sync(0xffffffffu, nv, src), sp = p0 + src, sginc = __shfl_sync(0xffffffffu, ginc, src);
        if (kFish) {
          // one HOME cell per lane and round: every output bin is listed once, under the source cell holding the top-left
          // corner of its source box (second inverse index), so a prim spanning many cells meets each candidate bin once;
          // the range of home cells is the prim's cell range grown up / left by the largest box extent of the LUT
          const int sminx = __shfl_sync(0xffffffffu, pminx, src), smaxx = __shfl_sync(0xffffffffu, pmaxx, src);
          const int sminy = __shfl_sync(0xffffffffu, pminy, src), smaxy = __shfl_sync(0xffffffffu, pmaxy, src);
          const int hx0 = max(__shfl_sync(0xffffffffu, bx0, src) - ft.ext_x, 0), sbx1 = __shfl_sync(0xffffffffu, bx1, src);
          const int hy0 = max(__shfl_sync(0xffffffffu, by0, src) - ft.ext_y, 0), sby1 = __shfl_sync(0xffffffffu, by1, src);
          const int nbx = sbx1 - hx0 + 1, nb = nbx * (sby1 - hy0 + 1);
          for (int i = lane; i < nb; i += 32) {
            const int cy = hy0 + i / nbx, cx = hx0 + i % nbx, c = cy * cbins_x + cx;
            const int q1 = __ldg(ft.home_start + c + 1);
            for (int q = __ldg(ft.home_start + c); q < q1; q++) {
              const int4 e = __ldg(ft.home_ent + q);   // x0 | y0 << 16, x1 | y1 << 16, bin
              const int x0 = (int)(short)(e.x & 0xffff), y0 = e.x >> 16, x1 = (int)(short)(e.y & 0xffff), y1 = e.y >> 16;
              if (smaxx < x0 || sminx > x1 || smaxy < y0 || sminy > y1) continue;
              if (!box_overlaps(vx, vy, snv, x0 * kSub + 8, x1 * kSub + 56, y0 * kSub + 8, y1 * kSub + 56)) continue;
              const int pos = atomicAdd(&cnt[e.z], sginc) & kCountMask;
              if (pass == 1) pairs[start[e.z] + pos] = (uint32_t)sp | ((uint32_t)e.z << 16);
            }
          }
        } else {
          const int sbx0 = __shfl_sync(0xffffffffu, bx0, src), sbx1 = __shfl_sync(0xffffffffu, bx1, src);
          const int sby0 = __shfl_sync(0xffffffffu, by0, src), sby1 = __shfl_sync(0xffffffffu, by1, src);
          const int nbx = sbx1 - sbx0 + 1, nb = nbx * (sby1 - sby0 + 1);
          for (int i = lane; i < nb; i += 32) {
            const int by = sby0 + i / nbx, bx = sbx0 + i % nbx;
            if (!bin_overlaps(vx, vy, snv, bx * kCoarseW * kSub, by * kCoarseH * kSub)) continue;
            const int b = by * cbins_x + bx;
            const int pos = atomicAdd(&cnt[b], sginc) & kCountMask;
            if (pass == 1) pairs[start[b] + pos] = (uint32_t)sp | ((uint32_t)b << 16);
          }
        }
      }
    }
    __syncthreads();
    if (pass == 0) {
      if (wib == 0) {
        int carry = 0;
        for (int b0 = 0; b0 < cbins; b0 += 32) {
          const int b = b0 + lane;
          const int v = b < cbins ? (cnt[b] & kCountMask) : 0;
          int inc = v;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) { const int t_ = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += t_; }
          if (b < cbins) start[b] = carry + inc - v;
          carry += __shfl_sync(0xffffffffu, inc, 31);
        }
        if (lane == 0) {   // this env's run of the batch-wide pair pool
          const unsigned base = atomicAdd(reinterpret_cast<unsigned*>(fm.work) + 1, (unsigned)carry);
          s_total = carry; s_base = (int)base;
          s_ok = (unsigned long long)base + (unsigned)carry <= (unsigned long long)max_pairs;
        }
      }
      __syncthreads();
      const int base = s_base;
      const bool ok = s_ok != 0;
      for (int b = tid; b < cbins; b += nthr) {
        start[b] += base;
        fm.bin_count[(size_t)env * cbins + b] = ok ? (cnt[b] & kCountMask) : 0;   // lists that do not fit: the frame stays clear
        fm.bin_start[(size_t)env * cbins + b] = start[b];
      }
      if (!ok) {
        if (tid == 0) { fm.ctx[env].overflow = 1; atomicOr(err, 1); *reinterpret_cast<volatile int32_t*>(fm.status) = 1; }
        return;
      }
    }
  }
  // pass 2: one pair per thread -> its visibility record (the pairs were written by other threads of this CTA: the
  // barrier above orders those writes before these reads)
  const int pair0 = s_base, total = s_total;
  const bool solo_on = rc.obs_layout == DTS_OBS_HWC && rc.obs_dtype == DTS_OBS_U8 && (W & 3) == 0;
  BinRec* recs = fm.recs;
  for (int i = pair0 + tid; i < pair0 + total; i += nthr) {
    const uint32_t pair = pairs[i];
    const int p = (int)(pair & 0xffffu), b = (int)(pair >> 16);
    const int cby = b / cbins_x, cbx = b - cby * cbins_x;
    unsigned r;
    if (kFish) {
      const short4 cb = ft.cbox[b];
      r = build_binrec(prims + p, p, cb.x * kSub, cb.y * kSub, recs + i, ft.fbox + (size_t)b * 8);
    } else {
      r = build_binrec(prims + p, p, cbx * kCoarseW * kSub, cby * kCoarseH * kSub, recs + i);
    }
    {
      if (solo_on) {
        // the coarse bin lies inside this prim and holds no other (besides the ground, hidden below it): no visibility
        // work at all -> the bin goes to k_raster_solo, and k_raster skips it (negative count)
        const int c = cnt[b];
        const unsigned valid = fine_bins_inside(cbx, cby, W, H);
        // (... or it is the bin's only record: a stretch of bare ground)
        const bool alone = (r & 0x100u) ? (c & kCountMask) == 1 : (c & kCountMask) - (c >> 20) == 1;
        if (alone && (r & valid) == valid) {
          fm.bin_count[(size_t)env * cbins + b] = -(p + 1);
          const int slot = atomicAdd(fm.work + 3, 1);
          fm.solo[slot] = make_uint2((unsigned)env, (unsigned)b | ((unsigned)p << 16));
        }
      }
    }
  }
}

// Everything the inline store does not cover — wrapper layouts / dtypes, widths that are no multiple of 4, bins cut
// by the right border, and the gathering step's extra stores into every peer's buffer — out of line.
__device__ __noinline__ void emit_general(uint8_t* __restrict__ out, const GatherTab& gt, int n_peers, size_t env_off, int out_fmt,
                                          unsigned rgb, int lane, int bx, int by, int W, int H) {
  store_bin_any(out, out_fmt, rgb, lane, bx, by, W, H);
  for (int p = 0; p < n_peers; p++) store_bin_any(gt.base[p] + env_off, out_fmt, rgb, lane, bx, by, W, H);
}
// A finished run of image rows -> every rank's gather buffer (peer memory over NVLink): 16-byte vectors, 512 contiguous
// bytes per warp store.  The rows were written by this very warp (__syncwarp orders those stores before these loads).
__device__ __noinline__ void gather_rows_out(const uint8_t* __restrict__ src, const GatherTab& gt, size_t off, size_t nbytes, int lane) {
  __syncwarp();
  const uint8_t* s = src + off;
  if (((reinterpret_cast<size_t>(s) | nbytes) & 15) == 0) {
    bool aligned = true;
    for (int p = 0; p < gt.n; p++) aligned &= (reinterpret_cast<size_t>(gt.base[p] + off) & 15) == 0;
    if (aligned) {
      for (size_t i = (size_t)lane * 16; i < nbytes; i += 512) {
        const int4 v = __ldcg(reinterpret_cast<const int4*>(s + i));   // from L2, where this warp's stores went
        for (int p = 0; p < gt.n; p++) *reinterpret_cast<int4*>(gt.base[p] + off + i) = v;
      }
      return;
    }
  }
  for (size_t i = lane; i < nbytes; i += 32) {
    const uint8_t v = __ldcg(s + i);
    for (int p = 0; p < gt.n; p++) gt.base[p][off + i] = v;
  }
}

constexpr size_t kRasterSmem = (sizeof(BinRec) * 2 * kStage + 16 + 128 * sizeof(unsigned long long)) * kWarps;
// order-preserving map of a float onto unsigned (and back): depth keys of the tiny-triangle buffer
__device__ __forceinline__ unsigned float_key(float f) { const unsigned b = __float_as_uint(f); return b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u); }
__device__ __forceinline__ float key_float(unsigned k) { return __uint_as_float(k ^ ((k >> 31) ? 0x80000000u : 0xffffffffu)); }

// ------------------------------------------------------------------------------------------------ k_raster
template <bool kWrapFmt, bool kFish>   // kWrapFmt: a dts_output_format other than packed u8 HWC is written by the resolve;
                                       // kFish: every lane renders the SOURCE pixel the fisheye LUT names for its output pixel
__global__ void __launch_bounds__(kThreads, kRenderMinCtas)
k_raster(const DState S, const DMap* __restrict__ maps, RenderCfg rc, FrameMem fm, FishTab ft, GatherTab gt,
         uint8_t* __restrict__ obs, int max_prims, int max_pairs, int max_lat, int32_t* __restrict__ err) {
  // dynamic shared memory (kRasterSmem bytes): per warp two chunks of records in flight, their mbarriers, and a 128-sample
  // depth / winner buffer for the tiny triangles of the fine bin being drawn
  extern __shared__ __align__(128) unsigned char raster_smem[];
  BinRec (*stages)[2][kStage] = reinterpret_cast<BinRec (*)[2][kStage]>(raster_smem);
  uint64_t (*bars)[2] = reinterpret_cast<uint64_t (*)[2]>(raster_smem + sizeof(BinRec) * kWarps * 2 * kStage);
  unsigned long long* zb = reinterpret_cast<unsigned long long*>(raster_smem + sizeof(BinRec) * kWarps * 2 * kStage + 16 * kWarps) +
                           128 * (threadIdx.x >> 5);
  const int W = rc.width, H = rc.height;
  const int cbins_x = (W + kCoarseW - 1) / kCoarseW, cbins_y = (H + kCoarseH - 1) / kCoarseH, cbins = cbins_x * cbins_y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t frame_bytes = (size_t)W * H * 3;
  const int out_fmt = !kWrapFmt ? 0 : (rc.obs_layout | (rc.obs_dtype << 2));   // wrapper output format (0 = packed u8 HWC)
  const size_t out_elem = (kWrapFmt && rc.obs_dtype == DTS_OBS_F32_UNIT) ? 4 : 1;
  const int pxs = (lane & 7) * kSub, pys = (lane >> 3) * kSub;   // this lane's pixel inside a fine bin (sub-pixels)
  const StoreLane sl = make_store_lane(lane, W);
  const bool fast_fmt = !kWrapFmt && (W & 3) == 0;   // packed u8 HWC rows of whole words
  const bool planar_u8 = kWrapFmt && rc.obs_dtype == DTS_OBS_U8 &&
                         ((rc.obs_layout == DTS_OBS_CHW && (W & 3) == 0) || (rc.obs_layout == DTS_OBS_CWH && (H & 3) == 0));
  uint64_t* bar = bars[warp];
  if (lane == 0) { mbar_init(&bar[0], 1); mbar_init(&bar[1], 1); mbar_fence_init(); }
  __syncwarp();
  uint32_t parity = 0;   // bit s: the phase the next wait on slot s completes
  int cs = 0, ps = 0;    // consumer / producer slot
  const int n_work = rc.n_envs * cbins_y;   // work item = one row of coarse bins of one env
  int work = 0;
  if (lane == 0) work = atomicAdd(fm.work, 1);
  work = __shfl_sync(0xffffffffu, work, 0);
  while (work < n_work) {
    int next_work = 0;
    if (lane == 0) next_work = atomicAdd(fm.work, 1);   // consumed after this row: latency hidden
    const int env = work / cbins_y, cby = work - env * cbins_y;
    const DMap& m = maps[S.map_id[env]];
    const uint8_t* tex_pool = m.tex_pool;
    const PrimRec* prims = fm.prims + (size_t)env * max_prims;
    const BinRec* recs = fm.recs;   // bin_start holds pool indices
    const float4* lat_tab = fm.lat + (size_t)env * max_lat * 64;
    const size_t env_off = (size_t)env * frame_bytes * out_elem;
    uint8_t* out = obs + env_off;
    // one fine bin -> the caller's tensor and, on a gathering step, every peer's gather buffer (NVLink stores)
    // On a gathering step (gt.n > 0) the packed u8 HWC frame goes to the peers in BLOCKS: a work item is 8 whole image rows =
    // one contiguous run of bytes, copied to every rank's gather buffer with 16-byte vector stores once the item is drawn
    // (NVLink wants long writes: per-bin 4-byte stores reach a fifth of the link rate).  Other layouts store per bin.
    const bool gather_rows = gt.n > 0 && !kWrapFmt;
    auto emit = [&](unsigned rgb, int bx, int by) {
      if (fast_fmt && (gt.n == 0 || gather_rows) && bx * kBinW + kBinW <= W) {   // the common case inline: packed u8 HWC, whole bin inside
        store_bin_fast(out + ((size_t)(by * kBinH) * W + bx * kBinW) * 3, sl, rgb, min(kBinH, H - by * kBinH));
      } else if (kWrapFmt && gt.n == 0) {
        if (planar_u8 && bx * kBinW + kBinW <= W && by * kBinH + kBinH <= H) {
          store_bin_planar_u8(out, out_fmt & 3, rgb, lane, bx, by, W, H);   // CHW / CWH u8: 24 packed words per bin
        } else {
          const int gx = bx * kBinW + (lane & 7), gy = by * kBinH + (lane >> 3);
          if (gx < W && gy < H) store_px_fmt(out, out_fmt & 3, out_fmt >> 2, gx, gy, W, H, rgb);   // wrapper layout / dtype, inline
        }
      } else {
        emit_general(out, gt, gather_rows ? 0 : gt.n, env_off, out_fmt, rgb, lane, bx, by, W, H);
      }
    };
    const bool seg = (rc.mode & DTS_RENDER_SEGMENT) != 0;   // glClearColor(255, 0, 255): clamped to magenta (S:1752)
    const float clr[3] = {seg ? 1.0f : S.rep[env].horizon[0], seg ? 0.0f : S.rep[env].horizon[1], seg ? 1.0f : S.rep[env].horizon[2]};
    const unsigned clear_rgb = pack_rgb(clr[0], clr[1], clr[2]);
    // lane l holds the list of coarse bin (cby, l)
    int my_cnt = 0, my_start = 0;
    if (lane < cbins_x) {
      my_cnt = fm.bin_count[(size_t)env * cbins + cby * cbins_x + lane];
      my_start = fm.bin_start[(size_t)env * cbins + cby * cbins_x + lane];
    }
    const unsigned nz = __ballot_sync(0xffffffffu, my_cnt > 0);
    const unsigned fvalid_y = fine_row_mask(cby, H);
    // ---- producer: walks the row's chunk sequence one chunk ahead of the consumer.  A list of <= 32 records is
    // ONE chunk shared by the bin's 8 fine bins; a longer list is streamed chunk by chunk for each fine bin in turn
    // (the records are ready-made, re-reading them from L2 costs no arithmetic).
    int pcbx = nz ? __ffs(nz) - 1 : 32, pf = 0, pc = 0;
    auto valid8 = [&](int cbx) -> unsigned { return fvalid_y & fine_col_mask(cbx, W); };   // fine_bins_inside(cbx, cby, W, H)
    auto fine_valid = [&](int cbx, int f) -> bool { return (valid8(cbx) >> f) & 1u; };
    auto next_bin = [&]() {
      const unsigned rem = nz & ~((2u << pcbx) - 1u);
      pcbx = rem ? __ffs(rem) - 1 : 32;
      pf = 0; pc = 0;
    };
    auto issue = [&]() {
      if (pcbx >= 32) return;
      const int n = __shfl_sync(0xffffffffu, my_cnt, pcbx), st = __shfl_sync(0xffffffffu, my_start, pcbx);
      if (n > kStage) while (pf < kCFX * kCFY && !fine_valid(pcbx, pf)) pf++;   // fine bins outside the image are not visited
      if (n > kStage && pf >= kCFX * kCFY) { next_bin(); return; }               // (cannot happen: fine bin 0 is always inside)
      const int nch = min(kStage, n - pc);
      if (lane == 0) {
        mbar_expect_tx(&bar[ps], (uint32_t)(nch * sizeof(BinRec)));
        bulk_load(stages[warp][ps], recs + st + pc, (uint32_t)(nch * sizeof(BinRec)), &bar[ps]);
      }
      ps ^= 1;
      if (n <= kStage) { next_bin(); return; }
      pc += kStage;
      if (pc >= n) {
        pc = 0; pf++;
        while (pf < kCFX * kCFY && !fine_valid(pcbx, pf)) pf++;
        if (pf >= kCFX * kCFY) next_bin();
      }
    };
    issue();
    for (int cbx = 0; cbx < cbins_x; cbx++) {
      const int count = __shfl_sync(0xffffffffu, my_cnt, cbx);
      if (count < 0) continue;   // drawn by k_raster_solo (a bin inside one prim)
      const unsigned fvalid = valid8(cbx);
      DTS_COUNT(8, 1);
      if (count == 0) {
        DTS_COUNT(9, 1);
#pragma unroll 1
        for (int f = 0; f < kCFX * kCFY; f++)
          if ((fvalid >> f) & 1u) {
            unsigned rgb = clear_rgb;
            if (kFish && !fish_src(ft, (cbx * kCFX + (f & 3)) * kBinW + (lane & 7), (cby * kCFY + (f >> 2)) * kBinH + (lane >> 3), W, H).valid)
              rgb = 0u;
            emit(rgb, cbx * kCFX + (f & 3), cby * kCFY + (f >> 2));
          }
        continue;
      }
      const bool single = count <= kStage;
      DTS_COUNT(10, count);
      if (!single) { DTS_COUNT(14, 1); DTS_COUNT(15, count); }
      int ox = cbx * kCoarseW * kSub, oy = cby * kCoarseH * kSub;   // coarse bin corner, sub-pixels
      if (kFish) { const short4 cb = ft.cbox[cby * cbins_x + cbx]; ox = cb.x * kSub; oy = cb.y * kSub; }   // ... of its source box
#pragma unroll 1
      for (int g = 0; g < (single ? 1 : kCFX * kCFY); g++) {
        if (!single && !((fvalid >> g) & 1u)) continue;
        float z[4];
        unsigned wn[4];   // per sample: depth and winning prim (index into the env's slab)
        bool zb_used = false;   // tiny triangles of this fine bin went through the shared depth / winner buffer
#pragma unroll 1
        for (int c0 = 0; c0 < count; c0 += kStage) {
          // ---- acquire this chunk; the next one starts loading into the other slot meanwhile
          __syncwarp();   // every lane is done with the slot the producer is about to refill
          issue();
          mbar_wait(&bar[cs], (parity >> cs) & 1u);
          parity ^= 1u << cs;
          const BinRec* stage = stages[warp][cs];
          cs ^= 1;
          const int nch = min(kStage, count - c0);
          uint2 mine = make_uint2(0u, 0u);
          if (lane < nch) mine = *reinterpret_cast<const uint2*>(&stage[lane].prim_flags);
          const bool first = c0 == 0, last = c0 + kStage >= count;
          const unsigned ground_bits = __ballot_sync(0xffffffffu, (mine.y & 2u) != 0u);   // the ground quad's records in this chunk
          const unsigned tiny_bits = kFish ? 0u : __ballot_sync(0xffffffffu, (mine.y & 4u) != 0u);   // one-per-lane triangles
          const unsigned flat_bits = __ballot_sync(0xffffffffu, (mine.y & 8u) != 0u);   // road tiles (plane y = 0)
#if DTS_STATS
          if (single) {   // census: coarse bins lying inside ONE prim (besides the ground)
            const unsigned ng_ = __ballot_sync(0xffffffffu, !(mine.y & 2u) && ((mine.x >> 16) & fvalid) != 0u);
            const unsigned ngfull_ = __ballot_sync(0xffffffffu, !(mine.y & 2u) && ((mine.x >> 24) & fvalid) == fvalid);
            if (ng_ && !(ng_ & (ng_ - 1)) && (ng_ & ngfull_)) { DTS_COUNT(22, 1); DTS_COUNT(23, __popc(fvalid)); }
          }
#endif
#pragma unroll 1
          for (int f = (single ? 0 : g); f < (single ? kCFX * kCFY : g + 1); f++) {
            if (!((fvalid >> f) & 1u)) continue;
            const int bx = cbx * kCFX + (f & 3), by = cby * kCFY + (f >> 2);   // fine bin
            int pxc = pxs + (f & 3) * kBinW * kSub, pyc = pys + (f >> 2) * kBinH * kSub;   // this lane's pixel, coarse-relative
            bool px_valid = true;
            if (kFish) {   // the source pixel of this lane's output pixel
              const FishSrc s = fish_src(ft, bx * kBinW + (lane & 7), by * kBinH + (lane >> 3), W, H);
              px_valid = s.valid;
              pxc = s.x - ox; pyc = s.y - oy;
            }
            const bool live = (mine.x >> (16 + f)) & 1u;
            const unsigned live_mask = __ballot_sync(0xffffffffu, live);
            const unsigned ground_mask = live_mask & ground_bits;
            bool simple = false;
            if (single) {
              // ---- simple bin: ONE prim (besides the ground quad) and it covers every sample of the bin.
              // All four samples then carry its colour (depth cleared to 1 passes, the ground lies below
              // every other surface and fails GL_LESS), and the mean of four equal floats is exact.
              const unsigned full_mask = __ballot_sync(0xffffffffu, live && ((mine.x >> (24 + f)) & 1u));
              const unsigned others = live_mask & ~ground_mask;
              const unsigned pick = others ? others : live_mask;
              if (pick && !(pick & (pick - 1)) && (pick & full_mask)) {
                simple = true;
                DTS_COUNT(13, 1);
                const unsigned w = stage[__ffs(pick) - 1].prim_flags & 0xffffu;
                wn[0] = w; wn[1] = w; wn[2] = w; wn[3] = w;
              }
            }
            // every prim of the bin besides the ground quad is a road tile: the tiles are coplanar and (up to slivers where
            // two neighbours snapped their shared border differently) disjoint, so a sample belongs to the one tile that
            // covers it — no depth arithmetic; the ground lies below them and takes what is left.  A sample that turns
            // out to be covered twice sends the whole bin through the depth-tested path (exactly the spec's answer).
            bool coplanar = single && !(live_mask & ~ground_mask & ~flat_bits);
            if (coplanar && !simple) DTS_COUNT(20, 1);
            if (!simple) {
              if (first) {
#pragma unroll
                for (int s = 0; s < 4; s++) { z[s] = 1.0f; wn[s] = kNoPrim; }
                zb_used = false;
              }
              // ---- visibility: everything else first, the ground quad last (it is almost always hidden)
#pragma unroll 1
              for (int phase = 0; phase < 2; phase++) {
                unsigned todo = phase == 0 ? (live_mask & ~ground_mask & ~tiny_bits) : ground_mask;
                // every sample of the bin already belongs to a surface above the ground plane: the ground quad
                // (y = -0.008, below everything else) cannot pass GL_LESS anywhere — same argument as the simple bin
                if (phase == 1 && todo &&
                    __all_sync(0xffffffffu, wn[0] != kNoPrim && wn[1] != kNoPrim && wn[2] != kNoPrim && wn[3] != kNoPrim))
                  todo = 0;
                int seen = 0, twice = 0;   // (coverage-only mode) samples of this pixel covered so far / covered by two tiles
                while (todo) {
                  const int k = __ffs(todo) - 1;
                  todo &= todo - 1;
                  const BinRec& br = stage[k];
                  const uint32_t pflags = br.prim_flags;
                  DTS_COUNT(16, 1);
                  if ((pflags >> (24 + f)) & 1u) DTS_COUNT(17, 1);
                  int mask = 15;
                  if (!((pflags >> (24 + f)) & 1u)) {
                    const int4 E = *reinterpret_cast<const int4*>(br.E0);
                    const int4 A = *reinterpret_cast<const int4*>(br.A);
                    const int4 B = *reinterpret_cast<const int4*>(br.B);
                    const int ec0 = E.x + A.x * pxc + B.x * pyc;
                    const int ec1 = E.y + A.y * pxc + B.y * pyc;
                    const int ec2 = E.z + A.z * pxc + B.z * pyc;
                    mask = 0;
                    if (br.kind & 1) {
                      const int ec3 = E.w + A.w * pxc + B.w * pyc;
#pragma unroll
                      for (int s = 0; s < 4; s++) {
                        const int e0 = ec0 + A.x * sample_x(s) + B.x * sample_y(s);
                        const int e1 = ec1 + A.y * sample_x(s) + B.y * sample_y(s);
                        const int e2 = ec2 + A.z * sample_x(s) + B.z * sample_y(s);
                        const int e3 = ec3 + A.w * sample_x(s) + B.w * sample_y(s);
                        if ((e0 | e1 | e2 | e3) >= 0) mask |= 1 << s;
                      }
                    } else {
#pragma unroll
                      for (int s = 0; s < 4; s++) {
                        const int e0 = ec0 + A.x * sample_x(s) + B.x * sample_y(s);
                        const int e1 = ec1 + A.y * sample_x(s) + B.y * sample_y(s);
                        const int e2 = ec2 + A.z * sample_x(s) + B.z * sample_y(s);
                        if ((e0 | e1 | e2) >= 0) mask |= 1 << s;
                      }
                    }
                    if (!mask) continue;
                  }
                  if (coplanar && phase == 0) {
                    twice |= seen & mask;
                    seen |= mask;
#pragma unroll
                    for (int s = 0; s < 4; s++)
                      if (mask >> s & 1) wn[s] = pflags & 0xffffu;
                    continue;
                  }
                  // ---- depth of the covered samples, GL_LESS in draw order
                  const float4 zp = *reinterpret_cast<const float4*>(&br.z0);   // z0 zx zy id
                  const int2 xy0 = *reinterpret_cast<const int2*>(&br.x0);
                  const float cdx = (float)(pxc + 32 - xy0.x) * 0.015625f, cdy = (float)(pyc + 32 - xy0.y) * 0.015625f;
                  float zs[4];
                  int lt = 0, eq = 0;
#pragma unroll
                  for (int s = 0; s < 4; s++) {
                    // sample offset from the pixel centre is a multiple of 1/64: cdx + off is exact, i.e.
                    // identical to the spec's (float)(X_sample - x0) / 64
                    const float sdx = cdx + (float)(sample_x(s) - 32) * 0.015625f, sdy = cdy + (float)(sample_y(s) - 32) * 0.015625f;
                    zs[s] = fmaf(zp.z, sdy, fmaf(zp.y, sdx, zp.x));
                    lt |= (zs[s] < z[s]) << s;
                    eq |= (zs[s] == z[s]) << s;
                  }
                  int pass_mask = mask & lt;
                  const int tie = mask & eq;
                  if (tie) {   // exact depth ties are rare: the earlier draw keeps the sample (its id comes from the slab)
                    const int my_id = __float_as_int(zp.w);
#pragma unroll
                    for (int s = 0; s < 4; s++)
                      if ((tie >> s & 1) && wn[s] != kNoPrim && my_id < __ldg(&prims[wn[s]].id)) pass_mask |= 1 << s;
                  }
                  if (!pass_mask) continue;
                  const unsigned me = pflags & 0xffffu;
#pragma unroll
                  for (int s = 0; s < 4; s++)
                    if (pass_mask >> s & 1) { z[s] = zs[s]; wn[s] = me; }
                }
                if (coplanar && phase == 0) {
                  if (__any_sync(0xffffffffu, twice != 0)) {   // rare: start the bin over, depth-tested
                    coplanar = false;
                    DTS_COUNT(21, 1);
#pragma unroll
                    for (int s = 0; s < 4; s++) wn[s] = kNoPrim;
                    phase = -1;
                  } else {
#pragma unroll
                    for (int s = 0; s < 4; s++)
                      if (seen >> s & 1) z[s] = -1.0f;   // the ground (phase 1) can neither pass nor tie there
                  }
                }
              }
            }
            if (!kFish && !simple && (live_mask & tiny_bits)) {
              // ---- tiny triangles, ONE PER LANE: each lane walks the few pixels of its triangle inside this fine bin and
              // resolves GL_LESS (ties to the lower draw id) with a 64-bit atomicMin on depth | id | prim per sample —
              // 32 triangles per pass instead of one warp-wide visit per triangle
              if (!zb_used) {
                zb_used = true;
#pragma unroll
                for (int s = 0; s < 4; s++) zb[lane * 4 + s] = ~0ull;
                __syncwarp();
              }
              DTS_COUNT(18, 1);
              DTS_COUNT(19, __popc(live_mask & tiny_bits));
              if ((live_mask & tiny_bits) >> lane & 1u) {
                const BinRec& br = stage[lane];
                const int4 E = *reinterpret_cast<const int4*>(br.E0);
                const int4 A = *reinterpret_cast<const int4*>(br.A);
                const int4 B = *reinterpret_cast<const int4*>(br.B);
                const float4 zp = *reinterpret_cast<const float4*>(&br.z0);
                const int2 xy0 = *reinterpret_cast<const int2*>(&br.x0);
                const int fx0 = (f & 3) * kBinW, fy0 = (f >> 2) * kBinH;
                const int x_lo = max(E.w & 0xffff, fx0), x_hi = min(A.w & 0xffff, fx0 + kBinW - 1);
                const int y_lo = max(E.w >> 16, fy0), y_hi = min(A.w >> 16, fy0 + kBinH - 1);
                const unsigned long long tail = ((unsigned long long)(unsigned)__float_as_int(zp.w) << 16) | (br.prim_flags & 0xffffu);
                for (int py = y_lo; py <= y_hi; py++)
                  for (int px = x_lo; px <= x_hi; px++) {
                    const int X = px * kSub, Y = py * kSub;
                    const int ec0 = E.x + A.x * X + B.x * Y, ec1 = E.y + A.y * X + B.y * Y, ec2 = E.z + A.z * X + B.z * Y;
#pragma unroll
                    for (int s = 0; s < 4; s++) {
                      const int e0 = ec0 + A.x * sample_x(s) + B.x * sample_y(s);
                      const int e1 = ec1 + A.y * sample_x(s) + B.y * sample_y(s);
                      const int e2 = ec2 + A.z * sample_x(s) + B.z * sample_y(s);
                      if ((e0 | e1 | e2) < 0) continue;
                      const float sdx = (float)(X + sample_x(s) - xy0.x) * 0.015625f, sdy = (float)(Y + sample_y(s) - xy0.y) * 0.015625f;
                      const float zs = fmaf(zp.z, sdy, fmaf(zp.y, sdx, zp.x));
                      atomicMin(&zb[((py - fy0) * kBinW + (px - fx0)) * 4 + s], ((unsigned long long)float_key(zs) << 32) | tail);
                    }
                  }
              }
              __syncwarp();
            }
            if (!(last || simple)) continue;
            if (!kFish && !simple && zb_used) {
              // merge the tiny triangles' winners into the per-sample state: GL_LESS, ties to the lower draw id
#pragma unroll
              for (int s = 0; s < 4; s++) {
                const unsigned long long k = zb[lane * 4 + s];
                if (k == ~0ull) continue;
                const float zt = key_float((unsigned)(k >> 32));
                bool win = zt < z[s];
                if (zt == z[s] && wn[s] != kNoPrim) win = (int)((k >> 16) & 0xffffu) < __ldg(&prims[wn[s]].id);
                if (win) { z[s] = zt; wn[s] = (unsigned)(k & 0xffffu); }
              }
              __syncwarp();   // the buffer is re-initialised by the next fine bin
            }
            // ---- deferred shading: once per distinct winner of this pixel, then the box resolve
            DTS_COUNT(11, 1);
            const int pxa = ox + pxc, pya = oy + pyc;
            const bool same = wn[1] == wn[0] && wn[2] == wn[0] && wn[3] == wn[0];
            const bool all_same = simple || __all_sync(0xffffffffu, same);
            unsigned rgb;
            {
              float c3[3] = {clr[0], clr[1], clr[2]};
              if (wn[0] != kNoPrim) shade_prim(prims, wn[0], tex_pool, lat_tab, pxa, pya, c3);   // every lane: its first winner
              if (all_same) rgb = pack_rgb(c3[0], c3[1], c3[2]);   // four equal samples: the mean is the value itself
              else {
                // edge pixels: the other winners of this pixel (at most three more), summed in the resolve's order
                float s01[3] = {c3[0], c3[1], c3[2]}, s23[3] = {0.f, 0.f, 0.f};   // 0 + c == c
                unsigned pend = 0xeu;
                if (wn[1] == wn[0]) { pend &= ~2u; s01[0] = s01[0] + c3[0]; s01[1] = s01[1] + c3[1]; s01[2] = s01[2] + c3[2]; }
#pragma unroll
                for (int t = 2; t < 4; t++)
                  if (wn[t] == wn[0]) { pend &= ~(1u << t); s23[0] = s23[0] + c3[0]; s23[1] = s23[1] + c3[1]; s23[2] = s23[2] + c3[2]; }
#pragma unroll 1
                while (__any_sync(0xffffffffu, pend != 0u)) {
                  DTS_COUNT(12, 1);
                  if (pend) {
                    const int s = __ffs(pend) - 1;
                    const unsigned w = s == 1 ? wn[1] : (s == 2 ? wn[2] : wn[3]);
                    float d3[3] = {clr[0], clr[1], clr[2]};
                    if (w != kNoPrim) shade_prim(prims, w, tex_pool, lat_tab, pxa, pya, d3);
#pragma unroll
                    for (int t = 1; t < 4; t++)
                      if ((pend >> t & 1u) && wn[t] == w) {
                        pend &= ~(1u << t);
                        if (t < 2) { s01[0] = s01[0] + d3[0]; s01[1] = s01[1] + d3[1]; s01[2] = s01[2] + d3[2]; }
                        else { s23[0] = s23[0] + d3[0]; s23[1] = s23[1] + d3[1]; s23[2] = s23[2] + d3[2]; }
                      }
                  }
                }
                rgb = pack_rgb((s01[0] + s23[0]) * 0.25f, (s01[1] + s23[1]) * 0.25f, (s01[2] + s23[2]) * 0.25f);
              }
            }
            if (kFish && !px_valid) rgb = 0u;   // cv2.remap BORDER_CONSTANT
            emit(rgb, bx, by);
          }
        }
      }
    }
    if (gather_rows) {   // the item's rows are complete: ship them to every rank
      const int rows = min(kCoarseH, H - cby * kCoarseH);
      gather_rows_out(obs, gt, env_off + (size_t)cby * kCoarseH * W * 3, (size_t)rows * W * 3, lane);
    }
    work = __shfl_sync(0xffffffffu, next_work, 0);
  }
}

// ------------------------------------------------------------------------------------------------ k_raster_solo
// Coarse bins that lie inside ONE prim (k_bin found: one record besides the ground quad, covering every sample of every
// fine bin — 22 of the 55 non-empty coarse bins of a c2 frame, 40 % of the shaded pixels) need no records, no staging, no
// visibility state: a warp fetches the prim's planes once and shades the bin's 256 pixels.  A separate kernel so that the
// lean loop gets its own register allocation (the same fast path inside k_raster cost more than it saved).
// Packed u8 HWC output with whole-word rows only (k_bin marks no bin otherwise).  Runs before k_raster.
template <bool kFish>   // true: each lane shades the source pixel the fisheye LUT names for its output pixel
__global__ void __launch_bounds__(256, kSoloMinCtas) k_raster_solo(const DState S, const DMap* __restrict__ maps, RenderCfg rc, FrameMem fm,
                                                                   FishTab ft, uint8_t* __restrict__ obs, int max_prims, int max_lat) {
  const int W = rc.width, H = rc.height;
  const int cbins_x = (W + kCoarseW - 1) / kCoarseW;
  const int lane = threadIdx.x & 31;
  const StoreLane sl = make_store_lane(lane, W);
  const size_t frame_bytes = (size_t)W * H * 3;
  const int n = fm.work[3];
  const int warps = (gridDim.x * blockDim.x) >> 5;
  for (int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += warps) {
    const uint2 e = fm.solo[i];
    const int env = (int)e.x, b = (int)(e.y & 0xffffu);
    const unsigned p = e.y >> 16;
    const int cby = b / cbins_x, cbx = b - cby * cbins_x;
    const uint8_t* tex_pool = maps[S.map_id[env]].tex_pool;
    const float4* lat_tab = fm.lat + (size_t)env * max_lat * 64;
    const ShadeIn si = load_shade(fm.prims + (size_t)env * max_prims, p);
    uint8_t* out = obs + (size_t)env * frame_bytes;
    const int nx = fine_cols_in_image(cbx, W), ny = fine_row_mask(cby, H) == 0xffu ? 2 : 1;   // the fine bins of fine_bins_inside
#pragma unroll 1
    for (int fy = 0; fy < ny; fy++)
#pragma unroll 1
      for (int fx = 0; fx < nx; fx++) {
        const int bx = cbx * kCFX + fx, by = cby * kCFY + fy;
        int pxa = (bx * kBinW + (lane & 7)) * kSub, pya = (by * kBinH + (lane >> 3)) * kSub;
        bool px_valid = true;
        if (kFish) {
          const FishSrc s = fish_src(ft, bx * kBinW + (lane & 7), by * kBinH + (lane >> 3), W, H);
          px_valid = s.valid;
          pxa = s.x; pya = s.y;
        }
        float c3[3];
        shade_eval(si, tex_pool, lat_tab, pxa, pya, c3);
        unsigned rgb = pack_rgb(c3[0], c3[1], c3[2]);
        if (kFish && !px_valid) rgb = 0u;   // cv2.remap BORDER_CONSTANT
        if (bx * kBinW + kBinW <= W) store_bin_fast(out + ((size_t)(by * kBinH) * W + bx * kBinW) * 3, sl, rgb, min(kBinH, H - by * kBinH));
        else store_bin(out, rgb, lane, bx, by, W, H);
      }
  }
}

// ------------------------------------------------------------------------------------------------ k_resize
// ResizeWrapper (wrappers.py:111-141): cv2.resize(..., interpolation=cv2.INTER_CUBIC) of the rendered frame, on the
// device, so that a training stack's 84x84 payload (21 KB per env instead of 57.6 KB) is what crosses PCIe.  OpenCV's
// 8-bit bicubic is fixed point: per output column / row four int16 taps = cvRound(2048 * w_k(frac)), w = the a = -0.75
// cubic kernel evaluated in float32 at frac = (d + 0.5) * scale - 0.5 - floor(.), source indices clamped to the
// image; horizontal pass in int32, then (sum_k beta_k * row_k + 2^21) >> 22, saturated.  The tap tables are built on
// the host (dts_set_resize, cubic_axis_table), one int4 per output column / row: 4 int16 source indices, then the 4
// int16 taps, unpacked by unpack_taps.  One thread per output pixel (3 channels); reads the full-size u8 HWC render.
struct Taps { int i[4], w[4]; };
__device__ __forceinline__ Taps unpack_taps(int4 t) {
  return {{(short)(t.x & 0xffff), t.x >> 16, (short)(t.y & 0xffff), t.y >> 16},
          {(short)(t.z & 0xffff), t.z >> 16, (short)(t.w & 0xffff), t.w >> 16}};
}
__global__ void __launch_bounds__(256) k_resize(const uint8_t* __restrict__ src, int W, int H, int ow, int oh, int n_envs,
                                                const int16_t* __restrict__ xtab /*[ow][8]: 4 indices, 4 taps*/,
                                                const int16_t* __restrict__ ytab /*[oh][8]*/, void* __restrict__ dst, int layout,
                                                int dtype) {
  const size_t total = (size_t)n_envs * ow * oh;
  for (size_t g = blockIdx.x * (size_t)blockDim.x + threadIdx.x; g < total; g += (size_t)gridDim.x * blockDim.x) {
    const int x = (int)(g % ow), y = (int)((g / ow) % oh);
    const size_t env = g / ((size_t)ow * oh);
    const Taps xt = unpack_taps(__ldg(reinterpret_cast<const int4*>(xtab + 8 * x)));
    const Taps yt = unpack_taps(__ldg(reinterpret_cast<const int4*>(ytab + 8 * y)));
    const uint8_t* frame = src + env * (size_t)W * H * 3;
    long long acc[3] = {0, 0, 0};
#pragma unroll
    for (int r = 0; r < 4; r++) {
      const uint8_t* row = frame + (size_t)yt.i[r] * W * 3;
      int h0 = 0, h1 = 0, h2 = 0;
#pragma unroll
      for (int c = 0; c < 4; c++) {
        const uint8_t* px = row + xt.i[c] * 3;
        h0 += (int)px[0] * xt.w[c]; h1 += (int)px[1] * xt.w[c]; h2 += (int)px[2] * xt.w[c];
      }
      acc[0] += (long long)h0 * yt.w[r]; acc[1] += (long long)h1 * yt.w[r]; acc[2] += (long long)h2 * yt.w[r];
    }
    unsigned rgb = 0;
#pragma unroll
    for (int ch = 0; ch < 3; ch++) {
      long long v = (acc[ch] + (1LL << 21)) >> 22;
      v = v < 0 ? 0 : (v > 255 ? 255 : v);
      rgb |= (unsigned)v << (8 * ch);
    }
    void* out = reinterpret_cast<uint8_t*>(dst) + env * (size_t)ow * oh * 3 * (dtype == DTS_OBS_F32_UNIT ? 4 : 1);
    store_px_fmt(out, layout, dtype, x, y, ow, oh, rgb);
  }
}

// ------------------------------------------------------------------------------------------------ k_blend4
// MotionBlurWrapper (learning/utils/wrappers.py:8-54): np.average(window, axis=0, weights=[0.8, 0.15, 0.04, 0.01]) of four
// uint8 frames -> float64, in numpy's order: products in float64, summed frame by frame, divided by the weight sum.
__global__ void __launch_bounds__(256) k_blend4(const uint8_t* __restrict__ f0, const uint8_t* __restrict__ f1,
                                                const uint8_t* __restrict__ f2, const uint8_t* __restrict__ f3, double w0,
                                                double w1, double w2, double w3, double scl, double* __restrict__ out, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    double a = (double)f0[i] * w0;
    a = a + (double)f1[i] * w1;
    a = a + (double)f2[i] * w2;
    a = a + (double)f3[i] * w3;
    out[i] = a / scl;
  }
}
void launch_blend4(const uint8_t* const f[4], const double w[4], double* out, size_t n, cudaStream_t st) {
  const double scl = ((w[0] + w[1]) + w[2]) + w[3];   // numpy: wgt.sum() of four float64 (pairwise == sequential below 8 terms)
  const size_t blocks = (n + 255) / 256;
  k_blend4<<<(unsigned)(blocks < 148 * 32 ? blocks : 148 * 32), 256, 0, st>>>(f[0], f[1], f[2], f[3], w[0], w[1], w[2], w[3], scl, out, n);
}

// The same resize, tiled: a CTA per (band of `R` output rows, env).  The band's source rows (contiguous bytes of the
// render) are copied to shared memory with 16-byte loads, the horizontal pass runs once per source row into an int32
// buffer in shared memory, the vertical pass reads it and writes four output bytes per thread as one word — instead
// of every output pixel fetching its own 48 source bytes from global memory (k_resize above: 0.49 ms at 4096 x
// 160x120 -> 84x84).  Integer arithmetic identical to k_resize.  `cap` = the largest source-row span of any band
// (computed on the host from the same tap table).
__global__ void __launch_bounds__(256) k_resize_band(const uint8_t* __restrict__ src, int W, int H, int ow, int oh,
                                                     const int16_t* __restrict__ xtab, const int16_t* __restrict__ ytab,
                                                     void* __restrict__ dst, int layout, int dtype, int R, int cap) {
  extern __shared__ __align__(16) unsigned char rs_smem[];
  const int bands = (oh + R - 1) / R;
  const int env = blockIdx.x / bands, r0 = (blockIdx.x - env * bands) * R, r1 = min(r0 + R, oh);
  const int s_lo = ytab[8 * r0], s_hi = ytab[8 * (r1 - 1) + 3], nrows = min(s_hi - s_lo + 1, cap);
  const int rowb = W * 3, ow3 = ow * 3;
  int4* xt = reinterpret_cast<int4*>(rs_smem);                                      // [ow] tap table
  uint8_t* sb = rs_smem + (size_t)ow * 16;                                          // [cap][rowb] source bytes
  int* hb = reinterpret_cast<int*>(sb + (((size_t)cap * rowb + 15) & ~(size_t)15));   // [cap][ow3] horizontal sums
  const uint8_t* band = src + (size_t)env * W * H * 3 + (size_t)s_lo * rowb;
  const int nbytes = nrows * rowb;
  if ((reinterpret_cast<uintptr_t>(band) & 15) == 0 && (nbytes & 15) == 0) {
    for (int i = threadIdx.x; i < nbytes / 16; i += blockDim.x) reinterpret_cast<int4*>(sb)[i] = __ldg(reinterpret_cast<const int4*>(band) + i);
  } else {
    for (int i = threadIdx.x; i < nbytes; i += blockDim.x) sb[i] = __ldg(band + i);
  }
  for (int i = threadIdx.x; i < ow; i += blockDim.x) xt[i] = __ldg(reinterpret_cast<const int4*>(xtab) + i);
  __syncthreads();
  // horizontal pass: a warp per source row, a lane per output column (no index divisions), three channels
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  for (int x = lane; x < ow; x += 32) {
    const Taps xa = unpack_taps(xt[x]);
    for (int row = warp; row < nrows; row += nwarps) {
      const uint8_t* rp = sb + row * rowb;
      int h0 = 0, h1 = 0, h2 = 0;
#pragma unroll
      for (int c = 0; c < 4; c++) {
        const uint8_t* px = rp + xa.i[c] * 3;
        h0 += (int)px[0] * xa.w[c]; h1 += (int)px[1] * xa.w[c]; h2 += (int)px[2] * xa.w[c];
      }
      int* hp = hb + row * ow3 + x * 3;
      hp[0] = h0; hp[1] = h1; hp[2] = h2;
    }
  }
  __syncthreads();
  // vertical pass
  const size_t out_elem = dtype == DTS_OBS_F32_UNIT ? 4 : 1;
  uint8_t* out = reinterpret_cast<uint8_t*>(dst) + (size_t)env * ow3 * oh * out_elem;
  const bool words = layout == DTS_OBS_HWC && dtype == DTS_OBS_U8 && (ow3 & 3) == 0 && (reinterpret_cast<uintptr_t>(dst) & 3) == 0;
  if (words) {
    const int wpr = ow3 / 4;   // words per output row
    for (int y = r0 + warp; y < r1; y += nwarps) {   // a warp per output row, a lane per word of four bytes
      const Taps ya = unpack_taps(__ldg(reinterpret_cast<const int4*>(ytab) + y));
      for (int j = lane; j < wpr; j += 32) {
        const int e = 4 * j;
        // int32 like OpenCV's own vertical pass (|sum| <= 255 * sum|xw| * sum|yw| < 2^31 for cubic taps: 255 * 2621^2 = 1.75e9)
        int acc[4] = {0, 0, 0, 0};
#pragma unroll
        for (int r = 0; r < 4; r++) {
          const int4 hv = *reinterpret_cast<const int4*>(hb + (ya.i[r] - s_lo) * ow3 + e);
          acc[0] += hv.x * ya.w[r]; acc[1] += hv.y * ya.w[r]; acc[2] += hv.z * ya.w[r]; acc[3] += hv.w * ya.w[r];
        }
        unsigned word = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const int v = min(max((acc[k] + (1 << 21)) >> 22, 0), 255);
          word |= (unsigned)v << (8 * k);
        }
        *reinterpret_cast<unsigned*>(out + (size_t)y * ow3 + e) = word;
      }
    }
  } else {
    for (int i = threadIdx.x; i < (r1 - r0) * ow3; i += blockDim.x) {
      const int yy = i / ow3, e = i - yy * ow3, y = r0 + yy, x = e / 3, ch = e - 3 * x;
      const Taps ya = unpack_taps(__ldg(reinterpret_cast<const int4*>(ytab) + y));
      long long acc = 0;
#pragma unroll
      for (int r = 0; r < 4; r++) acc += (long long)hb[(ya.i[r] - s_lo) * ow3 + e] * ya.w[r];
      long long v = (acc + (1LL << 21)) >> 22;
      v = v < 0 ? 0 : (v > 255 ? 255 : v);
      const size_t oi = fmt_index(layout, x, y, ch, ow, oh);
      if (dtype == DTS_OBS_F32_UNIT) reinterpret_cast<float*>(out)[oi] = (float)(unsigned)v / 255.0f;
      else out[oi] = (uint8_t)v;
    }
  }
}

size_t resize_band_smem(int W, int ow, int cap) {
  return (size_t)ow * 16 + (((size_t)cap * W * 3 + 15) & ~(size_t)15) + (size_t)cap * ow * 3 * 4 + 16;   // (+16: word loads may run past the last row)
}

void launch_resize(const uint8_t* src, int W, int H, int ow, int oh, int n_envs, const int16_t* xtab, const int16_t* ytab,
                   void* dst, int layout, int dtype, int band_rows, int band_cap, cudaStream_t st) {
  if (band_rows > 0) {   // tiled form (dts_set_resize found a band height whose rows fit in shared memory)
    const size_t smem = resize_band_smem(W, ow, band_cap);
    static size_t opted = 0;
    if (smem > 48 * 1024 && smem > opted) { cudaFuncSetAttribute(k_resize_band, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); opted = smem; }
    k_resize_band<<<(unsigned)(((oh + band_rows - 1) / band_rows) * (size_t)n_envs), 256, smem, st>>>(src, W, H, ow, oh, xtab, ytab, dst, layout, dtype,
                                                                                      band_rows, band_cap);
    return;
  }
  const size_t total = (size_t)n_envs * ow * oh;
  const int blocks = (int)((total + 255) / 256 < 148 * 16 ? (total + 255) / 256 : 148 * 16);
  k_resize<<<blocks, 256, 0, st>>>(src, W, H, ow, oh, n_envs, xtab, ytab, dst, layout, dtype);
}

// Test hook (dts_debug_frame): what k_frame_setup / k_geometry left in frame memory for one env of the last render —
// the camera model-view and projection, the prim / lattice counts, and the lit 8x8 lattice of every road tile that
// was emitted, re-ordered by grid cell (i * grid_h + j; cells that were culled stay NaN).
int debug_frame_copy(void* scratch, int n, int max_prims, int cbins, int max_pairs, int max_lat, size_t geo_items,
                     int env, double* V, float* P, int32_t* counts, float* lattice_by_cell, int n_cells, int tris_per_tile) {
  const FrameMem fm = carve(scratch, n, max_prims, cbins, max_pairs, max_lat, geo_items);
  FrameCtx c;
  if (cudaMemcpy(&c, fm.ctx + env, sizeof c, cudaMemcpyDeviceToHost) != cudaSuccess) return 1;
  for (int k = 0; k < 12; k++) V[k] = c.V[k];
  P[0] = c.P00; P[1] = c.P11; P[2] = c.P22; P[3] = c.P23;
  counts[0] = c.n_prims; counts[1] = c.n_lat; counts[2] = c.overflow; counts[3] = 0;
  cudaMemcpy(&counts[3], fm.work + 1, sizeof(int32_t), cudaMemcpyDeviceToHost);   // (prim, coarse bin) pairs of the whole batch
  const int np = c.n_prims < max_prims ? c.n_prims : max_prims;
  PrimRec* prims = new PrimRec[np > 0 ? np : 1];
  float4* lat = new float4[(size_t)max_lat * 64];
  int rc = 0;
  if (np && cudaMemcpy(prims, fm.prims + (size_t)env * max_prims, (size_t)np * sizeof(PrimRec), cudaMemcpyDeviceToHost) != cudaSuccess) rc = 1;
  if (cudaMemcpy(lat, fm.lat + (size_t)env * max_lat * 64, (size_t)max_lat * 64 * sizeof(float4), cudaMemcpyDeviceToHost) != cudaSuccess) rc = 1;
  for (int k = 0; k < n_cells * 64 * 3; k++) lattice_by_cell[k] = nanf("");
  for (int p = 0; p < np && !rc; p++) {
    const int slot = (prims[p].ltq & 0xffff) - 1;
    if (slot < 0 || slot >= max_lat) continue;
    const int cell = (prims[p].id - 2) / tris_per_tile;   // tiles are drawn i outer, j inner: cell = i * grid_h + j
    if (cell < 0 || cell >= n_cells) continue;
    for (int v = 0; v < 64; v++) {
      lattice_by_cell[(cell * 64 + v) * 3 + 0] = lat[slot * 64 + v].x;
      lattice_by_cell[(cell * 64 + v) * 3 + 1] = lat[slot * 64 + v].y;
      lattice_by_cell[(cell * 64 + v) * 3 + 2] = lat[slot * 64 + v].z;
    }
  }
  delete[] prims;
  delete[] lat;
  return rc;
}

int launch_render(const DState& S, const DMap* maps, const RenderCfg& rc, void* obs_any, void* scratch, int n_ctas,
                  int max_prims, int max_pairs, int max_lat, int items_max, const FishTab& fish, const GatherTab& gather,
                  int32_t* err_flag, int32_t* status_dev, cudaEvent_t* marks, int mark_level, cudaStream_t st) {
  const int W = rc.width, H = rc.height;
  uint8_t* obs = reinterpret_cast<uint8_t*>(obs_any);
  const int cbins = ((W + kCoarseW - 1) / kCoarseW) * ((H + kCoarseH - 1) / kCoarseH);
  const bool fisheye = (rc.flags & DTS_FLAG_DISTORTION) != 0;
  FrameMem fm = carve(scratch, rc.n_envs, max_prims, cbins, max_pairs, max_lat, (size_t)items_max);
  fm.status = status_dev;
  int mk = 0;
  // level 2: an event at every kernel boundary; level 1: only the two around k_raster (marks 3 and 4), so that the
  // timed region of a benchmark carries two event records per step instead of six
  auto mark = [&]() { if (marks && (mark_level >= 2 || mk == 3 || mk == 4)) cudaEventRecord(marks[mk], st); mk++; };
  cudaMemsetAsync(fm.work, 0, 256, st);
  mark();
  k_frame_setup<<<(rc.n_envs + 127) / 128, 128, 0, st>>>(S, maps, rc, fm);
  mark();
  const size_t pairs_total = (size_t)rc.n_envs * items_max;
  k_cull<<<(unsigned)((pairs_total + 255) / 256), 256, 0, st>>>(S, maps, rc, fm, items_max);
  const int geo_ctas = (n_ctas / kRenderMinCtas) * kGeoMinCtas / kGeoWarps;   // SMs x resident geometry CTAs
  if (rc.tessellate) k_geometry<true><<<geo_ctas, kGeoWarps * 32, 0, st>>>(S, maps, rc, fm, max_prims, max_lat, err_flag);
  else k_geometry<false><<<geo_ctas, kGeoWarps * 32, 0, st>>>(S, maps, rc, fm, max_prims, max_lat, err_flag);
  mark();
  const size_t bin_smem_bytes = (size_t)2 * cbins * sizeof(int);
  const int bin_grid = rc.n_envs;   // CTA per env: one warp where a frame has few bins and prims (160x120: 75 bins — more warps
  // only add barriers and CTA launches, measured 58 -> 88 us), four for large cameras (640x480: 9.0 -> 3.3 ms)
  const int bin_threads = cbins > 128 ? kBinWarps * 32 : 32;
  if (fisheye) {
    if (bin_smem_bytes > 48 * 1024) cudaFuncSetAttribute(k_bin<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bin_smem_bytes);
    k_bin<true><<<bin_grid, bin_threads, bin_smem_bytes, st>>>(rc, fm, fish, max_prims, max_pairs, err_flag);
  } else {
    if (bin_smem_bytes > 48 * 1024)   // cameras beyond ~640x480 (cbins > 1536): opt in to large dynamic shared memory
      cudaFuncSetAttribute(k_bin<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bin_smem_bytes);
    k_bin<false><<<bin_grid, bin_threads, bin_smem_bytes, st>>>(rc, fm, fish, max_prims, max_pairs, err_flag);
  }
  mark();
  const bool wrap = (rc.obs_layout | rc.obs_dtype) != 0;
  int launches = 5;
  if (!wrap && (W & 3) == 0) {   // (inside the k_raster event bracket: it is rasterisation time)
    const int solo_ctas = max(1, n_ctas * kSoloMinCtas / kRenderMinCtas);   // (n_ctas can be 1 for a handful of envs)
    if (fisheye) k_raster_solo<true><<<solo_ctas, 256, 0, st>>>(S, maps, rc, fm, fish, obs, max_prims, max_lat);
    else k_raster_solo<false><<<solo_ctas, 256, 0, st>>>(S, maps, rc, fm, fish, obs, max_prims, max_lat);
    launches++;
  }
  static bool smem_opt_in = false;
  if (!smem_opt_in) {   // > 48 KB of dynamic shared memory per CTA needs the opt-in, once per kernel
    cudaFuncSetAttribute(k_raster<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kRasterSmem);
    cudaFuncSetAttribute(k_raster<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kRasterSmem);
    cudaFuncSetAttribute(k_raster<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kRasterSmem);
    cudaFuncSetAttribute(k_raster<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kRasterSmem);
    smem_opt_in = true;
  }
  if (fisheye) {
    if (wrap) k_raster<true, true><<<n_ctas, kThreads, kRasterSmem, st>>>(S, maps, rc, fm, fish, gather, obs, max_prims, max_pairs, max_lat, err_flag);
    else k_raster<false, true><<<n_ctas, kThreads, kRasterSmem, st>>>(S, maps, rc, fm, fish, gather, obs, max_prims, max_pairs, max_lat, err_flag);
  } else {
    if (wrap) k_raster<true, false><<<n_ctas, kThreads, kRasterSmem, st>>>(S, maps, rc, fm, fish, gather, obs, max_prims, max_pairs, max_lat, err_flag);
    else k_raster<false, false><<<n_ctas, kThreads, kRasterSmem, st>>>(S, maps, rc, fm, fish, gather, obs, max_prims, max_pairs, max_lat, err_flag);
  }
  mark();
  mark();   // (post passes: none yet)
  return launches;
}

}  // namespace dts
