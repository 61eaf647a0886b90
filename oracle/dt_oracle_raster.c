/* dt_oracle_raster.c — CPU ORACLE (test infrastructure, NOT product code): software restatement
 * of what Simulator._render_img asks OpenGL to do (simulator.py:1707-1951, objects.py:123-148,
 * objmesh.py:360-375, graphics.py:172-251) plus the fisheye gather (distortion.py:85-125).
 *
 * PARITY UNPINNED for pixels: the reference's pixels come out of an OpenGL driver that cannot run
 * here (no pyglet/GL/display) and GL leaves rasterisation details implementation-defined.  This file
 * therefore DEFINES pixel truth for the project by fixing one deterministic interpretation of the
 * fixed-function pipeline (DESIGN.md "render spec"):
 *   - matrices in float64, rounded once to float32; vertex / lighting / clip / raster math in
 *     float32 with the exact operation order written below (built with -ffp-contract=off)
 *   - per-vertex (Gouraud) lighting, one light, GL_COLOR_MATERIAL ambient+diffuse, global ambient 0.3
 *   - clip against near/far and a 4x guard band, intersections computed from the inside vertex
 *   - vertices snapped to 1/64 px, integer edge functions, shared-edge ownership rule
 *   - 4x MSAA at (.375,.125)(.875,.375)(.125,.625)(.625,.875), colour shaded once per pixel centre,
 *     depth per sample, float32 depth, GL_LESS, draw order = reference draw order
 *   - bilinear RGBA8 textures, REPEAT wrap, GL_MODULATE
 *   - resolve = mean of 4 samples, u8 = rint(255*c), image row 0 = top
 *   - road tiles, two interpretations selectable with orr_set_tile_mode():
 *       0 "tessellated": the literal vertex list of simulator.py:386-507 — 7x7 quads = 98 triangles
 *         per tile, Gouraud colours interpolated per small triangle;
 *       1 "analytic" (DEFAULT, the parity spec): ONE quad (2 triangles) per tile for coverage, depth
 *         and uv, and the colour is the same piecewise-linear Gouraud interpolant of the 8x8 lit
 *         lattice evaluated at the pixel's (u,v).  Mathematically identical to mode 0 (perspective-
 *         correct interpolation is linear in tile coordinates and continuous across the interior
 *         edges); the two differ only by rounding and by <=1/64 px of edge placement on the tile
 *         outline (tests/test_oracle_raster.py quantifies it).  The tessellation exists in the
 *         reference only to approximate per-pixel lighting with fixed-function GL.
 * It is written for clarity (brute force over every triangle and every pixel of its bounding box),
 * not speed; the CUDA rasteriser is structured differently (binning, lattice sharing) and must
 * reproduce these numbers exactly.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "dt_oracle.h"


typedef struct { float cx, cy, cz, cw, r, g, b, u, v; } vtx; /* clip-space vertex with attributes */

typedef struct {
  int W, H;
  float* col;   /* [H][W][4 samples][3] */
  float* depth; /* [H][W][4] */
} framebuf;

static const int SX[4] = {24, 56, 8, 40}, SY[4] = {8, 24, 40, 56}; /* sample offsets in 1/64 px */
static int g_tile_mode = 1;
void orr_set_tile_mode(int mode) { g_tile_mode = mode; }
static int g_render_mode = 0; /* 1 = segment (S:1730-1733, 1752, 1808, 1814), 2 = top_down (S:1786-1798, 1923-1929) */
void orr_set_render_mode(int mode) { g_render_mode = mode; }
/* test-side statistics of the triangles handed to the rasteriser (single-threaded use): [0] set-up triangles on screen,
 * [1] of those with no sample position inside their bounding box, [2] with no covered sample, [3] pixel box <= 2x2,
 * [4] pixel box <= 4x4, [5] quads */
static __thread long long g_stats[8]; /* per thread: the OpenMP batch paths neither share nor contend on them */
void orr_stats_read(long long out[8], int reset) { for (int k = 0; k < 8; k++) { out[k] = g_stats[k]; if (reset) g_stats[k] = 0; } }
#define SEGMENT (g_render_mode & 1)
#define TOP_DOWN (g_render_mode & 2)

/* top_down=True: gluLookAt from (a, H, b) to (a, 0, b - 0.01), up +y (S:1786-1798) */
static void top_down_view(double grid_w, double grid_h, double tile_size, double fov_y_deg, double V[12]) {
  const double a = (grid_w * tile_size) / 2, b = (grid_h * tile_size) / 2;
  const double Hh = ((a > b ? a : b) + 0.1) / tan(fov_y_deg * 0.017453292519943295 / 2);
  const double ex = a, ey = Hh, ez = b;
  double fx = 0.0, fy = 0.0 - Hh, fz = (b - 0.01) - b;
  const double fn = sqrt(fx * fx + fy * fy + fz * fz);
  fx /= fn; fy /= fn; fz /= fn;
  double sx = fy * 0.0 - fz * 1.0, sy = fz * 0.0 - fx * 0.0, sz = fx * 1.0 - fy * 0.0;
  const double sn = sqrt(sx * sx + sy * sy + sz * sz);
  sx /= sn; sy /= sn; sz /= sn;
  const double ux = sy * fz - sz * fy, uy = sz * fx - sx * fz, uz = sx * fy - sy * fx;
  const double L[12] = {sx, sy, sz, -(sx * ex + sy * ey + sz * ez), ux, uy, uz, -(ux * ex + uy * ey + uz * ez),
                        -fx, -fy, -fz, (fx * ex + fy * ey + fz * ez)};
  for (int k = 0; k < 12; k++) V[k] = L[k];
}
#define GUARD 4.0f

/* ---- camera (simulator.py:1758-1803), float64 ------------------------------------------------ */
static void camera_view(double px, double pz, double angle, const orr_episode* ep, int domain_rand, double V[12]) {
  double ex = px, ey = 0.0, ez = pz;
  if (domain_rand) { ex += (double)ep->cam_noise[0]; ey += (double)ep->cam_noise[1]; ez += (double)ep->cam_noise[2]; }
  ey += (double)ep->cam_height;
  double fx = cos(angle), fy = 0.0, fz = -sin(angle);
  double fn = sqrt(fx * fx + fy * fy + fz * fz);
  fx /= fn; fy /= fn; fz /= fn;
  double sx = fy * 0.0 - fz * 1.0, sy = fz * 0.0 - fx * 0.0, sz = fx * 1.0 - fy * 0.0;
  double sn = sqrt(sx * sx + sy * sy + sz * sz);
  sx /= sn; sy /= sn; sz /= sn;
  double ux = sy * fz - sz * fy, uy = sz * fx - sx * fz, uz = sx * fy - sy * fx;
  double L[12] = {sx, sy, sz, -(sx * ex + sy * ey + sz * ez), ux, uy, uz, -(ux * ex + uy * ey + uz * ez),
                  -fx, -fy, -fz, (fx * ex + fy * ey + fz * ez)};
  L[11] += (double)0.066f; /* glTranslatef(0, 0, CAMERA_FORWARD_DIST): a GLfloat argument */
  double th = (double)ep->cam_angle_deg * 0.017453292519943295;
  double c = cos(th), s = sin(th);
  for (int k = 0; k < 4; k++) {
    V[k] = L[k];
    V[4 + k] = c * L[4 + k] - s * L[8 + k];
    V[8 + k] = s * L[4 + k] + c * L[8 + k];
  }
}

/* MV = V * T(t) * S(s) * Ry(c,s_) ; N = rot(V) * Ry / s   (both rounded to float32) */
static void model_view(const double V[12], const double t[3], double sc, double c, double s, float MV[12], float N[9]) {
  /* Ry = [[c,0,s],[0,1,0],[-s,0,c]] (glRotatef about +y) */
  double R[9] = {c, 0, s, 0, 1, 0, -s, 0, c};
  for (int r = 0; r < 3; r++) {
    for (int k = 0; k < 3; k++) {
      double a = V[4 * r + 0] * R[0 + k] + V[4 * r + 1] * R[3 + k] + V[4 * r + 2] * R[6 + k];
      MV[4 * r + k] = (float)(a * sc);
      N[3 * r + k] = (float)(a / sc);
    }
    MV[4 * r + 3] = (float)(V[4 * r + 0] * t[0] + V[4 * r + 1] * t[1] + V[4 * r + 2] * t[2] + V[4 * r + 3]);
  }
}

typedef struct {
  float MV[12], N[9];
  float P00, P11, P22, P23;
  const orr_episode* ep;
} xform;

/* object-space vertex -> lit clip-space vertex (fixed-function T&L, float32, no FMA) */
static vtx shade_vertex(const xform* x, const float p[3], const float n[3], const float col[3], float u, float v) {
  const float* M = x->MV;
  float e[3], ne[3];
  for (int r = 0; r < 3; r++) {
    float t = M[4 * r] * p[0];
    t = t + M[4 * r + 1] * p[1];
    t = t + M[4 * r + 2] * p[2];
    e[r] = t + M[4 * r + 3];
    float q = x->N[3 * r] * n[0];
    q = q + x->N[3 * r + 1] * n[1];
    ne[r] = q + x->N[3 * r + 2] * n[2];
  }
  const float* lp = x->ep->light_eye;
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
  vtx o;
  float lit[3];
  for (int k = 0; k < 3; k++) {
    float s = 0.3f + x->ep->ambient[k];
    s = s + ndl * x->ep->diffuse[k];
    float c = SEGMENT ? col[k] : col[k] * s; /* segment=True: GL_LIGHTING off, the vertex colour is the material colour */
    lit[k] = c < 0.0f ? 0.0f : (c > 1.0f ? 1.0f : c);
  }
  o.r = lit[0]; o.g = lit[1]; o.b = lit[2];
  o.u = u; o.v = v;
  o.cx = x->P00 * e[0];
  o.cy = x->P11 * e[1];
  o.cz = x->P22 * e[2] + x->P23;
  o.cw = -e[2];
  return o;
}

static float plane_dist(const vtx* a, int pl) {
  switch (pl) {
    case 0: return a->cz + a->cw;          /* near:  z >= -w */
    case 1: return a->cw - a->cz;          /* far:   z <=  w */
    case 2: return a->cx + GUARD * a->cw;  /* x >= -G w */
    case 3: return GUARD * a->cw - a->cx;
    case 4: return a->cy + GUARD * a->cw;
    default: return GUARD * a->cw - a->cy;
  }
}
/* point on the edge from the INSIDE vertex `in` towards the OUTSIDE vertex `out` */
static vtx clip_lerp(const vtx* in, const vtx* out, float din, float dout) {
  float t = din / (din - dout);
  vtx o;
  const float* a = (const float*)in; const float* b = (const float*)out; float* c = (float*)&o;
  for (int k = 0; k < 9; k++) { float d = b[k] - a[k]; c[k] = a[k] + t * d; }
  return o;
}
static int clip_polygon(vtx* poly, int n) {
  vtx tmp[12];
  for (int pl = 0; pl < 6; pl++) {
    int m = 0, any_out = 0;
    float d[12];
    for (int k = 0; k < n; k++) { d[k] = plane_dist(&poly[k], pl); if (!(d[k] >= 0.0f)) any_out = 1; }
    if (!any_out) continue;
    for (int k = 0; k < n; k++) {
      int k2 = (k + 1) % n;
      int in1 = d[k] >= 0.0f, in2 = d[k2] >= 0.0f;
      if (in1) tmp[m++] = poly[k];
      if (in1 && !in2) tmp[m++] = clip_lerp(&poly[k], &poly[k2], d[k], d[k2]);
      else if (!in1 && in2) tmp[m++] = clip_lerp(&poly[k2], &poly[k], d[k2], d[k]);
    }
    n = m;
    memcpy(poly, tmp, sizeof(vtx) * n);
    if (n < 3) return 0;
  }
  return n;
}

static inline float tex_byte(const orr_texture* t, int i, int j, int c) { return (float)t->rgba[((size_t)j * t->w + i) * 4 + c]; }

/* one screen-space triangle (already clipped); `id` only documents draw order (drawn in order, GL_LESS) */
/* Rasterise triangle (a,b,c) — or, with `d`, the QUAD a,b,c,d of an unclipped road tile (spec tile mode 1):
 * attribute planes of triangle (a,b,c), coverage by the quad's four edges.  Returns 0 without drawing when the
 * snapped quad is not strictly convex: the caller then draws (a,b,c)(a,c,d). */
static int raster_triangle(framebuf* fb, vtx a, vtx b, vtx c, const orr_texture* tex, const float* lat, const vtx* d) {
  vtx* vs[3] = {&a, &b, &c};
  int X[3], Y[3];
  float zw[3], q[3];
  const float Wf = (float)fb->W, Hf = (float)fb->H;
  for (int k = 0; k < 3; k++) {
    float iw = 1.0f / vs[k]->cw;
    float nx = vs[k]->cx * iw, ny = vs[k]->cy * iw, nz = vs[k]->cz * iw;
    float sx = (nx * 0.5f + 0.5f) * Wf;
    float sy = (0.5f - ny * 0.5f) * Hf;
    X[k] = (int)rintf(sx * 64.0f);
    Y[k] = (int)rintf(sy * 64.0f);
    zw[k] = nz * 0.5f + 0.5f;
    q[k] = iw;
  }
  int64_t area2 = (int64_t)(X[1] - X[0]) * (Y[2] - Y[0]) - (int64_t)(X[2] - X[0]) * (Y[1] - Y[0]);
  if (area2 == 0) return 0;
  int i0 = 0, i1 = 1, i2 = 2;
  if (area2 < 0) { i1 = 2; i2 = 1; }
  const int ix[3] = {i0, i1, i2};
  int x0 = X[i0], y0 = Y[i0], x1 = X[i1], y1 = Y[i1], x2 = X[i2], y2 = Y[i2];
  /* polygon in positive orientation, edge k: vertex k -> k+1 ; E(x,y) = (xb-xa)(y-ya) - (yb-ya)(x-xa) >= 0 inside */
  int nv = 3, qx[4] = {x0, x1, x2, 0}, qy[4] = {y0, y1, y2, 0};
  if (d) {
    float iw = 1.0f / d->cw;
    float sx = ((d->cx * iw) * 0.5f + 0.5f) * Wf, sy = (0.5f - (d->cy * iw) * 0.5f) * Hf;
    int X3 = (int)rintf(sx * 64.0f), Y3 = (int)rintf(sy * 64.0f);
    nv = 4;
    if (area2 > 0) { qx[1] = X[1]; qy[1] = Y[1]; qx[2] = X[2]; qy[2] = Y[2]; qx[3] = X3; qy[3] = Y3; }   /* a b c d */
    else { qx[1] = X3; qy[1] = Y3; qx[2] = X[2]; qy[2] = Y[2]; qx[3] = X[1]; qy[3] = Y[1]; }             /* a d c b */
    for (int k = 0; k < 4; k++) { /* strictly convex */
      int k1 = (k + 1) & 3, k2 = (k + 2) & 3;
      int64_t cr = (int64_t)(qx[k1] - qx[k]) * (qy[k2] - qy[k1]) - (int64_t)(qx[k2] - qx[k1]) * (qy[k1] - qy[k]);
      if (cr <= 0) return 0;
    }
  }
  int ax[4], ay[4], bx[4], by[4], bias[4];
  for (int k = 0; k < nv; k++) {
    int k1 = (k + 1) % nv;
    ax[k] = qx[k]; ay[k] = qy[k]; bx[k] = qx[k1]; by[k] = qy[k1];
    int dx = bx[k] - ax[k], dy = by[k] - ay[k];
    bias[k] = (dy > 0 || (dy == 0 && dx < 0)) ? 0 : 1;  /* non-owner edges exclude E == 0 */
  }
  /* attribute planes anchored at v0 (float32) */
  const float dx1 = (float)(x1 - x0) * 0.015625f, dy1 = (float)(y1 - y0) * 0.015625f;
  const float dx2 = (float)(x2 - x0) * 0.015625f, dy2 = (float)(y2 - y0) * 0.015625f;
  const float areaf = dx1 * dy2 - dx2 * dy1;
  const float ia = 1.0f / areaf;
  float f0[7], fx[7], fy[7]; /* z, q, u*q, v*q, r*q, g*q, b*q */
  for (int at = 0; at < 7; at++) {
    float v[3];
    for (int k = 0; k < 3; k++) {
      const vtx* p = vs[ix[k]];
      float qq = q[ix[k]];
      switch (at) {
        case 0: v[k] = zw[ix[k]]; break;
        case 1: v[k] = qq; break;
        case 2: v[k] = p->u * qq; break;
        case 3: v[k] = p->v * qq; break;
        case 4: v[k] = p->r * qq; break;
        case 5: v[k] = p->g * qq; break;
        default: v[k] = p->b * qq; break;
      }
    }
    float d1 = v[1] - v[0], d2 = v[2] - v[0];
    f0[at] = v[0];
    fx[at] = (d1 * dy2 - d2 * dy1) * ia;
    fy[at] = (d2 * dx1 - d1 * dx2) * ia;
  }
  int minx = x0 < x1 ? x0 : x1; minx = minx < x2 ? minx : x2;
  int maxx = x0 > x1 ? x0 : x1; maxx = maxx > x2 ? maxx : x2;
  int miny = y0 < y1 ? y0 : y1; miny = miny < y2 ? miny : y2;
  int maxy = y0 > y1 ? y0 : y1; maxy = maxy > y2 ? maxy : y2;
  if (nv == 4) {
    int X3 = area2 > 0 ? qx[3] : qx[1], Y3 = area2 > 0 ? qy[3] : qy[1];
    minx = minx < X3 ? minx : X3; maxx = maxx > X3 ? maxx : X3;
    miny = miny < Y3 ? miny : Y3; maxy = maxy > Y3 ? maxy : Y3;
  }
  int px0 = minx >> 6, px1 = maxx >> 6, py0 = miny >> 6, py1 = maxy >> 6;
  if (px0 < 0) px0 = 0;
  if (py0 < 0) py0 = 0;
  if (px1 >= fb->W) px1 = fb->W - 1;
  if (py1 >= fb->H) py1 = fb->H - 1;
  int any_cov = 0;
  if (px0 <= px1 && py0 <= py1) {
    g_stats[0]++;
    if (nv == 4) g_stats[5]++;
    int has = 0;
    for (int s = 0; s < 4; s++) {
      /* pixels p with minx <= 64 p + SX <= maxx, and the same in y, for the SAME sample index */
      int lo = minx - SX[s], hi = maxx - SX[s], lo2 = miny - SY[s], hi2 = maxy - SY[s];
      int pxl = (lo + 63) >> 6, pxh = hi >> 6, pyl = (lo2 + 63) >> 6, pyh = hi2 >> 6;
      if (pxl < 0) pxl = 0;
      if (pyl < 0) pyl = 0;
      if (pxh >= fb->W) pxh = fb->W - 1;
      if (pyh >= fb->H) pyh = fb->H - 1;
      if (pxl <= pxh && pyl <= pyh) has = 1;
    }
    if (!has) g_stats[1]++;
    if (px1 - px0 < 2 && py1 - py0 < 2) g_stats[3]++;
    if (px1 - px0 < 4 && py1 - py0 < 4) g_stats[4]++;
  }
  for (int py = py0; py <= py1; py++)
    for (int px = px0; px <= px1; px++) {
      int mask = 0;
      for (int s = 0; s < 4; s++) {
        int sx = px * 64 + SX[s], sy = py * 64 + SY[s];
        int inside = 1;
        for (int k = 0; k < nv; k++) {
          int64_t E = (int64_t)(bx[k] - ax[k]) * (sy - ay[k]) - (int64_t)(by[k] - ay[k]) * (sx - ax[k]);
          if (E - bias[k] < 0) inside = 0;
        }
        if (inside) mask |= 1 << s;
      }
      if (!mask) continue;
      any_cov = 1;
      /* shade once at the pixel centre */
      const float cdx = (float)(px * 64 + 32 - x0) * 0.015625f, cdy = (float)(py * 64 + 32 - y0) * 0.015625f;
      float at[7];
      for (int k = 1; k < 7; k++) at[k] = fmaf(fy[k], cdy, fmaf(fx[k], cdx, f0[k]));
      float qq = at[1];
      if (!(qq > 1e-20f)) qq = 1e-20f;
      const float rq = 1.0f / qq;
      const float u = at[2] * rq, v = at[3] * rq;
      float lit[3] = {at[4] * rq, at[5] * rq, at[6] * rq};
      if (lat) { /* analytic tile: Gouraud interpolant of the lit 8x8 lattice at (u,v); lattice index a <-> u,
                  * b <-> 1-v (S:394-401); cell split (0,1,2)(0,2,3) as drawn */
        float fa_ = u * 7.0f, fb_ = (1.0f - v) * 7.0f;
        int ia = (int)floorf(fa_), ib = (int)floorf(fb_);
        ia = ia < 0 ? 0 : (ia > 6 ? 6 : ia);
        ib = ib < 0 ? 0 : (ib > 6 ? 6 : ib);
        float fa = fa_ - (float)ia, fb = fb_ - (float)ib;
        const float* c00 = lat + (ia * 8 + ib) * 3;
        const float* c10 = lat + ((ia + 1) * 8 + ib) * 3;
        const float* c11 = lat + ((ia + 1) * 8 + ib + 1) * 3;
        const float* c01 = lat + (ia * 8 + ib + 1) * 3;
        for (int ch = 0; ch < 3; ch++)
          lit[ch] = (fb <= fa) ? fmaf(fb, c11[ch] - c10[ch], fmaf(fa, c10[ch] - c00[ch], c00[ch]))
                               : fmaf(fa, c11[ch] - c01[ch], fmaf(fb, c01[ch] - c00[ch], c00[ch]));
      }
      float colr[3];
      if (tex) {
        float tx = u * (float)tex->w - 0.5f, ty = v * (float)tex->h - 0.5f;
        float txf = floorf(tx), tyf = floorf(ty);
        float ffx = tx - txf, ffy = ty - tyf;
        int ti0 = ((int)txf) & (tex->w - 1), ti1 = (ti0 + 1) & (tex->w - 1);
        int tj0 = ((int)tyf) & (tex->h - 1), tj1 = (tj0 + 1) & (tex->h - 1);
        for (int ch = 0; ch < 3; ch++) {
          float t00 = tex_byte(tex, ti0, tj0, ch), t10 = tex_byte(tex, ti1, tj0, ch);
          float t01 = tex_byte(tex, ti0, tj1, ch), t11 = tex_byte(tex, ti1, tj1, ch);
          float ta = fmaf(ffx, t10 - t00, t00);
          float tb = fmaf(ffx, t11 - t01, t01);
          float tc = fmaf(ffy, tb - ta, ta);
          colr[ch] = tc * (lit[ch] * 0.00392156862745098f);
        }
      } else { colr[0] = lit[0]; colr[1] = lit[1]; colr[2] = lit[2]; }
      for (int s = 0; s < 4; s++) {
        if (!(mask >> s & 1)) continue;
        const float sdx = (float)(px * 64 + SX[s] - x0) * 0.015625f, sdy = (float)(py * 64 + SY[s] - y0) * 0.015625f;
        const float z = fmaf(fy[0], sdy, fmaf(fx[0], sdx, f0[0]));
        size_t si = ((size_t)py * fb->W + px) * 4 + s;
        if (z < fb->depth[si]) {
          fb->depth[si] = z;
          fb->col[si * 3] = colr[0]; fb->col[si * 3 + 1] = colr[1]; fb->col[si * 3 + 2] = colr[2];
        }
      }
    }
  if (px0 <= px1 && py0 <= py1 && !any_cov) g_stats[2]++;
  return 1;
}

/* 0 = visible without clipping, 1 = needs the clipper, 2 = outside one true-frustum plane (invisible) */
static int classify3(const vtx* a, const vtx* b, const vtx* c) {
  const vtx* v[3] = {a, b, c};
  int out[6] = {0, 0, 0, 0, 0, 0}, need = 0;
  for (int k = 0; k < 3; k++) {
    float x = v[k]->cx, y = v[k]->cy, z = v[k]->cz, w = v[k]->cw;
    out[0] += !(z + w >= 0.0f); out[1] += !(w - z >= 0.0f);
    out[2] += x < -w; out[3] += x > w; out[4] += y < -w; out[5] += y > w;
    need |= !(x + GUARD * w >= 0.0f) | !(GUARD * w - x >= 0.0f) | !(y + GUARD * w >= 0.0f) | !(GUARD * w - y >= 0.0f);
  }
  need |= out[0] | out[1];
  for (int p = 0; p < 6; p++) if (out[p] == 3) return 2;
  return need ? 1 : 0;
}

static void draw_shaded(framebuf* fb, vtx a, vtx b, vtx c, const orr_texture* tex, const float* lat);
static void draw_triangle(framebuf* fb, const xform* x, const float* p, const float* n, const float* uv, const float* col,
                          const orr_texture* tex) {
  vtx v[3];
  for (int k = 0; k < 3; k++) v[k] = shade_vertex(x, p + 3 * k, n + 3 * k, col + 3 * k, uv[2 * k], uv[2 * k + 1]);
  draw_shaded(fb, v[0], v[1], v[2], tex, 0);
}
static void draw_shaded(framebuf* fb, vtx a, vtx b, vtx c, const orr_texture* tex, const float* lat) {
  vtx poly[12];
  poly[0] = a; poly[1] = b; poly[2] = c;
  /* trivial reject: all three outside one plane */
  for (int pl = 0; pl < 6; pl++) {
    int out = 0;
    for (int k = 0; k < 3; k++) out += !(plane_dist(&poly[k], pl) >= 0.0f);
    if (out == 3) return;
  }
  int m = clip_polygon(poly, 3);
  for (int k = 1; k + 1 < m; k++) raster_triangle(fb, poly[0], poly[k], poly[k + 1], tex, lat, NULL);
}

/* Render one env. out: u8 [H][W][3], row 0 = top.  lut_x/lut_y: NULL or fisheye LUT [H][W]. */
void orr_render(const orr_scene* sc, double px, double pz, double angle, const orr_episode* ep, int W, int H,
                int domain_rand, const float* lut_x, const float* lut_y, uint8_t* out) {
  /* per-thread sample buffers, kept across frames (a malloc/free of ~1 MB per frame turns into
   * mmap/munmap + page faults and serialises the OpenMP batch) */
  static _Thread_local float* tl_col = 0;
  static _Thread_local float* tl_depth = 0;
  static _Thread_local size_t tl_px = 0;
  if (tl_px < (size_t)W * H) {
    free(tl_col); free(tl_depth);
    tl_px = (size_t)W * H;
    tl_col = (float*)malloc(sizeof(float) * tl_px * 12);
    tl_depth = (float*)malloc(sizeof(float) * tl_px * 4);
  }
  framebuf fb;
  fb.W = W; fb.H = H;
  fb.col = tl_col;
  fb.depth = tl_depth;
  const float clear[3] = {SEGMENT ? 1.0f : ep->horizon[0], SEGMENT ? 0.0f : ep->horizon[1], SEGMENT ? 1.0f : ep->horizon[2]};
  for (size_t k = 0; k < (size_t)W * H * 4; k++) {  /* glClear S:1753-1756; segment: glClearColor(255, 0, 255) clamps to magenta */
    fb.depth[k] = 1.0f;
    fb.col[3 * k] = clear[0]; fb.col[3 * k + 1] = clear[1]; fb.col[3 * k + 2] = clear[2];
  }
  double V[12];
  if (TOP_DOWN) top_down_view((double)sc->grid_w, (double)sc->grid_h, sc->tile_size, (double)ep->cam_fov_y_deg, V);
  else camera_view(px, pz, angle, ep, domain_rand, V);
  xform x;
  x.ep = ep;
  {  /* gluPerspective(fovy, W/H, 0.04, 100) S:1761 */
    double f = 1.0 / tan((double)ep->cam_fov_y_deg * 0.017453292519943295 / 2.0), aspect = (double)W / (double)H;
    double zn = 0.04, zf = 100.0;
    x.P00 = (float)(f / aspect); x.P11 = (float)f;
    x.P22 = (float)((zf + zn) / (zn - zf)); x.P23 = (float)(2.0 * zf * zn / (zn - zf));
  }
  const double zero3[3] = {0, 0, 0};
  /* 1. ground quad S:1805-1812: glScalef(50,0.01,50) of (+-1,-0.8,+-1); colour ground_color; normal fixed to
   *    unit +y in world space (the reference leaves it undefined, SURVEY R2) */
  {
    model_view(V, zero3, 1.0, 1.0, 0.0, x.MV, x.N);
    const float gy = (float)(-0.8 * 0.01);
    const float P[4][3] = {{-50.f, gy, 50.f}, {-50.f, gy, -50.f}, {50.f, gy, -50.f}, {50.f, gy, 50.f}};
    const float nrm[9] = {0, 1, 0, 0, 1, 0, 0, 1, 0}, uv[6] = {0, 0, 0, 0, 0, 0};
    float col[9];
    const float magenta[3] = {255.f, 0.f, 255.f}; /* glColor3f(255, 0, 255) S:1808 */
    const float* gc = SEGMENT ? magenta : ep->ground;
    for (int k = 0; k < 3; k++) { col[k] = gc[k]; col[3 + k] = gc[k]; col[6 + k] = gc[k]; }
    const int tri[2][3] = {{0, 1, 2}, {0, 2, 3}};
    for (int t = 0; t < 2; t++) {
      float p[9];
      for (int k = 0; k < 3; k++) memcpy(p + 3 * k, P[tri[t][k]], 12);
      draw_triangle(&fb, &x, p, nrm, uv, col, NULL);
    }
  }
  /* 2. road tiles S:1852-1884, vertex list S:386-507: i outer, j inner; 7x7 quads, (0,1,2)(0,2,3) split */
  const double ts = sc->tile_size;
  float lat[8];
  for (int k = 0; k < 8; k++) lat[k] = (float)(-ts / 2 + ((double)k / 7.0) * ts);
  for (int i = 0; i < sc->grid_w; i++)
    for (int j = 0; j < sc->grid_h; j++) {
      int idx = j * sc->grid_w + i;
      if (sc->tile_kind[idx] < 0) continue;
      /* glRotatef(angle*90+180, 0,1,0): multiples of 90 degrees -> exact cos/sin */
      int quarter = (sc->tile_angle[idx] + 2) & 3;
      const double cs[4] = {1, 0, -1, 0}, sn[4] = {0, 1, 0, -1};
      /* glTranslatef((i + 0.5) * TS, 0, (j + 0.5) * TS) S:1870: GLfloat arguments */
      const double t[3] = {(double)(float)((i + 0.5) * ts), 0.0, (double)(float)((j + 0.5) * ts)};
      model_view(V, t, 1.0, cs[quarter], sn[quarter], x.MV, x.N);
      int tile_tex = sc->tile_tex[idx];
      if (SEGMENT && tile_tex >= 0 && sc->tex_segment) tile_tex = sc->tex_segment[tile_tex];
      const orr_texture* tex = tile_tex >= 0 ? &sc->textures[tile_tex] : NULL;
      const float white[9] = {1, 1, 1, 1, 1, 1, 1, 1, 1}, up[9] = {0, 1, 0, 0, 1, 0, 0, 1, 0};
      if (g_tile_mode == 1) {
        /* analytic: light the 8x8 lattice once, draw the tile as one quad (0,1,2)(0,2,3) */
        float lat_rgb[64 * 3];
        vtx corner[4];
        const int ca[4] = {0, 7, 7, 0}, cb[4] = {0, 0, 7, 7};
        for (int a = 0; a < 8; a++)
          for (int b = 0; b < 8; b++) {
            const float p[3] = {lat[a], 0.0f, lat[b]};
            vtx v = shade_vertex(&x, p, up, white, (float)((double)a / 7.0), (float)(1.0 - (double)b / 7.0));
            lat_rgb[(a * 8 + b) * 3] = v.r; lat_rgb[(a * 8 + b) * 3 + 1] = v.g; lat_rgb[(a * 8 + b) * 3 + 2] = v.b;
            for (int k = 0; k < 4; k++) if (a == ca[k] && b == cb[k]) corner[k] = v;
          }
        for (int k = 0; k < 4; k++) { corner[k].r = 0.0f; corner[k].g = 0.0f; corner[k].b = 0.0f; }
        /* a tile that needs no clipping is ONE quad prim; otherwise (or if the snapped quad is not convex) two triangles */
        if (classify3(&corner[0], &corner[1], &corner[2]) == 0 && classify3(&corner[0], &corner[2], &corner[3]) == 0 &&
            raster_triangle(&fb, corner[0], corner[1], corner[2], tex, lat_rgb, &corner[3]))
          continue;
        draw_shaded(&fb, corner[0], corner[1], corner[2], tex, lat_rgb);
        draw_shaded(&fb, corner[0], corner[2], corner[3], tex, lat_rgb);
        continue;
      }
      for (int a = 0; a < 7; a++)
        for (int b = 0; b < 7; b++) {
          const int qa[4] = {a, a + 1, a + 1, a}, qb[4] = {b, b, b + 1, b + 1};
          const int tri[2][3] = {{0, 1, 2}, {0, 2, 3}};
          for (int tt = 0; tt < 2; tt++) {
            float p[9], uv[6];
            for (int k = 0; k < 3; k++) {
              int u_ = qa[tri[tt][k]], v_ = qb[tri[tt][k]];
              p[3 * k] = lat[u_]; p[3 * k + 1] = 0.0f; p[3 * k + 2] = lat[v_];
              uv[2 * k] = (float)((double)u_ / 7.0);
              uv[2 * k + 1] = (float)(1.0 - (double)v_ / 7.0);
            }
            draw_triangle(&fb, &x, p, up, uv, white, tex);
          }
        }
    }
  /* 3. objects S:1905-1907, O:123-148, M:360-375; top-down views then draw the agent's own mesh at cur_pos (S:1923-1929) */
  for (int o = 0; o <= sc->n_objects; o++) {
    orr_object agent = sc->agent;
    const orr_object* ob;
    if (o < sc->n_objects) {
      if (ep->hidden[o >> 5] >> (o & 31) & 1u) continue;
      ob = &sc->objects[o];
    } else {
      if (!TOP_DOWN || sc->agent.tri_count == 0) break;
      agent.pos[0] = (float)px; agent.pos[1] = 0.0f; agent.pos[2] = (float)pz;   /* glTranslatef(*cur_pos) */
      agent.scale = 1.0f;
      agent.y_rot_deg = (float)(angle * 180.0 / 3.141592653589793);              /* glRotatef(cur_angle * 180 / pi, 0, 1, 0) */
      ob = &agent;
    }
    const double t[3] = {ob->pos[0], ob->pos[1], ob->pos[2]};
    const double th = (double)ob->y_rot_deg * 0.017453292519943295;
    model_view(V, t, (double)ob->scale, cos(th), sin(th), x.MV, x.N);
    for (int k = 0; k < ob->tri_count; k++) {
      size_t ti = (size_t)ob->tri_offset + k;
      int tid = sc->tri_tex[ti];
      if (tid >= 0 && tid == ob->tex_from) tid = ob->tex_to;   /* TrafficLightObj card swap O:453,462 */
      if (SEGMENT) tid = ob->seg_tex;                          /* get_mesh(name, segment=True): flat class colour M:268-290 */
      const orr_texture* tex = tid >= 0 ? &sc->textures[tid] : NULL;
      draw_triangle(&fb, &x, sc->tri_pos + ti * 9, sc->tri_nrm + ti * 9, sc->tri_uv + ti * 6, sc->tri_col + ti * 9, tex);
    }
  }
  /* 4. resolve + readback S:1931-1949 (+ fused fisheye gather distortion.py:118) */
  for (int y = 0; y < H; y++)
    for (int xx = 0; xx < W; xx++) {
      int sx = xx, sy = y, valid = 1;
      if (lut_x) {
        const float fx = lut_x[(size_t)y * W + xx], fy = lut_y[(size_t)y * W + xx];
        /* NaN, +-inf and |v| >= 2^31 have no int value (the cast would be undefined): outside */
        valid = fabsf(fx) < 2147483648.0f && fabsf(fy) < 2147483648.0f;
        if (valid) {
          sx = (int)rintf(fx);
          sy = (int)rintf(fy);
          valid = sx >= 0 && sx < W && sy >= 0 && sy < H;  /* cv2.remap BORDER_CONSTANT -> 0 */
        }
      }
      for (int ch = 0; ch < 3; ch++) {
        uint8_t v = 0;
        if (valid) {
          const float* s = fb.col + ((size_t)sy * W + sx) * 12 + ch;
          float c = ((s[0] + s[3]) + (s[6] + s[9])) * 0.25f;
          c = c < 0.0f ? 0.0f : (c > 1.0f ? 1.0f : c);
          v = (uint8_t)rintf(c * 255.0f);
        }
        out[((size_t)y * W + xx) * 3 + ch] = v;
      }
    }
}

/* Test hook for the GL call-trace golden (tests/golden/gltrace_*.npz): the transforms and the lit tile lattices this
 * renderer uses for one frame.  item 0 = ground, 1.. = every grid cell in draw order (i outer, j inner; absent tiles
 * zero), then the objects.  item_mv [items][12], item_n [items][9], lattice [cells][64][3] (a outer, b inner). */
void orr_debug_frame(const orr_scene* sc, double px, double pz, double angle, const orr_episode* ep, int W, int H,
                     int domain_rand, double* V_out, float* P_out, float* item_mv, float* item_n, float* lattice) {
  double V[12];
  if (TOP_DOWN) top_down_view((double)sc->grid_w, (double)sc->grid_h, sc->tile_size, (double)ep->cam_fov_y_deg, V);
  else camera_view(px, pz, angle, ep, domain_rand, V);
  memcpy(V_out, V, sizeof V);
  xform x;
  x.ep = ep;
  {
    double f = 1.0 / tan((double)ep->cam_fov_y_deg * 0.017453292519943295 / 2.0), aspect = (double)W / (double)H;
    double zn = 0.04, zf = 100.0;
    x.P00 = (float)(f / aspect); x.P11 = (float)f;
    x.P22 = (float)((zf + zn) / (zn - zf)); x.P23 = (float)(2.0 * zf * zn / (zn - zf));
    P_out[0] = x.P00; P_out[1] = x.P11; P_out[2] = x.P22; P_out[3] = x.P23;
  }
  const double zero3[3] = {0, 0, 0};
  int item = 0;
  model_view(V, zero3, 1.0, 1.0, 0.0, x.MV, x.N);
  memcpy(item_mv, x.MV, 48); memcpy(item_n, x.N, 36);
  item++;
  const double ts = sc->tile_size;
  float lat[8];
  for (int k = 0; k < 8; k++) lat[k] = (float)(-ts / 2 + ((double)k / 7.0) * ts);
  for (int i = 0; i < sc->grid_w; i++)
    for (int j = 0; j < sc->grid_h; j++, item++) {
      int idx = j * sc->grid_w + i;
      float* L = lattice + (size_t)(item - 1) * 64 * 3;
      memset(item_mv + 12 * item, 0, 48); memset(item_n + 9 * item, 0, 36); memset(L, 0, 64 * 3 * 4);
      if (sc->tile_kind[idx] < 0) continue;
      int quarter = (sc->tile_angle[idx] + 2) & 3;
      const double cs[4] = {1, 0, -1, 0}, sn[4] = {0, 1, 0, -1};
      const double t[3] = {(double)(float)((i + 0.5) * ts), 0.0, (double)(float)((j + 0.5) * ts)};
      model_view(V, t, 1.0, cs[quarter], sn[quarter], x.MV, x.N);
      memcpy(item_mv + 12 * item, x.MV, 48); memcpy(item_n + 9 * item, x.N, 36);
      const float white[3] = {1, 1, 1}, up[3] = {0, 1, 0};
      for (int a = 0; a < 8; a++)
        for (int b = 0; b < 8; b++) {
          const float p[3] = {lat[a], 0.0f, lat[b]};
          vtx v = shade_vertex(&x, p, up, white, 0.f, 0.f);
          L[(a * 8 + b) * 3] = v.r; L[(a * 8 + b) * 3 + 1] = v.g; L[(a * 8 + b) * 3 + 2] = v.b;
        }
    }
  for (int o = 0; o < sc->n_objects; o++, item++) {
    const orr_object* ob = &sc->objects[o];
    const double t[3] = {ob->pos[0], ob->pos[1], ob->pos[2]};
    const double th = (double)ob->y_rot_deg * 0.017453292519943295;
    model_view(V, t, (double)ob->scale, cos(th), sin(th), x.MV, x.N);
    memcpy(item_mv + 12 * item, x.MV, 48); memcpy(item_n + 9 * item, x.N, 36);
  }
}

/* batch over envs (OpenMP): the cpu_baseline / --impl reference leg of bench.py */
void orr_render_batch(const orr_scene* sc, int n, const double* px, const double* pz, const double* angle,
                      const orr_episode* eps, int W, int H, int domain_rand, const float* lut_x, const float* lut_y,
                      uint8_t* out, int threads) {
#pragma omp parallel for schedule(dynamic, 1) num_threads(threads)
  for (int e = 0; e < n; e++)
    orr_render(sc, px[e], pz[e], angle[e], &eps[e], W, H, domain_rand, lut_x, lut_y, out + (size_t)e * W * H * 3);
}
