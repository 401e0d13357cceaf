// Pillow's polygon fill (ImageDraw.polygon(xy, fill=1) on a mode-F image, Pillow 12.2) for one four-corner polygon,
// one scan line at a time.  Used by box_raster_kernel (boxes.cu).  These rules were established from Pillow's output,
// not from its source, and are pinned by tests/test_box_raster_gpu.py against Pillow itself:
//   * vertices are truncated toward zero to int;
//   * edges are built as ImagingDrawPolygon does: a horizontal segment that continues the previous horizontal segment in
//     the same x direction extends it; the closing edge is added only when the last vertex differs from the first;
//   * horizontal edges are drawn as whole lines [xmin, xmax] on their row;
//   * every other edge crosses row y (ymin <= y <= ymax) at x = float((y - y0) * dx + x0), dx = float(x1 - x0) / (y1 - y0),
//     each operation rounded separately; an edge ending at row y below the polygon's last row contributes x twice;
//   * "corner" rule: an edge that crosses row y at its own end point, at an integral x, with dx != 0, looks through the
//     earlier edges that also end on row y.  The first such edge with exactly the same x decides: if its dx has the
//     other sign, nothing happens; else, when the other edge also covers row y + o (o = -1 at the current edge's lower
//     end, +1 otherwise), a = the current edge's x and b = the other's on row y + o, and x lies more than one pixel beyond
//     both, x moves to roundf(max(a, b)) + 1 (x to the right) or roundf(min(a, b)) - 1 (x to the left);
//   * the crossings are sorted and paired; span [ROUND_UP(x0), ROUND_DOWN(x1)] with Pillow's sign-symmetric rounding
//     (floor(|f| + .5) and ceil(|f| - .5), sign restored) is drawn when not empty, clipped to the image.
// The one known difference: a polygon that retraces an edge (the same vertex visited twice, e.g. corners a, b, a, c) can
// differ from Pillow by a few pixels on the row of that vertex; a few in 10^4 random integer or half-pixel quadrilaterals
// do.  Boxes built from a rectangle (the dataset's corner order) never retrace.  The test suite pins one such
// quad as an expected failure (test_retraced_vertex_matches_pillow), so a fix or a regression shows.
#pragma once

namespace box_raster {

constexpr int kMap = 800;          // the reference's 800 x 800 map
constexpr int kMaxCross = 8;       // 4 edges, each at most twice

struct Edge {
  int x0, y0, ymin, ymax, xmin, xmax;
  float dx;
  int pad;
};

struct Poly {
  Edge e[4];
  int n;                           // edges in e (horizontal and sloped, in ImagingDrawPolygon's order)
  int ymin, ymax;                  // over all edges
  int pad;
};

__device__ __forceinline__ void add_edge(Edge& e, int x0, int y0, int x1, int y1) {
  e.xmin = x0 <= x1 ? x0 : x1;
  e.xmax = x0 <= x1 ? x1 : x0;
  e.ymin = y0 <= y1 ? y0 : y1;
  e.ymax = y0 <= y1 ? y1 : y0;
  e.dx = y0 == y1 ? 0.f : __fdiv_rn((float)(x1 - x0), (float)(y1 - y0));
  e.x0 = x0;
  e.y0 = y0;
  e.pad = 0;
}

// corners in drawing order (integer pixel coordinates) -> edge list
__device__ __forceinline__ void build(Poly& p, const int (&x)[4], const int (&y)[4]) {
  int n = 0;
  for (int i = 0; i < 3; ++i) {
    const int x0 = x[i], y0 = y[i], x1 = x[i + 1], y1 = y[i + 1];
    if (y0 == y1 && i != 0 && y0 == y[i - 1]) {        // a horizontal segment right after another one
      if (x1 > x0 && x0 > x[i - 1]) { p.e[n - 1].xmax = x1; continue; }
      if (x1 < x0 && x0 < x[i - 1]) { p.e[n - 1].xmin = x1; continue; }
    }
    add_edge(p.e[n++], x0, y0, x1, y1);
  }
  if (x[3] != x[0] || y[3] != y[0]) add_edge(p.e[n++], x[3], y[3], x[0], y[0]);
  p.n = n;
  p.ymin = p.e[0].ymin;
  p.ymax = p.e[0].ymax;
  for (int i = 1; i < n; ++i) {
    p.ymin = p.e[i].ymin < p.ymin ? p.e[i].ymin : p.ymin;
    p.ymax = p.e[i].ymax > p.ymax ? p.e[i].ymax : p.ymax;
  }
  p.pad = 0;
}

__device__ __forceinline__ float x_at(const Edge& e, int y) {
  return __fadd_rn(__fmul_rn((float)(y - e.y0), e.dx), (float)e.x0);
}

__device__ __forceinline__ int round_up(float f) {
  return f >= 0.f ? (int)floorf(__fadd_rn(f, 0.5f)) : -(int)floorf(__fadd_rn(fabsf(f), 0.5f));
}

__device__ __forceinline__ int round_down(float f) {
  return f >= 0.f ? (int)ceilf(__fsub_rn(f, 0.5f)) : -(int)ceilf(__fsub_rn(fabsf(f), 0.5f));
}

__device__ __forceinline__ bool ends_on(const Edge& e, int y) { return y == e.ymin || y == e.ymax; }

// Pillow's spans of polygon p on image row y: emit(x_first, x_last) per span, clipped to [0, kMap), possibly
// overlapping.  xx: kMaxCross floats of scratch, element k at xx[k * stride].
template <class Emit>
__device__ __forceinline__ void row_spans(const Poly& p, int y, float* xx, int stride, Emit&& emit) {
  if (y < p.ymin || y > p.ymax) return;
  auto clip_emit = [&](int a, int b) {
    if (a > b) { const int t = a; a = b; b = t; }
    if (b < 0 || a >= kMap) return;
    emit(a < 0 ? 0 : a, b >= kMap ? kMap - 1 : b);
  };
  int j = 0;
  for (int i = 0; i < p.n; ++i) {
    const Edge& cur = p.e[i];
    if (cur.ymin == cur.ymax) {                        // horizontal: a whole line
      if (y == cur.ymin) clip_emit(cur.xmin, cur.xmax);
      continue;
    }
    if (y < cur.ymin || y > cur.ymax) continue;
    float x = x_at(cur, y);
    xx[j++ * stride] = x;
    if (y == cur.ymax && y < p.ymax) {                 // lower end inside the polygon: counted twice
      xx[j++ * stride] = x;
    } else if (cur.dx != 0.f && ends_on(cur, y) && floorf(x) == x) {
      for (int k = 0; k < i; ++k) {                    // corner rule (see the header comment)
        const Edge& o = p.e[k];
        if (o.ymin == o.ymax || !ends_on(o, y)) continue;
        if (x != x_at(o, y)) continue;
        if ((cur.dx > 0.f && o.dx <= 0.f) || (cur.dx < 0.f && o.dx >= 0.f)) break;
        const int yo = y == cur.ymax ? y - 1 : y + 1;
        if (yo < o.ymin || yo > o.ymax) continue;
        const float a = x_at(cur, yo), b = x_at(o, yo);
        if (x > __fadd_rn(a, 1.f) && x > __fadd_rn(b, 1.f)) x = __fadd_rn(roundf(fmaxf(a, b)), 1.f);
        else if (x < __fsub_rn(a, 1.f) && x < __fsub_rn(b, 1.f)) x = __fsub_rn(roundf(fminf(a, b)), 1.f);
        xx[(j - 1) * stride] = x;
        break;
      }
    }
  }
  for (int i = 1; i < j; ++i) {                        // insertion sort, at most 8 values
    const float v = xx[i * stride];
    int k = i - 1;
    while (k >= 0 && xx[k * stride] > v) { xx[(k + 1) * stride] = xx[k * stride]; --k; }
    xx[(k + 1) * stride] = v;
  }
  for (int i = 1; i < j; i += 2) {
    const int a = round_up(xx[(i - 1) * stride]), b = round_down(xx[i * stride]);
    if (b >= a) clip_emit(a, b);
  }
}

}  // namespace box_raster
