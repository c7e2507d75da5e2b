// tiles.h — host-side estimates of a camera-grid frame's 16 x 16 tiles, before any ray is traced: the work each tile may
// cost (api.cu orders the tiles by it), which items each tile's primary rays can see (the kernel traces only those) and which
// tiles provably see nothing (the kernel writes those without tracing).
// Host-only C++, so that the CPU tests can run it on the real lowering.
#pragma once

#include <vector>

#include "lower.h"

namespace ftb {

struct V3 { double x, y, z; };
inline V3 sub(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
inline V3 cross(V3 a, V3 b) { return {a.y * b.z - a.z * b.y, b.x * a.z - b.z * a.x, a.x * b.y - a.y * b.x}; }
inline double dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
V3 normalise(V3 v);

// ImagePlane.create / fromCamera (Image.fs:48-53, 67-81), evaluated in double on the host: the camera's basis, the image
// plane's size, the pixel pitch and the centre of the top-left pixel.  resH = frame width, resV = frame height.
struct CameraBasis { V3 o, k, i, j; double width, height, pw, ph, tlx, tly; };
CameraBasis cameraBasis(const ftb_camera& c, int resH, int resV);

// The window's tile grid: its origin and size in the whole frame's sample grid, and its tiles.
struct TileGrid { int wx0, wy0, ww, wh, tiles_x, tiles_y; };

// A rectangle of the image plane, in the coordinates of d = k + x i + y j (x to the right, y up), outside which no primary ray
// has a crossing with an item at any t (clear_boxes.h).  valid = false: the item has none.  xl > xh: it has no crossings.
struct ImageRect { bool valid; double xl, xh, yl, yh; };

// The largest distance, in pixels along either axis, of a primary sample from its pixel's centre: the largest |jitter_xy|,
// 0.5 in corner sampling.
double sampleOffsetExtent(const ftb_render_params& p);

// For every tile of the window, row-major:
//   cost[t]  = 1 + the work weight of every item whose bounding sphere a primary ray of tile t may touch;
//   items[t] = bit i set when item i may give a primary sample of tile t a crossing that the kernel reports: its bounding sphere
//              is touched (and, with box_rects, its boxes' rectangle too), or it is unbounded and not a top-level plane that
//              all of the tile's rays leave behind.  A clear bit: the item can be left out of the tile's primary rays' trace
//              without changing any result.  Filled only for the pinhole camera and scenes of at most 32 items, else empty.
//   clear[t] = 1 when no primary sample of tile t has a crossing at t >= 0 with anything: the tile's mask is 0.  Such a
//              sample's colour is exactly zero.  Never set with depth of field or an unbounded item of another kind.
// `offset` = sampleOffsetExtent.  Returns false when no bounded item touches the window (every cost is 1).
// box_rects (per item, clear_boxes.h), when given: an item whose valid rectangle, widened by the samples' pixel slack, misses
// a tile keeps no bit in that tile even where its sphere is touched.  The costs use the spheres only.
// kept, with items filled: over the traced tiles, the bits the masks keep per bit the spheres alone keep (every unbounded item
// counted as kept by both): how much of phase A's candidate work the masks leave.
bool estimateTiles(const Lowered& L, int n_lights, const ftb_camera& c, int width, int height, int recursion_limit, double offset, const TileGrid& g,
                   std::vector<float>& cost, std::vector<unsigned char>& clear, const std::vector<ImageRect>* box_rects = nullptr,
                   std::vector<unsigned>* items = nullptr, double* kept = nullptr);

}  // namespace ftb
