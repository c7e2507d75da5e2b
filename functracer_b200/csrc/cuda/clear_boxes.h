// clear_boxes.h — a tighter proof than the bounding sphere that a primary ray sees nothing of an item: the image-plane
// rectangle of the item's world-space boxes (lower.h ItemBoxes), for estimateTiles' clear tiles (tiles.h).  Host-only C++,
// so that the CPU tests can run it on the real lowering.
#pragma once

#include <vector>

#include "tiles.h"

namespace ftb {

// Per item of L: the image-plane rectangle outside which no primary ray of the pinhole camera c, traced by the FP32 kernels,
// has a crossing with the item at any t (DESIGN.md §3 "Clear tiles").  Invalid for an item without boxes, with a box not
// wholly in front of the camera, or with a planar face that may report its t = 0 crossing at the camera; all invalid with
// depth of field.
std::vector<ImageRect> itemBoxRects(const Lowered& L, const ftb_camera& c, int width, int height);

}  // namespace ftb
