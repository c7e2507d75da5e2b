// lit_tiles.h — host-side proof, before any ray is traced, that the directional-light shadow rays of a camera-grid frame's
// ground fragments are unblocked: per 16 x 16 tile of the window and per directional light, "every primary sample of this
// tile that lands on the ground plane sees that light".  The FP32 kernels then set those lights' intensity to 1 without
// tracing the shadow rays.  Host-only C++, so that the CPU tests can run it on the real lowering.
#pragma once

#include <vector>

#include "tiles.h"

namespace ftb {

// lit[t], for every tile t of the window (row-major, the window's grid g): bit k (k < 8) set when every primary sample of
// tile t whose FP32 nearest hit is on the ground leaf has a shadow ray towards light k that the FP32 kernels would report
// unblocked (DESIGN.md §3 "Lit ground tiles").  Only directional and soft directional lights get bits.  The ground is the
// scene's only unbounded item, a top-level plane; without one, with another unbounded item or with depth of field every
// bit is 0.  `offset` = sampleOffsetExtent.  Returns the ground's leaf index when some bit is set, else -1.
int litTiles(const Lowered& L, const ftb_light* lights, int n_lights, const ftb_camera& c, int width, int height, double offset, const TileGrid& g,
             std::vector<unsigned char>& lit);

}  // namespace ftb
