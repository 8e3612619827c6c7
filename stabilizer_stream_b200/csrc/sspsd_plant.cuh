// sspsd_plant.cuh -- feeding a plant (sspsd_plant_*, defined in sspsd_plant.cu) straight into the handles that
// sspsd_group.cu holds by their C++ classes.
#pragma once
#include "sspsd_xcascade.cuh"

namespace sspsd {

// the next n positions of p into the handle, on the handle's stream (the rules of sspsd_*_process_plant)
int plant_feed(sspsd_plant* p, Cascade& c, size_t n);
int plant_feed(sspsd_plant* p, XCascade& x, size_t n);
int plant_feed(sspsd_plant* p, ZoomCascade& z, size_t n);
// the spec's own checks of sspsd_plant_create, with no device touched
int plant_check(const sspsd_plant_spec* spec);

}  // namespace sspsd
