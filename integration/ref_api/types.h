/*
 * types.h -- stand-in for the FlyDog_SDR_GPS top-level types.h, for building the adapter (integration/search_gpu.cpp)
 * without the receiver's source tree.  See gps/gps.h next to it.  The adapter uses none of the receiver's own
 * typedefs; it needs the fixed-width integer types.
 */
#pragma once
#include <stdint.h>
