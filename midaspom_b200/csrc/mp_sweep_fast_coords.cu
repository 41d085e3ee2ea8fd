// FP32 fast y sweep, coords geometry (see mp_sweep_fast.cuh); separate TU so the geometries compile in parallel.
#include "../../include/libmidaspom_cuda.h"
#define MP_FAST_GEOM MP_GEOM_COORDS
#define MP_FAST_HAS_POSITIONS 1
#include "mp_sweep_fast.cuh"
#include "mp_sweep_cull.cuh"
int mp_launch_sweep_fast_coords(mp_engine *h, int cs, int tpt) { return mp::launch_fast_any(h, cs, tpt); }
int mp_launch_sweep_cull_coords(mp_engine *h, int cs, int tpt, int nl_max, int nclusters, const void *btasks) { return mp::launch_cull_any(h, cs, tpt, nl_max, nclusters, btasks); }
