// scratch_plan.h -- how many units of work one scratch request can hold: the frames of a pair-engine sub-batch
// (pair.cu) and the channels of an FFT correlation group (fftcorr.cu).  Host only; exercised on the host by
// tests/native/scratch_plan_host.cpp.
//
// A call asks the arena for `fixed + units * per_unit` bytes.  mdp_ctx::arena_reserve rounds the request up to 256
// bytes, adds 4096 and refuses the total above the context's limit (mdp_scratch_reserved below is that total).  So the
// batch is sized on the same total: the largest unit count whose reserved total stays within the target.  Sizing on
// the bare `fixed + units * per_unit` instead lets the added bytes push the request over a limit that one unit fewer
// would have respected -- a call then fails at a limit just above one that works.
#pragma once
#include <stddef.h>

// the bytes mdp_ctx::arena_reserve checks against the limit for a request of `bytes`
static inline size_t mdp_scratch_reserved(size_t bytes)
{
    return ((bytes + 255) & ~(size_t)255) + 4096;
}

// the largest n in [1, max_units] with mdp_scratch_reserved(fixed + n * per_unit) <= target; 1 when not even one unit
// fits (that request exceeds the target, and arena_reserve reports it when the target is the limit).  Non-decreasing in
// target.  Uses round256(x) + 4096 <= t  <=>  x <= floor256(t - 4096).
static inline size_t mdp_scratch_units(size_t target, size_t fixed, size_t per_unit, size_t max_units)
{
    if (max_units < 1) max_units = 1;
    if (per_unit == 0) return max_units;
    if (target < 4096) return 1;
    const size_t room = (target - 4096) & ~(size_t)255;
    if (room < fixed) return 1;
    const size_t n = (room - fixed) / per_unit;
    return n < 1 ? 1 : n > max_units ? max_units : n;
}
