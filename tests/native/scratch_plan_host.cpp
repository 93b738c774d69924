// Host build of the scratch batch planner (mdproptools_b200/csrc/scratch_plan.h) used by pair.cu and fftcorr.cu.
// TEST INFRASTRUCTURE ONLY.
#include <stddef.h>

#include "../../mdproptools_b200/csrc/scratch_plan.h"

extern "C" unsigned long long plan_units(unsigned long long target, unsigned long long fixed, unsigned long long per_unit,
                                         unsigned long long max_units)
{
    return mdp_scratch_units((size_t)target, (size_t)fixed, (size_t)per_unit, (size_t)max_units);
}

extern "C" unsigned long long plan_reserved(unsigned long long bytes) { return mdp_scratch_reserved((size_t)bytes); }
