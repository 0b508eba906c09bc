/* ref_compat.h — force-included (nvcc -include) in front of the UNMODIFIED reference sources
 * when oracle/ref_build/Makefile compiles them for sm_100a.  TEST INFRASTRUCTURE ONLY.
 *
 * The reference does not compile as committed (SURVEY.md §8c):
 *   - `counterMax` (EventDrivenMap.cu:564) is defined nowhere           -> 100 (SURVEY Q6)
 *   - `__shfl_down` (EventDrivenMap.cu:847,848,885,921) was removed     -> the _sync form with
 *     for sm_70+                                                           a full-warp mask
 * Nothing else is changed: the reference translation units are compiled where they lie in the
 * reference checkout (REF / B200_REFERENCE_DIR), against this repo's Armadillo subset
 * (host/arma_shim) because Armadillo itself is not installed. */
#pragma once
#define counterMax 100
#define __shfl_down(v, o) __shfl_down_sync(0xffffffffu, (v), (o))
