// fused.cuh - what count.cu and select.cu share for dvs_count_select (counting with the selection rounds trailing)
#pragma once
#include <stdlib.h>

#include "common.cuh"

namespace dvs {
struct TrailArgs {
    const unsigned* d_ready;   // device word: positions of `order` below it have their rows, entropies and flags
    unsigned limit0;           // its value once `first_ready` has happened
    cudaEvent_t first_ready;   // the first chunk of records has been published
    cudaEvent_t count_done;    // all of them have
};
// How counting and the trailing selection share the GPU: the selection owns DVS_TRAIL_SMS whole SMs (default 36;
// measured 24..40 on the bench set).  The stand-alone 512-thread kernel on a high-priority stream takes the SMs the
// counting CTAs of a finished launch leave, and the counting goes on with the rest (its CTAs are work-stealing loops,
// so the ones that find no SM just start late and exit).
inline unsigned trail_sms(int sm_count) {
    const char* e = getenv("DVS_TRAIL_SMS");
    const int v = e ? atoi(e) : 36;
    return (unsigned)(v < 2 ? 2 : (v > sm_count / 2 ? sm_count / 2 : v));
}
int select_with_trail(dvs_ctx* ctx, const dvs_kfreqs* f, const uint32_t* order, uint32_t num, int mode, uint32_t min_size,
                      uint32_t max_size, uint32_t* sel_idx, double* sel_delta, double* stats5, uint32_t* size_out,
                      const TrailArgs* trail);
}  // namespace dvs
