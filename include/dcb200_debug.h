/* dcb200 -- developer / test hooks of libdcb200.so.  NOT part of the drop-in boundary (include/dcb200.h): nothing a
 * caller of the model path needs.  Used by tests/ and scripts/ to look inside a forward pass. */
#ifndef DCB200_DEBUG_H_
#define DCB200_DEBUG_H_

#include "dcb200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Debug/test hook: copy the fp32 residual stream after stage `stage` of the LAST chunk of the
 * last forward into out [tokens, 280] (row-major).  stage 0 = condenser+pos-enc,
 * 1+2n = attention sub-layer n, 2+2n = FFN sub-layer n.  Requires dcb_set_debug(e, 1). */
int dcb_set_debug(dcb_engine* e, int32_t enabled);
int dcb_debug_residual(dcb_engine* e, int32_t stage, float* out, int64_t out_elems);

/* Developer hook: cycle counters of the last traced kernel launch (the counter buffer is shared by
 * every kernel with trace hooks; only meaningful in a -DDCB_TRACE build; 16 uint64 per CTA). */
int dcb_debug_trace(uint64_t* out, int32_t n);

#ifdef __cplusplus
}
#endif
#endif /* DCB200_DEBUG_H_ */
