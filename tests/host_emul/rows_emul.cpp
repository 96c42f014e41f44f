// TEST-ONLY host build of the keyword checks of a solve (beta-sgp_b200/csrc/bsgp_rows.h): the shared keywords or one
// row per image, the rows' operator fields, the inputs each row needs, and the trace stride.  Not part of the product.
#define BSGP_HOST_EMUL 1
#include "../../beta-sgp_b200/csrc/bsgp_rows.h"

extern "C" int emul_check_batch_params(const bsgp_params* prm, const bsgp_params* rows, int batch, const bsgp_inputs* in,
                                       const bsgp_outputs* out, int* trace_stride, char* err, int errlen) {
    return bsgp::check_batch_params(prm, rows, batch, in, out, trace_stride, err, (size_t)errlen);
}
