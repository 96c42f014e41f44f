// TEST-ONLY host build of the iterate-snapshot checks of a solve (beta-sgp_b200/csrc/bsgp_rows.h): the interval, the
// destination and the number of slots per solve.  Not part of the product.
#define BSGP_HOST_EMUL 1
#include <stddef.h>

#include "../../beta-sgp_b200/csrc/bsgp_rows.h"

extern "C" int emul_check_snapshots(const bsgp_outputs* out, char* err, int errlen) {
    return bsgp::check_snapshots(out, err, (size_t)errlen);
}
extern "C" int emul_snapshot_slots(int trace_stride, int snap_every) { return bsgp::snapshot_slots(trace_stride, snap_every); }
extern "C" int emul_sizeof_outputs() { return (int)sizeof(bsgp_outputs); }
extern "C" int emul_offsetof_snap(int which) {
    return which == 0 ? (int)offsetof(bsgp_outputs, snap_x) : which == 1 ? (int)offsetof(bsgp_outputs, snap_every)
                                                                          : (int)offsetof(bsgp_outputs, snap_count);
}
