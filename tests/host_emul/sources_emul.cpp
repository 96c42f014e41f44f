// TEST-ONLY host build of the source-map checks of a solve (beta-sgp_b200/csrc/bsgp_rows.h): the map's indices and the
// number of PSF spectra it needs.  Not part of the product.
#define BSGP_HOST_EMUL 1
#include "../../beta-sgp_b200/csrc/bsgp_rows.h"

extern "C" int emul_check_sources(const bsgp_inputs* in, int batch, int n_psf, char* err, int errlen) {
    const int rc = bsgp::check_sources(in, batch, err, (size_t)errlen);
    return rc ? rc : bsgp::check_psf_count(n_psf, in, batch, err, (size_t)errlen);
}
