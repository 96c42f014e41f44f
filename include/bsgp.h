/* libbsgp — C ABI of the B200-native SGP / beta-SGP restoration loop.
 *
 * The reference (Yash-10/beta-sgp) is pure Python and has no FFI of its own; its boundary for this
 * path is three importable callables,
 *     restoration/sgp.py:41-47          sgp(gn, psf, bkg, ...)          -> (x, iters, discr, times, err)
 *     restoration/sgp.py:506-513        sgp_betaDiv(gn, psf, bkg, ...)  -> (x, iters, discr, times, None)
 *     restoration/flux_conserve_proj.py:7   projectDF(b, c, dia, scaling, ...) -> x
 * plus the helpers betaDiv / betaDivDeriv (sgp.py:441-495).  The entry points below are what a ctypes
 * binding of those callables calls (see INTEGRATION.md for the stub); the Python modules
 * beta-sgp_b200/sgp.py and beta-sgp_b200/flux_conserve_proj.py are that binding.
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or a BSGP_E_* code
 * and bsgp_last_error_string() describes the last failure of the calling thread.  "_host" entry
 * points take host pointers and do the host<->device staging themselves; the others take device
 * pointers, run asynchronously on `stream` (a cudaStream_t passed as void*) and never synchronise.
 * Images are row-major [batch][ny][nx] in the plan's dtype.  There is no CPU fallback: without a
 * CUDA device every compute entry point fails with BSGP_E_CUDA.
 *
 * Shapes.  Any ny x nx (the reference's numpy closure accepts any size, sgp.py:108-120; its star-stamp application
 * uses 31 x 31 cut-outs, application_sgp_star_stamps.py:24,58).  Sides that are powers of two in [16, 16384] run on
 * their own FFT grid and need 16-byte aligned image pointers.  Any other side n <= 32 keeps a grid of 16 or 32 slots and
 * is transformed by a dense DFT of length n; any other side n <= 8192 runs on a grid of side 2^k >= 2n - 1 ("wrapped":
 * linear convolution + fold).  A grid with a 16384-point side runs in frame mode and cannot pair with a dense axis
 * (BSGP_E_SHAPE otherwise); in BSGP_F64 its 16384-point axes run split transforms of two 8192-point halves.  Both are exactly the circular operator with the reference's np.fft.fftshift placement,
 * including its one-pixel offset for odd n; the library moves the caller's arrays to and from the grid itself and only
 * needs element alignment.
 *
 * Streams.  A plan owns mutable device state (PSF spectra, scratch, the work queue).  Launches on one plan are
 * serialised on the device: every device entry point makes `stream` wait for the plan's previous launch (an event),
 * so one plan may be used from several streams; use one plan per stream for concurrency.  Buffers passed to an
 * asynchronous call must stay alive until that call's work has completed.
 */
#ifndef BSGP_H
#define BSGP_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bsgp_plan bsgp_plan;

enum { BSGP_F64 = 0, BSGP_F32 = 1 };
enum { BSGP_DIV_KL = 0,      /* sgp():         KL objective, gradient 1 - A^T(gn/den)          sgp.py:260-265 */
       BSGP_DIV_BETA = 1 };  /* sgp_betaDiv(): beta-divergence objective / gradient            sgp.py:441-499 */

/* library-level error codes */
enum { BSGP_OK = 0, BSGP_E_ARG = 1, BSGP_E_SHAPE = 2, BSGP_E_CUDA = 3, BSGP_E_NOMEM = 4, BSGP_E_STATE = 5 };

/* per-image solve status (outputs.status) */
enum { BSGP_ST_OK = 0,
       BSGP_ST_BAD_FLUX = 1,        /* flux <= 0 or non-finite with proj_type = 1 (reference: ValueError at sgp.py:269/713) */
       BSGP_ST_EMPTY_BOUNDS = 2,    /* no positive entry in flux/(flux+bkg)*A^T(gn) (reference: ValueError at sgp.py:269/713) */
       BSGP_ST_PROJ_NO_BRACKET = 3, /* projection could not bracket the multiplier (reference: endless loop) */
       BSGP_ST_INPUT_TIMEOUT = 4    /* bsgp_solve_batch_pinned: the image's upload did not arrive within 20 s; image skipped */ };

/* Keyword arguments of sgp() / sgp_betaDiv(), same names and meaning (sgp.py:41-47, 506-513). */
typedef struct bsgp_params {
    int divergence;        /* BSGP_DIV_KL or BSGP_DIV_BETA */
    int init_recon;        /* 0 zeros, 1 caller-supplied x0 (the binding draws randn with seed 42), 2 gn, 3 flux/N */
    int proj_type;         /* 0 non-negativity, 1 flux-conserving projection */
    int stop_criterion;    /* 0/1 run to MAXIT, 2 step norm, 3 relative decrease, 4 discrepancy */
    int maxit;             /* MAXIT */
    double gamma;          /* line-search sufficient-decrease parameter */
    double ls_beta;        /* `beta`: line-search shrink factor */
    double alpha;          /* initial step length */
    double alpha_min, alpha_max;
    int m_alpha;           /* M_alpha, <= 16 */
    double tau;
    int m;                 /* M (non-monotone memory), <= 16 */
    int max_projs;
    int verbose;           /* only effect on the numbers: tol := tol^2 for stop_criterion 2 (sgp.py:291-294) */
    int has_flux;          /* inputs.flux is given (else flux = sum(gn - bkg)) */
    int has_sat;           /* ccd_sat_level is given */
    double ccd_sat_level;
    int scale_data;
    int errflag;           /* KL only: per-iteration relative error against inputs.obj */
    double tol_convergence;
    int adapt_beta;        /* beta-divergence only */
    double lr, lr_exp_param;
    int schedule_lr;
    /* Zero-padded ("astropy") operator, use_original_SGP_Afunction=False (sgp.py:121-161, 583-615).  The caller
     * embeds every image into the plan's power-of-two FFT grid; region = {r0, r1, c0, c1} is the window the image
     * occupies ([r0, r1) x [c0, c1)).  All zeros: the image is the whole grid (circular operator).  Pixel counts,
     * sums and the projection only see the window; operator outputs are divided by div_a (A) / div_at (A^T), the
     * kernel-weight constants of convolve_fft's nan_treatment='interpolate'. */
    int region[4];
    double div_a, div_at;
    int adjoint_second_psf;   /* A^T uses the spectrum set by bsgp_set_psf_adjoint (kernel psf.conj().T) instead of conj(TF) */
} bsgp_params;

typedef struct bsgp_inputs {
    const void* gn;        /* [batch][ny][nx] observed images */
    const void* bkg;       /* bkg_is_image ? [batch][ny][nx] : [batch] (one scalar per image, plan dtype) */
    int bkg_is_image;
    const double* flux;    /* [batch] or NULL (params.has_flux) */
    const double* beta0;   /* [batch] initial betaParam (BSGP_DIV_BETA) or NULL */
    const void* x0;        /* [batch][ny][nx] start images for init_recon = 1, else NULL */
    const void* obj;       /* [batch][ny][nx] ground truth for errflag, else NULL */
    const int* order;      /* [batch] permutation: the work queue hands out image order[0], order[1], ... (longest expected
                              solve first keeps the tail of the queue short); NULL = 0, 1, 2, ...  Results are always
                              stored at the image's own index. */
    /* Shared observations: solve i reads observation source[i], so several solves of one image (a beta sweep, KL and
     * beta-SGP runs of one sub-frame) need one copy of its pixels and one PSF spectrum.  source: [batch] in HOST memory
     * on every entry point (read before the call returns), each entry in [0, n_sources), n_sources >= 1; NULL = the
     * identity (n_sources ignored), which is the behaviour without this field.  With a map, everything that describes the
     * observation is indexed by source: gn, bkg (stack or per-image scalar), x0, obj, and the PSF spectra, whose count
     * must then be 1 or n_sources (bsgp_set_psf; the adjoint kernel the same).  Everything that describes the solve
     * stays indexed by solve: flux, beta0, order, the rows of a mixed batch, and every output.  A bad index is
     * BSGP_E_ARG naming the solve, before anything is launched. */
    const int* source;
    int n_sources;
} bsgp_inputs;

#define BSGP_NSCALARS 8    /* scaling, flux (scaled), X_low_bound, X_upp_bound, tol, fv_final, alpha_final, tau_final */

typedef struct bsgp_outputs {
    void* x;               /* [batch][ny][nx] restored images (un-scaled, like the reference's return value) */
    int* iters;            /* [batch] iteration count as returned by the reference */
    int* status;           /* [batch] BSGP_ST_* */
    /* Trace arrays: one row of `stride` entries per image, stride = maxit + 1 (err: maxit + 2).  A mixed batch
     * (bsgp_solve_batch_rows) uses the largest maxit of its rows for every image; entries past an image's own iters
     * (its own maxit + 1 for err) are left as the caller allocated them. */
    double* discr;         /* [batch][maxit+1]; entries [0, iters] valid */
    double* times;         /* [batch][maxit+1] seconds since the image's solve began (device %globaltimer) */
    double* stop_value;    /* [batch][maxit+1] quantity compared with tol (criteria 2-4); may be NULL */
    double* err;           /* [batch][maxit+2] errflag trace; may be NULL */
    double* beta_final;    /* [batch] final betaParam; may be NULL */
    int* proj_evals;       /* [batch] total full-image projection evaluations (E summed); may be NULL */
    int* ls_trials;        /* [batch] total line-search evaluations (T summed); may be NULL */
    double* scalars;       /* [batch][BSGP_NSCALARS]; may be NULL */
    /* optional per-iteration controller trace, each [batch][maxit+1] or NULL */
    double* trace_alpha;
    double* trace_lambda;
    double* trace_beta;
    int* trace_trials;
    int* trace_evals;
    /* Iterate snapshots: every snap_every-th iterate of each solve, stored from inside the kernel, so that "which
     * iteration to keep" needs one launch instead of one solve per candidate MAXIT.  snap_every = 0: none (the behaviour
     * without these fields); < 0 is BSGP_E_ARG, and so is snap_every > 0 with snap_x NULL.
     *   snap_x: [batch][n_snap][ny][nx] in the plan's dtype, n_snap = maxit / snap_every + 1 (a mixed batch: the largest
     *           maxit of its rows, as for the traces).  Slot j holds the iterate after j * snap_every passes of the main
     *           loop (sgp.py:302-425 / 748-882), un-scaled like x: slot 0 is the start image after the initial
     *           projection.  A pass that stops the solve still stores the iterate it formed (the one the reference then
     *           discards, x = prev_x) if its number is a multiple of snap_every.  So slot j is bit-identical to x of the
     *           same solve run with MAXIT = j * snap_every + 1 and stop rule 1.  Slots past the last one a solve writes
     *           are left as the caller allocated them.  The shape is the caller's image shape on every plan, including
     *           plans whose grid differs from the image (sides that are not powers of two).
     *   snap_count: [batch] or NULL: the number of slots each solve wrote, 1 + (passes made) / snap_every.
     * A launch with snapshots runs the mixed-batch kernels (shared keywords become equal rows).  The device and _host
     * entry points, plain and _rows, support them; bsgp_solve_batch_pinned and _rows_pinned refuse snap_every > 0 with
     * BSGP_E_ARG.  Memory: batch * n_snap * ny * nx * sizeof(dtype) bytes. */
    void* snap_x;
    int snap_every;
    int* snap_count;
} bsgp_outputs;

typedef struct bsgp_plan_info {
    int ny, nx, dtype, device;
    int cluster_size;      /* CTAs cooperating on one image (cluster size, or the grid size in frame mode) */
    int num_clusters;      /* images in flight */
    int threads;           /* threads per CTA */
    int smem_bytes;        /* dynamic shared memory per CTA */
    int num_sms;
    int resident_mask;     /* bit b set: per-image buffer b lives in shared memory */
    long long workspace_bytes;
    int grid_ny, grid_nx;  /* the power-of-two FFT grid (== ny, nx unless the plan is wrapped) */
} bsgp_plan_info;

/* One plan per (shape, dtype, device): twiddle tables, per-cluster scratch, PSF spectra.  Any shape with sides in
 * [1, 16384] (powers of two) or [1, 8192] (other sizes), with the limits on 16384-point grids of "Shapes" above.
 * BSGP_E_NOMEM (with the size in bsgp_last_error_string) when the device cannot hold the plan's buffers. */
int bsgp_plan_create(int ny, int nx, int dtype, int device, bsgp_plan** plan);
int bsgp_plan_destroy(bsgp_plan* plan);
int bsgp_plan_get_info(const bsgp_plan* plan, bsgp_plan_info* info);
/* Tuning knobs (0 = automatic): cluster size and threads per CTA.  Call before bsgp_set_psf.
 * cluster_size = -1 selects frame mode (one image at a time over the whole GPU, cooperative launch), which is
 * the automatic choice for images of 2^20 pixels or more; info.cluster_size then reports the grid size. */
int bsgp_plan_configure(bsgp_plan* plan, int cluster_size, int threads);

/* TF = fftn(fftshift(psf)) for n_psf PSFs of the image shape (sgp.py:109 / 571); n_psf is 1 (shared by
 * the whole batch) or the batch size (one PSF per image).  A solve with a source map (bsgp_inputs.source) needs 1 or
 * n_sources PSFs, one per observation: every solve of an observation uses its spectrum. */
int bsgp_set_psf(bsgp_plan* plan, const void* psf_dev, int n_psf, void* stream);
int bsgp_set_psf_host(bsgp_plan* plan, const void* psf_host, int n_psf);
/* Second kernel for A^T (sgp.py:157: convolve_fft(x, psf.conj().T, ...)); same n_psf as bsgp_set_psf.  Power-of-two
 * plans only (BSGP_E_STATE otherwise: wrapped plans use both spectra for the circular operator itself). */
int bsgp_set_psf_adjoint(bsgp_plan* plan, const void* psf_dev, int n_psf, void* stream);
int bsgp_set_psf_adjoint_host(bsgp_plan* plan, const void* psf_host, int n_psf);

/* The restoration loop for `batch` independent images; one persistent kernel launch, no host sync. */
int bsgp_solve_batch(bsgp_plan* plan, const bsgp_params* params, int batch, const bsgp_inputs* in_dev,
                     const bsgp_outputs* out_dev, void* stream);
int bsgp_solve_batch_host(bsgp_plan* plan, const bsgp_params* params, int batch, const bsgp_inputs* in_host,
                          const bsgp_outputs* out_host);
/* The same call for PAGE-LOCKED host images (in.gn, in.bkg if it is an image stack, in.x0, in.obj, out.x; the small
 * arrays may live in any host memory), pipelined: the images are uploaded on a private copy stream in the order the
 * work queue hands them out while the persistent kernel is already restoring the first ones (it waits for a per-item
 * ready flag), and every restored image is stored straight into out.x (mapped, zero-copy) while others are still being
 * solved.  Ordered after the work already queued on `stream` (e.g. bsgp_set_psf); returns when all results are in host
 * memory.  This is what replaces the reference's per-image Python loop when the caller's data lives on the host
 * (application_sgp_star_stamps.py:56-105, application_sgp_subdivisions.py:83-107). */
int bsgp_solve_batch_pinned(bsgp_plan* plan, const bsgp_params* params, int batch, const bsgp_inputs* in_host,
                            const bsgp_outputs* out_host, void* stream);

/* Mixed batches: the same three calls with one bsgp_params per image, rows[0 .. batch-1] in host memory (read before the
 * call returns), so that images with different keywords (KL and beta-SGP, stop rule, maxit, projection, saturation, ...)
 * share one persistent launch.  Image i is exactly a solve of that image alone with rows[i].  The operator fields
 * (region, div_a, div_at, adjoint_second_psf) describe the plan's operator and must be equal in every row; a row with
 * has_flux, errflag, init_recon = 1 or the beta-divergence needs inputs.flux, inputs.obj (and outputs.err), inputs.x0 or
 * inputs.beta0, as with the shared keywords.  Any violation is BSGP_E_ARG, naming the row, before anything is launched.
 * The trace outputs have the stride of the largest maxit of the rows (see bsgp_outputs).  The device entry point copies
 * the rows to the plan's device memory on `stream`, behind the plan's previous launch. */
int bsgp_solve_batch_rows(bsgp_plan* plan, const bsgp_params* rows, int batch, const bsgp_inputs* in_dev,
                          const bsgp_outputs* out_dev, void* stream);
int bsgp_solve_batch_rows_host(bsgp_plan* plan, const bsgp_params* rows, int batch, const bsgp_inputs* in_host,
                               const bsgp_outputs* out_host);
int bsgp_solve_batch_rows_pinned(bsgp_plan* plan, const bsgp_params* rows, int batch, const bsgp_inputs* in_host,
                                 const bsgp_outputs* out_host, void* stream);

/* y = real(ifftn(TF * fftn(x))) (adjoint = 0) or with conj(TF) (adjoint = 1) for `batch` images: the
 * reference's A / A^T closures (sgp.py:111-120). PSF index = image index if n_psf > 1. */
int bsgp_apply_psf(bsgp_plan* plan, const void* x_dev, void* y_dev, int batch, int adjoint, void* stream);
int bsgp_apply_psf_host(bsgp_plan* plan, const void* x_host, void* y_host, int batch, int adjoint);

/* projectDF (flux_conserve_proj.py:7): `batch` independent problems of length n, fp64.
 * sat_cap < 0 or NaN: no upper clamp; else x <= sat_cap (the caller passes ccd_sat_level/scaling - eps).
 * lambda0, dlambda0, tol_lam, biter, siter, max_projs: the reference's keyword arguments of the same names; biter
 * and siter are the initial values of its two counters (the secant budget is max_projs - biter AFTER the bracketing,
 * flux_conserve_proj.py:103, and the loop runs while siter < budget, :106). */
int bsgp_project_df(const double* b_dev, const double* c_dev, const double* dia_dev, int n, int batch, double sat_cap,
                    double lambda0, double dlambda0, double tol_lam, int max_projs, int biter, int siter, double* x_dev,
                    int* evals_dev, int* status_dev, int device, void* stream);
int bsgp_project_df_host(const double* b, const double* c, const double* dia, int n, int batch, double sat_cap,
                         double lambda0, double dlambda0, double tol_lam, int max_projs, int biter, int siter, double* x,
                         int* evals, int* status, int device);

/* betaDiv(y, x, beta) (sgp.py:441-458): three partial sums -> out[0]; betaDivDeriv (sgp.py:462-495)
 * per element -> deriv (may be NULL).  fp64, host pointers. */
int bsgp_beta_div_host(const double* y, const double* x, long long n, double beta, double* value, double* deriv,
                       int device);

/* The two per-pixel pieces of betaDivDerivwrtY (sgp.py:498-499): p1 = den^(beta-1), u = gn*den^(beta-2);
 * the caller finishes with p1 - AT(u).  fp64, host pointers. */
int bsgp_beta_grad_terms_host(const double* den, const double* gn, long long n, double beta, double* p1, double* u,
                              int device);

/* Tiling of a frame into overlapping subdivisions and re-assembly: the callers either side of the batched solve
 * (utils.py:332-375 calculate_slice_bboxes, :378-389 create_subdivisions, :392-397 reconstruct_full_image_from_patches).
 * bsgp_tile_boxes (host): the reference's enumeration, boxes as [xmin, ymin, xmax, ymax]; boxes_xyxy may be NULL to
 * query the count.  bsgp_extract_tiles: tiles[t] = frame[y0:y0+tile_h, x0:x0+tile_w] for origins[t] = (y0, x0), zeros
 * outside the frame.  bsgp_assemble_tiles: weighted average of the tiles covering each pixel with a linear cross-fade
 * of `feather` pixels at tile borders (<= 1: plain average); replaces reproject_and_coadd, which needs WCS headers
 * and is not bit-comparable. */
int bsgp_tile_boxes(int height, int width, int tile_h, int tile_w, double overlap_h_ratio, double overlap_w_ratio,
                    int* boxes_xyxy, int max_boxes, int* n_boxes);
int bsgp_extract_tiles(const void* frame_dev, int height, int width, int dtype, const int* origins_dev, int n, int tile_h,
                       int tile_w, void* tiles_dev, int device, void* stream);
int bsgp_assemble_tiles(const void* tiles_dev, const int* origins_dev, int n, int tile_h, int tile_w, int dtype, int feather,
                        void* frame_dev, int height, int width, int device, void* stream);

/* DIAPL PSF model (psf/psf_calculate.py:52-111, PSF.calc_psf_pix / get_psf_mat / normalize_psf_mat): n PSFs, each from
 * a parameter row [cos, sin, ax, ay, sigma_inc, ngauss * 6 coefficients] (device, fp64), evaluated on the
 * (2 hw + 1)^2 support, optionally normalised to sum 1, and written centred at (ny/2, nx/2) of out[n][ny][nx] (zeros
 * elsewhere): the placement bsgp_set_psf expects. */
int bsgp_psf_model_eval(const double* params_dev, int n, int ngauss, int hw, int ny, int nx, int normalize, int dtype,
                        void* out_dev, int device, void* stream);

int bsgp_device_count(void);
/* Number of CUDA kernels this library has launched in the calling process so far (all plans, all streams). */
long long bsgp_launch_count(void);
const char* bsgp_last_error_string(void);
const char* bsgp_version(void);

#ifdef __cplusplus
}
#endif
#endif /* BSGP_H */
