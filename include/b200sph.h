/*
 * b200sph.h -- C-ABI of libb200sph.so: the B200-native (sm_100a) evaluator for
 * PySPH's per-timestep WCSPH hot path.
 *
 * The reference has no FFI for this path: the seam is the set of duck-typed
 * Python objects SPHCompiler installs (SURVEY.md 8b).  Each entry point below
 * names the reference interface it stands behind (file:line under
 * /root/reference); pysph_b200/ binds them with ctypes and INTEGRATION.md
 * shows the stub a PySPH maintainer would add.
 *
 * Conventions
 *   - plain C types only; every function returns 0 on success, <0 on error
 *     (b200sph_last_error gives the message), unless stated otherwise.
 *   - the library OWNS device memory.  Host pointers are borrowed for the
 *     duration of a push/pull call only (ParticleArray storage is re-allocated
 *     by resize/append, particle_array.pyx:439-700, so callers re-fetch them).
 *   - one context = one device + one stream; calls on a context are not
 *     re-entrant.  Multi-GPU = one context per rank/device.
 *   - host-side floating point properties are fp64 (ParticleArray is fp64);
 *     on the device the integrated state (x y z u v w rho h m and the *0
 *     copies) is fp64, derived fields (p cs arho au.. ax.. dt_cfl dt_force)
 *     are fp32, and the pair kernel works on fp32 cell-relative records.
 */
#ifndef B200SPH_H_INCLUDED
#define B200SPH_H_INCLUDED
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200SPH_MAX_ARRAYS 8
#define B200SPH_MAX_USER 16    /* user properties of the generic-equation fallback */
#define B200SPH_MAX_RANKS 16   /* ranks of one node in the peer protocol (b200sph_peer_*) */
#define B200SPH_ABI_VERSION 5

typedef struct b200sph_ctx b200sph_ctx;

/* smoothing kernels: pysph/base/kernels.py:29 (CubicSpline), :274
 * (WendlandQuintic), :1050 (QuinticSpline), :830 (Gaussian) */
enum {
    B200SPH_KERNEL_CUBIC_SPLINE = 0,
    B200SPH_KERNEL_WENDLAND_QUINTIC = 1,
    B200SPH_KERNEL_QUINTIC_SPLINE = 2,
    B200SPH_KERNEL_GAUSSIAN = 3
};

/* particle properties: pysph/base/utils.py:41-44,177-178 */
enum {
    /* fp64 on device */
    B200SPH_X = 0, B200SPH_Y, B200SPH_Z, B200SPH_U, B200SPH_V, B200SPH_W,
    B200SPH_RHO, B200SPH_H, B200SPH_M,
    B200SPH_X0, B200SPH_Y0, B200SPH_Z0, B200SPH_U0, B200SPH_V0, B200SPH_W0,
    B200SPH_RHO0,
    /* fp32 on device */
    B200SPH_P, B200SPH_CS, B200SPH_ARHO, B200SPH_AU, B200SPH_AV, B200SPH_AW,
    B200SPH_AX, B200SPH_AY, B200SPH_AZ, B200SPH_DT_CFL, B200SPH_DT_FORCE,
    B200SPH_NUM_REAL_PROPS,
    /* transport-velocity / EDAC extension (wc/edac.py:724-730).  fp64: advection
     * velocity and the EVOLVED pressure of the EDAC scheme (B200SPH_P above is the
     * fp32 pressure an equation of state derives); fp32: derived fields */
    B200SPH_UHAT = 27, B200SPH_VHAT, B200SPH_WHAT, B200SPH_PF, B200SPH_PF0,
    B200SPH_VOL = 32, B200SPH_PAVG, B200SPH_AUHAT, B200SPH_AVHAT, B200SPH_AWHAT,
    B200SPH_AP,
    B200SPH_NUM_PROPS = 38,
    /* elastic-dynamics extension (solid_mech/basic.py:52-59), device memory allocated
     * on first use.  Symmetric tensors as 00 01 02 11 12 22, the velocity gradient as
     * 00 01 02 10 11 12 20 21 22.  fp64: deviatoric stress (integrated) and its copy;
     * fp32: velocity gradient, artificial stress, stress rate.
     * NOTE: written after this round's GPU budget was spent -- compiled, not yet run on
     * hardware (tests/test_zz_gpu_solid_unvalidated.py) */
    B200SPH_S00 = 70, B200SPH_S01, B200SPH_S02, B200SPH_S11, B200SPH_S12, B200SPH_S22,
    B200SPH_S000 = 76, B200SPH_S010, B200SPH_S020, B200SPH_S110, B200SPH_S120, B200SPH_S220,
    B200SPH_V00 = 82, B200SPH_V01, B200SPH_V02, B200SPH_V10, B200SPH_V11, B200SPH_V12,
    B200SPH_V20, B200SPH_V21, B200SPH_V22,
    B200SPH_R00 = 91, B200SPH_R01, B200SPH_R02, B200SPH_R11, B200SPH_R12, B200SPH_R22,
    B200SPH_AS00 = 97, B200SPH_AS01, B200SPH_AS02, B200SPH_AS11, B200SPH_AS12, B200SPH_AS22,
    B200SPH_SOLID_PROPS_END = 103,
    /* 32-bit integer props */
    B200SPH_GID = 64, B200SPH_TAG = 65, B200SPH_PID = 66,
    /* fp64 properties the pool does not know, created on first use for the generic-equation
     * fallback (b200sph_user_property): ids B200SPH_USER0 .. B200SPH_USER0 + 15 */
    B200SPH_USER0 = 110
};

/* pair-equation bits of one (destination array, source array) loop */
enum {
    B200SPH_EQ_SUMMATION_DENSITY = 1, /* basic_equations.py:19-29   */
    B200SPH_EQ_CONTINUITY = 2,        /* basic_equations.py:180-192 */
    B200SPH_EQ_MOMENTUM = 4,          /* wc/basic.py:129-269        */
    B200SPH_EQ_XSPH = 8,              /* basic_equations.py:260-300 */
    B200SPH_EQ_MONAGHAN_AV = 16,      /* basic_equations.py:195-257 */
    B200SPH_EQ_LAMINAR = 32           /* LaminarViscosity wc/viscosity.py:5-27: WCSPHScheme(nu != 0), scheme.py:486-496 */
};

/* One Group's pair loops (acceleration_eval_cython.mako:10-154) after the
 * MegaGroup regrouping (acceleration_eval.py:127-162): eqmask[d][s] is the OR
 * of the equations with destination array d and source array s. */
typedef struct {
    uint32_t eqmask[B200SPH_MAX_ARRAYS][B200SPH_MAX_ARRAYS];
    int32_t real_only;          /* Group(real=True): dests = real particles  */
    int32_t tensile_correction; /* MomentumEquation(tensile_correction=...)  */
    double c0, alpha, beta;     /* MomentumEquation / MonaghanArtificialViscosity */
    double gx, gy, gz;          /* MomentumEquation body force               */
    double eps_xsph;            /* XSPHCorrection(eps=...)                   */
    double nu, eta;             /* LaminarViscosity(nu, eta = 0.01) (ABI 5: appended) */
} b200sph_pair_program;

/* pair-equation bits of the EDAC scheme's momentum group */
enum {
    B200SPH_TVF_PGRAD = 1,   /* MomentumEquationPressureGradient   wc/edac.py:389-488 */
    B200SPH_TVF_AV = 2,      /* MomentumEquationArtificialViscosity transport_velocity.py:389-448 */
    B200SPH_TVF_VISC = 4,    /* MomentumEquationViscosity          transport_velocity.py:328-386 */
    B200SPH_TVF_ASTRESS = 8, /* MomentumEquationArtificialStress   transport_velocity.py:451-545 */
    B200SPH_TVF_EDAC = 16,   /* EDACEquation                       wc/edac.py:354-386 */
    B200SPH_TVF_NOSLIP = 32, /* SolidWallNoSlipBC (sources: the walls) transport_velocity.py:548-638 */
    /* the external-flow branch (pb == 0, wc/edac.py:882-971) instead of PGRAD + ASTRESS: */
    B200SPH_TVF_MOM = 64,    /* edac.MomentumEquation (number density)  wc/edac.py:301-352 */
    B200SPH_TVF_XSPH = 128   /* XSPHCorrection(dest = f, sources = [f]) basic_equations.py:260-300 */
};

/* The Groups EDACScheme._get_internal_flow_equations (wc/edac.py:776-880) emits: every
 * fluid array is a destination and a source.  With solid walls (solid_mask; :815-822) group 1
 * continues on the wall arrays -- SourceNumberDensity, VolumeSummation, SolidWallPressureBC,
 * SetWallVelocity (k_tvf_wall) --, the average pressure becomes a Group of its own behind the
 * wall pressure (:840-842, passes bit 2) and the walls are sources of the fluids' density,
 * average pressure, pressure gradient, artificial viscosity, EDAC equation and of
 * SolidWallNoSlipBC.  A wall array keeps u v w (prescribed velocity) and au av aw (prescribed
 * acceleration); what the wall equations compute is read back under these property ids:
 * p -> B200SPH_P, V -> B200SPH_VOL, wij -> B200SPH_PAVG, uf vf wf -> B200SPH_AUHAT.., ug vg wg ->
 * B200SPH_UHAT.. (the transport-velocity slots a wall does not otherwise use). */
typedef struct {
    uint32_t fluid_mask; /* bit a: array a is a fluid                           */
    int32_t bql;         /* ComputeAveragePressure (wc/edac.py:62-79) in group 1 */
    uint32_t eqbits;     /* B200SPH_TVF_* of group 2                            */
    int32_t passes;      /* bit 0: group 1 (TVF SummationDensity [+ average p],
                          * real=False; + the wall equations), bit 1: group 2
                          * (real=True), bit 2: the average-pressure Group of a
                          * scheme with walls (real=True)                         */
    double pb, nu, edac_nu, c0, rho0, alpha;
    double gx, gy, gz;   /* body force; damped by tdamp at time t (:483-488); the
                          * wall pressure takes it undamped (:141-161)            */
    double tdamp, t;
    uint32_t solid_mask; /* bit a: array a is a solid wall (ABI 5: appended)     */
    int32_t clamp_p;     /* ClampWallPressure (wc/edac.py:169-174) on the walls   */
    double eps_xsph;     /* XSPHCorrection(eps) of the external-flow branch       */
} b200sph_tvf_program;

/* The two Groups of ElasticSolidsScheme.get_equations (solid_mech/basic.py:604-651) for
 * elastic solids (destinations and sources) and rigid `solids` (sources only).  Group 1: IsothermalEOS (:93-101), VelocityGradient2D/3D
 * (basic_equations.py:67-148), MonaghanArtificialStress (:104-242); group 2:
 * ContinuityEquation, MomentumEquationWithStress (:245-387),
 * MonaghanArtificialViscosity, HookesDeviatoricStressRate (:390-505), XSPHCorrection. */
typedef struct {
    uint32_t elastic_mask; /* bit a: array a is an elastic solid                    */
    int32_t grad3d;        /* 0 VelocityGradient2D (what the scheme emits), 1 ..3D  */
    int32_t passes;        /* bit 0: group 1, bit 1: group 2                        */
    int32_t ghost_group1;  /* != 0: group 1 also runs on ghosts (like Group(real=False));
                            * the slab decomposition then imports two kernel supports so
                            * that a ghost's p and artificial stress are THIS evaluation's,
                            * as in a serial run, instead of the carried values a
                            * reference Remote particle has (parallel_manager.pyx:512-530) */
    double eps;            /* MonaghanArtificialStress(eps)                         */
    double alpha, beta;    /* MonaghanArtificialViscosity                           */
    double eps_xsph;       /* XSPHCorrection(eps)                                   */
    /* the array constants of get_particle_array_elastic_dynamics (:61-83), per array */
    double c0_ref[B200SPH_MAX_ARRAYS], rho_ref[B200SPH_MAX_ARRAYS],
        wdeltap[B200SPH_MAX_ARRAYS], n[B200SPH_MAX_ARRAYS], G[B200SPH_MAX_ARRAYS];
    uint32_t source_mask;  /* bit a: array a is a source of the pair equations: the elastic
                            * arrays plus the scheme's rigid `solids` (all = solids +
                            * elastic_solids, :613), which are destinations of nothing and
                            * contribute with the p / s / r they carry.  0 = elastic_mask */
    uint32_t reserved;
} b200sph_solid_program;

typedef struct {
    double cell_size;  /* DomainManager.cell_size  nnps_base.pyx:942-978    */
    double hmin;       /* radius_scale * min(h)    nnps_base.pyx:970        */
    double xmin[3];    /* NNPS.xmin                nnps_base.pyx:1520-1575  */
    double xmax[3];
    int32_t ncells[3]; /* LinkedListNNPS.ncells_per_dim linked_list_nnps.pyx:293-326 */
    int64_t n_cells;
    int64_t n_particles; /* particles binned (all arrays, real + ghost)     */
} b200sph_grid_info;

typedef struct {
    double ms_nnps;     /* device time in nnps_update since last reset      */
    double ms_pair;     /* device time in pair_pass kernels                 */
    double ms_other;    /* eos / stage / reductions                         */
    int64_t pair_launches;
    int64_t kernel_launches; /* every kernel this library launched          */
    int64_t pairs;      /* directed pair interactions counted (if enabled)  */
    int64_t full_builds;   /* nnps_update calls that re-sorted the particles   */
    int64_t light_updates; /* nnps_update calls that only refreshed positions
                              (persistent neighbour lists still valid)          */
    int64_t list_builds;   /* neighbour list (re)builds                         */
    int64_t list_entries_per_particle; /* list capacity reserved per particle   */
    int64_t deferred_failed; /* deferred drift checks that forced a repeat      */
    int64_t fused_stages;  /* stage calls served by the fused stage + pack kernel      */
    int64_t overlapped;    /* pair passes that ran their ghost-free CTAs under the halo  */
    int64_t proactive_builds; /* list rebuilds done one evaluation early: the extrapolated drift
                              said the deferred check of that evaluation would fail        */
    int64_t chunks_interior, chunks_boundary; /* CTAs of the list consumers without / with a
                              ghost among their destinations or neighbours (current build;
                              0 / 0 without ghosts)                                          */
    double ms_halo_chain;  /* overlapped evaluations (profiling on): device time from the fork of the
                              communication stream to the end of the ghost scatter, summed      */
    double ms_pair_wall;   /* ... and to the end of BOTH pair launches (what the evaluation's
                              pair work costs in wall time, protocol included)                  */
    double ms_halo_sent, ms_halo_reduced; /* ... to the end of the sends / of the all-rank agreement */
} b200sph_stats;

/* ---- lifecycle: what selecting a backend does in the reference
 *      (get_config().use_cuda / use_opencl -> a compyle context,
 *      pysph/sph/acceleration_eval.py:214-223, pysph/base/device_helper.py:52-60) */
int b200sph_abi_version(void);
int b200sph_create(int device, b200sph_ctx **out);
int b200sph_destroy(b200sph_ctx *ctx);
const char *b200sph_last_error(b200sph_ctx *ctx);
/* run on this cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream) so
 * that torch.distributed collectives order with our kernels; NULL = a private
 * non-blocking stream.  The legacy default stream is cudaStreamLegacy = (void*)1 */
int b200sph_set_stream(b200sph_ctx *ctx, void *cuda_stream);
int b200sph_synchronize(b200sph_ctx *ctx);

/* ---- device mirror of the ParticleArrays: DeviceHelper push/pull/resize
 *      pysph/base/device_helper.py:47-250 --------------------------------- */
/* returns the array index (>= 0) */
int b200sph_add_array(b200sph_ctx *ctx, const char *name, int64_t n,
                      int64_t n_real, int64_t capacity);
int b200sph_resize_array(b200sph_ctx *ctx, int arr, int64_t n, int64_t n_real);
int b200sph_get_array_size(b200sph_ctx *ctx, int arr, int64_t *n, int64_t *n_real);
int b200sph_push_f64(b200sph_ctx *ctx, int arr, int prop, const double *host,
                     int64_t start, int64_t count);
int b200sph_pull_f64(b200sph_ctx *ctx, int arr, int prop, double *host,
                     int64_t start, int64_t count);
int b200sph_push_u32(b200sph_ctx *ctx, int arr, int prop, const uint32_t *host,
                     int64_t start, int64_t count);
int b200sph_pull_u32(b200sph_ctx *ctx, int arr, int prop, uint32_t *host,
                     int64_t start, int64_t count);
/* on != 0: push/pull only enqueue the copies on the context's stream and return;
 * the host buffers (which should be pinned) stay borrowed until the next
 * b200sph_synchronize.  Default off: every push/pull call is synchronous. */
int b200sph_set_async_copies(b200sph_ctx *ctx, int on);
/* device pointer of a property region of one array (for zero-copy use by
 * torch / NCCL plumbing); fp64 props -> double*, fp32 props -> float* */
int b200sph_device_ptr(b200sph_ctx *ctx, int arr, int prop, void **out);

/* ---- NNPS: kernel choice, DomainManager.update, NNPS.update ------------- */
/* kernel.__dict__ (dim, radius_scale via the kernel id)
 * acceleration_eval_cython_helper.py:242-246 */
int b200sph_set_kernel(b200sph_ctx *ctx, int kernel, int dim);
/* DomainManager(xmin.., periodic_in_x..) nnps_base.pyx:226-347: a periodic axis d
 * wraps positions into [lo[d], hi[d]] at every update_domain (_box_wrap_periodic,
 * :699-743) and lets particles interact with the periodic images of the others.
 * Images are NOT materialised as tag=Ghost particles (_create_ghosts_periodic,
 * :744-940): the cell grid tiles the axis exactly and neighbour cells wrap. */
int b200sph_set_domain(b200sph_ctx *ctx, const double lo[3], const double hi[3],
                       const int periodic[3]);
/* DomainManager(mirror_in_x ...) nnps_base.pyx:329-335, _create_ghosts_mirror :506-689
 * (after b200sph_set_domain, which gives the planes lo / hi): every particle within
 * n_layers cells (+ the list skin) of a mirror plane gets an image with tag = Ghost on the
 * other side -- position reflected, the normal velocity component negated, x y z u v w
 * rho h m copied (p, cs follow from the EOS) -- and images of images at the corners in the
 * reference's order (x, then y of real + x images, then z of everything).  The reference
 * re-selects at every update_domain; here the selection is made when the neighbour lists
 * are built and b200sph_nnps_update refreshes the images' values before every evaluation.
 * WCSPH arrays, one GPU (no slab decomposition), no periodic axis in the same domain. */
int b200sph_set_mirror(b200sph_ctx *ctx, const int mirror[3], double n_layers);
/* NNPS.update_domain -> CPUDomainManager._compute_cell_size_for_binning
 * nnps_base.pyx:450-483, :942-978 */
int b200sph_update_domain(b200sph_ctx *ctx);
/* NNPS.update nnps_base.pyx:1471-1510: bounds (:1520-1575), cell grid
 * (linked_list_nnps.pyx:293-343; error if > 2^28 cells), binning (:235-286)
 * -- here a deterministic counting sort + cell-relative fp32 repack */
int b200sph_nnps_update(b200sph_ctx *ctx);
/* The same update, but when the persistent neighbour lists are reused the
 * measurement that proves them valid (drift <= skin) is only ENQUEUED: the
 * caller enqueues the evaluation right behind it and then calls
 * b200sph_nnps_confirm, which waits for the measurement (the GPU is busy with
 * the evaluation meanwhile).  *redo = 1 means the lists were stale: call
 * b200sph_nnps_update (it rebuilds) and repeat the evaluation -- every field an
 * evaluation writes is overwritten by the repeat.  stage / dt_factors / pull /
 * halo_pack / migrate_out / get_neighbors fail on an unconfirmed stale update. */
int b200sph_nnps_update_deferred(b200sph_ctx *ctx);
int b200sph_nnps_confirm(b200sph_ctx *ctx, int *redo);
/* the attributes NNPS exposes after update(): cell_size, hmin, xmin, xmax,
 * ncells_per_dim, n_cells (nnps_base.pxd:279-371, linked_list_nnps.pyx:293-343) */
int b200sph_get_grid(b200sph_ctx *ctx, b200sph_grid_info *out);
/* NNPS.get_nearest_particles(src, dst, d_idx, nbrs) nnps_base.pyx:1268-1290:
 * runs the SAME accept test as the pair kernel.  Writes up to cap source
 * indices (ascending); returns the full neighbour count, or <0 on error. */
int64_t b200sph_get_neighbors(b200sph_ctx *ctx, int dst_arr, int src_arr,
                              int64_t d_idx, uint32_t *out, int64_t cap);

/* ---- AccelerationEval.compute building blocks --------------------------- */
/* TaitEOS.loop (hg=0) wc/basic.py:60-65 / TaitEOSHGCorrection.loop (hg=1)
 * wc/basic.py:118-126 on one array */
int b200sph_eos(b200sph_ctx *ctx, int arr, int hg, double rho0, double c0,
                double gamma, double p0, int real_only);
/* UpdateSmoothingLengthFerrari.loop wc/basic.py:458-463 */
int b200sph_ferrari_h(b200sph_ctx *ctx, int arr, double hdx, int dim,
                      int real_only);
/* one Group of pair equations: initialize + loop over all sources + post_loop
 * fused in one kernel.  pairs_out (may be NULL) receives the number of
 * directed pair interactions (sum of neighbour-list lengths over the enabled
 * (dest, source) loops); counting costs one extra atomic per warp. */
int b200sph_pair_pass(b200sph_ctx *ctx, const b200sph_pair_program *prog,
                      int64_t *pairs_out);
/* on != 0: no program or stepper run on this context writes h or m on the device (host pushes
 * may still change them).  With it, a pair pass of the WCSPH Group may gather one 32-byte record
 * per neighbour instead of 48 bytes when every particle has the same h, m is uniform within each
 * source class and every source array's equation of state is Tait with gamma = 7 (at most two
 * source classes, no ghosts; env B200SPH_PAIR_R32=0 turns it off).  b200sph_ferrari_h and a
 * generic launch that writes h switch it off.  Default off. */
int b200sph_set_hm_static(b200sph_ctx *ctx, int on);
/* Group(start_idx, stop_idx) (equation.py:448-520; D_START_IDX / NP_DEST of the generated
 * loop, acceleration_eval_cython_helper.py:259-284): the NEXT b200sph_pair_pass only touches
 * the destinations [start, stop) of array `arr` (indices into the array; stop = -1: to the end,
 * i.e. what real_only admits); arrays not named keep all their destinations.  One-shot: the
 * pass clears it. */
int b200sph_set_dest_range(b200sph_ctx *ctx, int arr, int64_t start, int64_t stop);

/* ---- generic-equation fallback (SURVEY.md 8f-4) -----------------------------------------
 * Stands where the reference compiles ANY Equation's Python bodies (pysph/sph/equation.py:
 * 389-420, acceleration_eval_cython.mako:10-155): pysph_b200/codegen.py translates the
 * initialize / loop / post_loop bodies of equations the library has no hand-written kernel
 * for into CUDA C, compiles it with NVRTC for sm_100a, and hands the cubin to the library:
 *   user_property    create (zero-filled) the fp64 property `prop` (B200SPH_USER0 + k) for every
 *                    array; push_f64 / pull_f64 / device_ptr accept the id afterwards
 *   generic_load     load a cubin whose kernels take one b200sph_generic_args by value
 *                    (pysph_b200/csrc/generic_args.h); returns a module handle >= 0
 *   generic_launch   run phase 0 (initialize) / 1 (loop over the persistent neighbour lists,
 *                    same accept test as the hand-written pair kernels) / 2 (post_loop) of
 *                    kernel `kernel` for the destinations of array dest_arr; honours
 *                    b200sph_set_dest_range; `writes` bit 0: a body stores to x y z h, bit 1:
 *                    to any other property the packed pair records are made from
 * One GPU only (the slab decomposition does not carry user properties). */
int b200sph_user_property(b200sph_ctx *ctx, int prop);
int b200sph_generic_load(b200sph_ctx *ctx, const void *image, int64_t size);
int b200sph_generic_launch(b200sph_ctx *ctx, int module, const char *kernel, int dest_arr, int phase,
                           unsigned src_mask, int real_only, double t, double dt, int writes);

/* The two Groups of EDACScheme._get_internal_flow_equations (wc/edac.py:776-880) in
 * the generated AccelerationEval.compute (acceleration_eval_cython.mako:10-154): group 1 computes
 * V = sum W, rho = m V (transport_velocity.py:24-58) and the neighbour-average
 * pressure; group 2 the momentum terms (au.., auhat..) and ap.  Both walk the same
 * persistent neighbour lists as pair_pass.  pairs_out may be NULL. */
int b200sph_tvf_pass(b200sph_ctx *ctx, const b200sph_tvf_program *prog,
                     int64_t *pairs_out);
/* EDACTVFStep wc/edac.py:491-540; which: 0 initialize, 1 stage1, 2 stage2 */
int b200sph_stage_tvf(b200sph_ctx *ctx, int arr, int which, double dt);
/* the same with dt read from the device-resident time-control block */
int b200sph_stage_tvf_dev(b200sph_ctx *ctx, int arr, int which);
/* EDACStep (wc/edac.py:82-133), the stepper of the scheme WITHOUT transport velocity (pb == 0):
 * as stage_tvf, but positions move with the XSPH-corrected velocity ax ay az */
int b200sph_stage_edac(b200sph_ctx *ctx, int arr, int which, double dt);
int b200sph_stage_edac_dev(b200sph_ctx *ctx, int arr, int which);

/* The elastic-dynamics evaluation (see b200sph_solid_program); same neighbour lists as
 * pair_pass.  NOT YET RUN ON HARDWARE (see the property block above). */
int b200sph_solid_pass(b200sph_ctx *ctx, const b200sph_solid_program *prog,
                       int64_t *pairs_out);
/* SolidMechStep integrator_step.py:173-252 (e / ae are not mirrored: the scheme has no
 * energy equation, so e stays what it is) */
int b200sph_stage_solid(b200sph_ctx *ctx, int arr, int which, double dt);
int b200sph_stage_solid_dev(b200sph_ctx *ctx, int arr, int which);

/* ---- Integrator stages: WCSPHStep integrator_step.py:38-91 -------------- */
/* which: 0 initialize, 1 stage1, 2 stage2; arr = -1 -> every array */
int b200sph_stage(b200sph_ctx *ctx, int arr, int which, double dt);
/* out = {max dt_cfl, max dt_force (real particles; -1 if none),
 *        min h (all particles, starting from 1.0)}
 * Integrator._get_dt_adapt_factors / compute_h_minimum integrator.py:62-81,146-159 */
int b200sph_dt_factors(b200sph_ctx *ctx, double out[3]);

/* ---- device-resident time step: the adaptive dt (Integrator.compute_time_step
 *      integrator.py:161-200), its damping and the t += dt bookkeeping of the solve
 *      loop (solver.py:478-491, :647-688) without a host round trip per step.
 * The time-control block is 8 doubles of DEVICE memory:
 *   [0] dt of the next step (damped)   [1] t   [2] proposed dt (local; the caller may
 *   MIN-reduce it over ranks between dt_propose and dt_commit)   [3] h_minimum
 * external_block8 != NULL: use the caller's device memory (e.g. a torch tensor a
 * collective can reduce in place); NULL: the library's own.  *dev_block = its address */
int b200sph_time_control(b200sph_ctx *ctx, double *external_block8, double **dev_block);
int b200sph_time_set(b200sph_ctx *ctx, double t, double dt);
/* out = {dt, t}; waits for the stream */
int b200sph_time_get(b200sph_ctx *ctx, double out[2]);
/* b200sph_stage with dt read from the block (which = 1 uses dt / 2).
 * Fast path (both b200sph_stage and b200sph_stage_dev, arr = -1, which = 1 or 2, a reusable
 * neighbour build, no periodic / mirror domain; B200SPH_FUSE=0 switches it off): ONE kernel
 * does the stage, refreshes the packed pair records of the real particles for the next
 * evaluation (positions, drift of the build, state with the equation-of-state calls of
 * the last evaluation applied to the records) and, after stage2, reduces the adaptive-dt
 * factors -- the work of k_stage + k_pack_pos_light + k_pack_state + k_reduce_dt in one
 * sweep over the state.  Results are bitwise those of the separate kernels; the pool's
 * rho / p / cs change only when the next evaluation issues its b200sph_eos calls. */
int b200sph_stage_dev(b200sph_ctx *ctx, int arr, int which);
/* enqueue: reduce dt_cfl / dt_force / h, then block[2] = cfl * min(hmin / max_cfl,
 * sqrt(hmin / sqrt(max_force))), or 1e20 when nothing constrains it (solver.py:655-660);
 * fixed_h keeps the first hmin (integrator.py:170-176) */
int b200sph_dt_propose(b200sph_ctx *ctx, double cfl, int fixed_h);
/* enqueue: if (advance) t += dt;  undamped = dt / prev_factor;
 * dt = new_factor * (adaptive ? (block[2] < 1e20 || in_parallel ? block[2] : undamped)
 *                             : undamped)                          (solver.py:647-688)
 * snapshot_slot 0/1: also copy {dt, t} to pinned host memory for b200sph_time_snapshot;
 * -1: no snapshot */
int b200sph_dt_commit(b200sph_ctx *ctx, double prev_factor, double new_factor,
                      int in_parallel, int adaptive, int advance, int snapshot_slot);
/* b200sph_dt_propose + b200sph_dt_commit in one launch for a run on ONE rank (nothing to
 * reduce between them): the whole of Solver._get_timestep + `t += dt` (solver.py:478-491,
 * :647-688, :756-776) is one tiny kernel per step.  When the fused stage kernel has left the
 * factors of the last evaluation in the reduction slots (see b200sph_stage_dev) no
 * reduction runs here. */
int b200sph_dt_advance(b200sph_ctx *ctx, double cfl, int fixed_h, double prev_factor,
                       double new_factor, int adaptive, int advance, int snapshot_slot);
/* wait for the snapshot of `slot` only (not for later work): out = {dt, t} */
int b200sph_time_snapshot(b200sph_ctx *ctx, int slot, double out[2]);
/* the final time of the run and the tolerance it is compared with (solver.py:757-760,
 * :771-773; the reference's eps grows with the iteration count, :488, so the caller sets
 * it before every commit): dt_commit then makes the last step land on t_final --
 * dt = t_final - t when t + dt > t_final - eps -- and leaves dt alone once
 * |t_final - t| < eps.  Default: +inf (never). */
int b200sph_time_final(b200sph_ctx *ctx, double t_final, double eps);

/* ---- halo exchange helpers (replace ParallelManager.update,
 *      parallel_manager.pyx:512-632).  Buffers are DEVICE pointers owned by
 *      the caller (torch tensors handed to NCCL). ------------------------- */
#define B200SPH_HALO_FIELDS 9     /* x y z u v w rho h m (fp64 each)          */
#define B200SPH_MIGRATE_FIELDS 17 /* the 16 fp64 state props (x..m, x0..rho0) + gid */
/* once an elastic-dynamics property has been named (solid_mech/basic.py:32-90) the
 * deviatoric stress travels too, and cs (which no equation of that scheme recomputes):
 * ghosts carry s00 s01 s02 s11 s12 s22 cs after the 9 fields, migrating particles
 * s00..s22, the stage copies s000..s220 and cs after the 17 */
#define B200SPH_HALO_FIELDS_SOLID 16
#define B200SPH_MIGRATE_FIELDS_SOLID 30
/* the field counts of THIS context's messages (9 / 17, or 16 / 30): what the caller sizes
 * its buffers with and passes to b200sph_halo_append as nfields */
int b200sph_halo_layout(b200sph_ctx *ctx, int *halo_fields, int *migrate_fields);
/* select the real particles of `arr` with lo <= x < hi and write their
 * B200SPH_HALO_FIELDS doubles field-major and TIGHT (field f of particle k at
 * dev_buf[f * count + k]); *count = number selected; error if count > cap.
 * slot = 0 / 1 (left / right neighbour) also remembers the selection for
 * b200sph_halo_pack_selected; slot = -1 does not */
int b200sph_halo_pack(b200sph_ctx *ctx, int arr, int slot, double lo, double hi,
                      double *dev_buf, int64_t cap, int64_t *count);
/* pack the CURRENT values of the particles remembered by the last
 * b200sph_halo_pack(arr, slot, ...) -- the per-evaluation ghost refresh that
 * replaces a full re-import while the neighbour lists stay valid */
int b200sph_halo_pack_selected(b200sph_ctx *ctx, int arr, int slot, double *dev_buf,
                               int64_t cap, int64_t *count);
/* overwrite the B200SPH_HALO_FIELDS of the existing ghosts
 * [ghost_first, ghost_first + n) of `arr` (indices among the ghosts) */
int b200sph_halo_overwrite(b200sph_ctx *ctx, int arr, int64_t ghost_first,
                           const double *dev_buf, int64_t stride, int64_t n);
/* the refresh message of ALL arrays for neighbour `slot` in one kernel: the block
 * of array a starts at 9 * (count_0 + .. + count_{a-1}) doubles, field-major and
 * tight.  dev_buf may be a PEER pointer obtained with b200sph_ipc_open (the
 * neighbour's staging buffer): pack and send are then the same kernel, writing
 * over NVLink */
int b200sph_halo_pack_selected_all(b200sph_ctx *ctx, int slot, double *dev_buf,
                                   int64_t cap_doubles, int64_t *ndoubles);
/* the inverse on the receiving rank: counts[a] particles of array a (block
 * layout as above) over the existing ghosts starting at ghost_first[a] */
int b200sph_halo_overwrite_all(b200sph_ctx *ctx, const int64_t *ghost_first,
                               const int64_t *counts, const double *dev_buf);
/* peer-memory staging buffers (ranks of one node): allocate + export a 64-byte
 * cudaIpcMemHandle_t / map a neighbour's buffer / unmap (owner = 0) or free (1) */
int b200sph_ipc_alloc(b200sph_ctx *ctx, int64_t bytes, void **dev_ptr, void *handle64);
int b200sph_ipc_open(b200sph_ctx *ctx, const void *handle64, void **dev_ptr);
int b200sph_ipc_close(b200sph_ctx *ctx, void *dev_ptr, int owner);
/* out[0] = 2 max|x - x_build| + k max(h - h_build) over the particles of the
 * current neighbour build (-1 if there is no reusable build), out[1] = the skin
 * S: the build can be reused while out[0] <= out[1] */
int b200sph_nnps_drift(b200sph_ctx *ctx, double out[2]);
/* the same measurement without a host round trip: writes out[0] / out[1] (the
 * fraction of the skin used up) to a DEVICE double, stream ordered, so that a
 * collective can reduce it directly.  Returns 1 (and writes nothing) if there is
 * no reusable build, 0 otherwise */
int b200sph_nnps_drift_device(b200sph_ctx *ctx, double *dev_ratio);
/* the caller decided (collectively, over all ranks) that the current build is
 * kept for the next nnps_update: that update then only refreshes the packed
 * positions and does not repeat the drift measurement (saves a host sync) */
int b200sph_nnps_keep_build(b200sph_ctx *ctx);

/* ---- peer protocol: the ghost refresh of an evaluation, overlapped with the interior
 *      pair work, and the scalar agreements that go with it -- no library collective.
 * Replaces, for the ranks of ONE node, what the reference does serially in front of every
 * evaluation (ParallelManager.update, parallel_manager.pyx:512-530, called from
 * Integrator.compute_accelerations, integrator.py:274-286) and its dt all-reduce
 * (update_time_steps, parallel_manager.pyx:454-465).
 * Every rank owns a small mailbox in device memory that the other ranks write into over
 * NVLink (cudaIpc); payload, __threadfence_system(), then an epoch word the reader polls.
 *   peer_init     allocate + export this rank's mailbox (handle64: 64 bytes)
 *   peer_connect  map every rank's mailbox (handles: world x 64 bytes, rank order)
 * One refresh epoch, in THIS order; every call only enqueues work on two further
 * high-priority streams (communication, agreement).  publish + send are merged into ONE
 * launch at peer_reduce and the recv calls into one at peer_end; the agreement has its own
 * stream because a rank's ghosts need its two neighbours only, the decision every rank:
 *   peer_begin    measure the drift of the neighbour build if the fused stage kernel has
 *                 not, then let the communication stream wait for the main stream;
 *                 returns 1 if there is no reusable build (publish says so to everyone)
 *   peer_publish  {used-up fraction of the list skin, dt proposal | +inf} to every rank
 *   peer_send     b200sph_halo_pack_selected_all into the neighbour's staging buffer
 *                 (remote_staging: its buffer mapped with b200sph_ipc_open) + the
 *                 data-ready flag in its mailbox; side = 0: I am its RIGHT neighbour's
 *                 left... precisely: side is the slot the RECEIVER reads, 0 = message from
 *                 its left neighbour, 1 = from its right neighbour
 *   peer_reduce   wait for every rank's scalars: MAX fraction -> the decision (device,
 *                 and pinned host memory for peer_decision), MIN dt -> block[2]
 *   peer_recv     wait for the data-ready flag `side`, then b200sph_halo_overwrite_all
 *                 from the local staging buffer, including the ghosts' packed pair
 *                 records (position + state with the last evaluation's EOS calls)
 *   peer_end      from here b200sph_pair_pass may run the destinations that do not
 *                 depend on ghosts while the above is still in flight; every other entry
 *                 point that touches particle data first waits for it
 *   peer_decision (host) wait for the decision of the current epoch only: *ratio_max > 0.9
 *                 means some rank's lists have expired -- discard the evaluation, run the
 *                 full exchange (the caller's protocol, as with b200sph_nnps_confirm)
 *   peer_allreduce_dt  the stand-alone agreement on the time step: block[2] = MIN over
 *                 ranks of block[2], enqueued on the main stream (between b200sph_dt_propose
 *                 and b200sph_dt_commit) */
int b200sph_peer_init(b200sph_ctx *ctx, int rank, int world, void *handle64);
int b200sph_peer_connect(b200sph_ctx *ctx, const void *handles);
int b200sph_peer_begin(b200sph_ctx *ctx);
int b200sph_peer_publish(b200sph_ctx *ctx, int have_build, int with_dt);
int b200sph_peer_send(b200sph_ctx *ctx, int slot, int nb_rank, int side, double *remote_staging,
                      int64_t cap_doubles);
int b200sph_peer_reduce(b200sph_ctx *ctx, int with_dt);
int b200sph_peer_recv(b200sph_ctx *ctx, int side, const int64_t *ghost_first, const int64_t *counts,
                      const double *local_staging);
/* b200sph_dt_commit behind the agreement (on its stream), between peer_reduce(with_dt = 1)
 * and peer_end: the time-step agreement of the step that has just ended rides on the refresh of
 * the next step's first evaluation (the new dt is first needed by its stage1) */
int b200sph_peer_commit_dt(b200sph_ctx *ctx, double prev_factor, double new_factor, int adaptive,
                           int advance, int snapshot_slot);
int b200sph_peer_end(b200sph_ctx *ctx);
int b200sph_peer_decision(b200sph_ctx *ctx, double *ratio_max);
int b200sph_peer_allreduce_dt(b200sph_ctx *ctx);
/* append n particles from dev_buf (field f of particle k at
 * dev_buf[f * stride + k]) after the current particles of `arr`.
 * nfields = B200SPH_HALO_FIELDS: ghosts (tag Remote), other props zeroed;
 * nfields = B200SPH_MIGRATE_FIELDS with as_real != 0: real particles arriving
 * by migration (the array must hold no ghosts at that moment) */
int b200sph_halo_append(b200sph_ctx *ctx, int arr, const double *dev_buf,
                        int64_t stride, int64_t n, int nfields, int as_real);
/* drop every ghost particle of `arr` (n <- n_real)
 * parallel_manager.pyx:519 remove_remote_particles */
int b200sph_drop_ghosts(b200sph_ctx *ctx, int arr);
/* remove the real particles of `arr` with x outside [lo, hi) after packing
 * their B200SPH_MIGRATE_FIELDS doubles into dev_buf: the particles that left
 * below lo first (field-major, stride count[0]) then those at x >= hi
 * (field-major, stride count[1], starting at dev_buf + 17 * count[0]) */
int b200sph_migrate_out(b200sph_ctx *ctx, int arr, double lo, double hi,
                        double *dev_buf, int64_t cap, int64_t count[2]);

/* ---- asynchronous output (Solver.dump_output at pfreq, solver.py:520-560; the
 * reference's GPU arrays copy every property back with the loop stopped) ------------
 * take: snapshot `nseg` (array, property) segments of count[i] leading particles each
 *   (count = n_real drops the ghosts) into a library-owned device buffer, in stream
 *   order: fp64 properties as they are, fp32 ones widened to double, integer ones as
 *   4-byte values; arr[i] = -1 snapshots the first count[i] doubles {dt, t, ...} of the
 *   time-control block.  Returns at once; the time loop continues.
 * fetch: copy segment `seg` to host memory (8 * count bytes, 4 * count for integers) on
 *   a private stream and wait for THAT copy only; may be called from another host
 *   thread while the owner keeps stepping.
 * release: the buffer may be overwritten by the next take.  One snapshot at a time.
 * Threading: only snapshot_fetch / snapshot_release (and b200sph_last_error) may be called
 * from a second host thread; the error message and the "snapshot open" flag they share
 * with the time loop's thread are guarded. */
int b200sph_snapshot_take(b200sph_ctx *ctx, int nseg, const int *arr, const int *prop,
                          const int64_t *count);
int b200sph_snapshot_fetch(b200sph_ctx *ctx, int seg, void *host, int64_t count);
int b200sph_snapshot_release(b200sph_ctx *ctx);

/* load re-balancing (parallel_manager.pyx:512-530 lb_count/lb_freq, :532-613
 * update_partition): add the number of REAL particles of `arr` per x column
 * [x0 + k / inv_width, x0 + (k + 1) / inv_width), k clamped to 0..nbins-1, to the
 * device counters dev_counts[0..nbins).  The caller zeroes them, weights the arrays
 * (scheme.py:523-527 weights solids lower), sums over ranks and moves the cut planes */
int b200sph_column_counts(b200sph_ctx *ctx, int arr, double x0, double inv_width, int nbins,
                          unsigned long long *dev_counts);

/* ---- bookkeeping -------------------------------------------------------- */
int b200sph_get_stats(b200sph_ctx *ctx, b200sph_stats *out);
/* pair passes since the last reset_stats that ran the 32-byte-record list kernel
 * (b200sph_set_hm_static); kept out of b200sph_stats so that its layout stays */
int b200sph_get_pair_r32_launches(b200sph_ctx *ctx, int64_t *out);
int b200sph_reset_stats(b200sph_ctx *ctx);
/* per-phase CUDA-event timing: 0 off, 1 every phase (ms_nnps, ms_pair, ms_other),
 * 2 the pair kernels only (ms_pair; two events per pair pass instead of ~25 per
 * step).  Event pairs are recorded on the stream (no sync) and resolved by
 * b200sph_get_stats */
int b200sph_set_profiling(b200sph_ctx *ctx, int on);

#ifdef __cplusplus
}
#endif
#endif
