// b200sph.cu -- B200 (sm_100a) evaluator for PySPH's WCSPH per-timestep hot path.
//
// What lives here (see DESIGN.md for the data layout and rooflines):
//   * device mirror of the ParticleArrays: one pool, SoA, fp64 integrated state
//     + fp32 derived fields            (reference: pysph/base/device_helper.py)
//   * NNPS build: bounds/h reductions, cell keys, deterministic counting sort,
//     cell-relative fp32 repack        (reference: pysph/base/nnps_base.pyx:1471-1575,
//                                       linked_list_nnps.pyx:235-382; GPU precedent
//                                       z_order_gpu_nnps_kernels.py:7-47)
//   * fused pair kernel: initialize + loop over all sources + post_loop of
//     SummationDensity / ContinuityEquation / MomentumEquation(+AV) /
//     XSPHCorrection / MonaghanArtificialViscosity
//                                      (reference: acceleration_eval_cython.mako:10-154,
//                                       equation.py:188-297, wc/basic.py:129-269,
//                                       basic_equations.py:19-29,180-300)
//   * TaitEOS / TaitEOSHGCorrection / UpdateSmoothingLengthFerrari, WCSPHStep
//     stages, adaptive-dt reductions   (wc/basic.py:9-126,417-463,
//                                       integrator_step.py:38-91, integrator.py:62-81)
//   * halo pack / append / migrate helpers for the slab decomposition
//                                      (replaces parallel_manager.pyx:512-632)
//
// One translation unit: this file holds the context, the pool and every C-ABI entry
// point; the kernels are included below by family (pool_kernels, scan, nnps_kernels,
// sph_kernels, pair_kernel, pair_list, tvf_kernels, solid_kernels, halo_kernels .cuh).
//
// No CPU fallback: every entry point needs a CUDA device.
#include "b200sph.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <memory>
#include <mutex>
#include <vector>

// --------------------------------------------------------------------------
// small helpers
// --------------------------------------------------------------------------
#define N_F64 16
#define N_F32 11
#define N_U32 3
#define N_F64X 5   // UHAT VHAT WHAT PF PF0 (ids 27..31)
#define N_F32X 6   // VOL PAVG AUHAT AVHAT AWHAT AP (ids 32..37)
#define PT_INVALID 0xFFu
#define PT_GHOST 0x08u

static inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

struct ArrayInfo {
    std::string name;
    int64_t off = 0, cap = 0, n = 0, n_real = 0;
};

struct GridDev {
    double xmin[3];
    double cell[3];   // cell edge per axis (a periodic axis is tiled exactly: L / nc)
    int nc[3];
    int periodic[3];
    int zorder;       // 1: cell ROWS are ordered along the Z-curve of (cy, cz), see grid_row
};

// Cell key = row(cy, cz) * ncx + cx.  x is always the fastest axis, so the 27 neighbour
// cells of a cell are 9 contiguous ranges of the sorted arrays (what the list builder
// streams); the ROWS are ordered row-major (cy + ncy cz) or, zorder, along the Z-curve
// (Morton code) of (cy, cz) -- rows that are close in space are then close in memory
// whatever the aspect ratio of the grid (the reference's GPU NNPS sorts particles by the
// 3-D Morton key of their cell, z_order_nnps.pyx:252-355, z_order.h:24-46).
__host__ __device__ static inline uint32_t part1by1(uint32_t v)
{
    v &= 0x0000ffffu;
    v = (v | (v << 8)) & 0x00ff00ffu;
    v = (v | (v << 4)) & 0x0f0f0f0fu;
    v = (v | (v << 2)) & 0x33333333u;
    v = (v | (v << 1)) & 0x55555555u;
    return v;
}
__host__ __device__ static inline uint32_t compact1by1(uint32_t v)
{
    v &= 0x55555555u;
    v = (v | (v >> 1)) & 0x33333333u;
    v = (v | (v >> 2)) & 0x0f0f0f0fu;
    v = (v | (v >> 4)) & 0x00ff00ffu;
    v = (v | (v >> 8)) & 0x0000ffffu;
    return v;
}
__host__ __device__ static inline uint32_t grid_row(const int zorder, const uint32_t ncy, const uint32_t cy, const uint32_t cz)
{
    return zorder ? (part1by1(cy) | (part1by1(cz) << 1)) : cy + ncy * cz;
}
__host__ __device__ static inline void grid_decode(const int zorder, const uint32_t ncx, const uint32_t ncy, const uint32_t key,
                                                   uint32_t &cx, uint32_t &cy, uint32_t &cz)
{
    cx = key % ncx;
    const uint32_t row = key / ncx;
    if (zorder) {
        cy = compact1by1(row);
        cz = compact1by1(row >> 1);
    } else {
        cy = row % ncy;
        cz = row / ncy;
    }
}

// equation-of-state calls wait here until the next k_pack_state applies them in the
// same pass that gathers the state into the pair records (saves one launch and one
// sweep over rho/p/cs per array and evaluation); eos_flush() runs them stand-alone
// if something reads rho/p/cs before that.
struct EosTab {
    int on[B200SPH_MAX_ARRAYS], hg[B200SPH_MAX_ARRAYS], real_only[B200SPH_MAX_ARRAYS];
    double rho0[B200SPH_MAX_ARRAYS], c0[B200SPH_MAX_ARRAYS], gamma[B200SPH_MAX_ARRAYS], p0[B200SPH_MAX_ARRAYS];
};

// ratio^gamma and ratio^((gamma - 1) / 2) of the Tait equation of state (wc/basic.py:60-65,
// :118-126).  Water's gamma = 7 -- every WCSPH example of the reference -- needs no pow():
// five fp64 multiplications, within 3 ulp of pow() (the results are stored as fp32); any
// other exponent takes the library route.  ONE function for every kernel that evaluates
// the EOS, so that they all produce the same bits.
__host__ __device__ static inline void tait_powers(const double ratio, const double gamma, double &rg, double &rh)
{
    if (gamma == 7.0) {
        const double r2 = ratio * ratio;
        rh = r2 * ratio;
        rg = rh * rh * ratio;
    } else {
        rg = pow(ratio, gamma);
        rh = pow(ratio, 0.5 * (gamma - 1.0));
    }
}

struct PendingEvent {
    cudaEvent_t e0, e1;
    int slot;  // 0 nnps, 1 pair, 2 other
};

struct b200sph_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;            // last error of the calling threads' entry points ...
    std::string err_out;        // ... and the copy b200sph_last_error hands out
    std::mutex err_mu;          // the output thread (snapshot_fetch / release) reports errors too

    int narr = 0;
    ArrayInfo arr[B200SPH_MAX_ARRAYS];
    int64_t pool_cap = 0;   // allocated particles in the pool
    int64_t pool_end = 0;   // off[last] + cap[last]
    double *f64[N_F64] = {nullptr};
    float *f32[N_F32] = {nullptr};
    uint32_t *u32[N_U32] = {nullptr};
    double *f64x[N_F64X] = {nullptr};   // transport-velocity / EDAC extension
    float *f32x[N_F32X] = {nullptr};
    float4 *Dv = nullptr;               // sorted: (uhat-u, vhat-v, what-w, pavg)
    // elastic-dynamics extension, allocated on first use (ensure_solid)
    bool solid_alloc = false;
    double *f64s[12] = {nullptr};       // s00 s01 s02 s11 s12 s22, then their *0 copies
    float *f32s[21] = {nullptr};        // v00..v22 (9), r00..r22 (6), as00..as22 (6)
    float4 *T01 = nullptr, *T2R = nullptr, *R2 = nullptr;   // sorted stress records
    float2 *PT = nullptr;               // sorted: (p, type)
    uint8_t *ptype = nullptr;
    bool ptype_dirty = true;

    int kernel = 0, dim = 3;
    double radius_scale = 2.0;

    // domain manager
    bool periodic[3] = {false, false, false};
    double dom_lo[3] = {0, 0, 0}, dom_hi[3] = {0, 0, 0};
    // mirror boundaries (b200sph_set_mirror): images are materialised as tag=Ghost particles
    bool mirror[3] = {false, false, false};
    double mirror_layers = 2.0;
    struct MirrorSeg {
        int arr, axis, side;
        int64_t count = 0, cap = 0, ghost_first = 0;   // ghost_first: relative to the array's first ghost
        uint32_t *idx = nullptr;                        // sources, relative to the array's offset
    };
    std::vector<MirrorSeg> mirror_segs;                 // in creation order (corner images read earlier ones)
    bool mirror_built = false;
    double cell_size = 1.0, hmin_scaled = 1.0;
    bool domain_valid = false;
    // grid
    b200sph_grid_info grid;
    bool grid_valid = false;
    bool packed_valid = false;  // A / AB hold the CURRENT positions (set by nnps_drift_device, kept by halo_overwrite_all)
    double last_domain_size = 0.0;

    // sort / cell list buffers
    int64_t sort_cap = 0;        // particles
    int64_t cell_cap = 0;        // cells (+1)
    uint32_t *key_of = nullptr;  // [pool] cell key per particle
    uint32_t *off_in = nullptr;  // [pool] arrival rank inside the cell
    uint32_t *cell_cnt = nullptr;
    uint32_t *cell_start = nullptr;
    uint32_t *blk_sums = nullptr;
    int64_t blk_cap = 0;
    uint32_t *perm_tmp = nullptr, *perm = nullptr, *skey = nullptr, *rank = nullptr;
    float4 *A = nullptr, *B = nullptr, *C = nullptr;
    float4 *AB = nullptr;  // {A, B} interleaved (32 B = one sector per particle) for the list consumer's 256-bit gathers
    float4 *R = nullptr;   // 32-byte source records of the R32 list kernel (PairArgs.R)
    int64_t n_sorted = 0;
    bool state_packed = false;
    int force_kernel = 0;       // 0 lists (default), 1 warp kernel (env B200SPH_PAIR_KERNEL)
    int pair_minb = 7;          // resident CTAs per SM k_pair_list is compiled for (env B200SPH_PAIR_MINB: 6, 7, 8)
    int pair_minb_r32 = 8;      // ... its R32 form (7 or 8; the same env sets both): 8 measured 5 % faster than 7
    bool zorder = false;        // cell rows along the Z-curve of (cy, cz) (env B200SPH_ZORDER; measured: profiles/)
    bool pair_spec = true;      // use the WCSPH-only variant of k_pair_list when the program allows (env B200SPH_PAIR_SPEC)
    // persistent neighbour lists
    double skin = 0.1;          // S = skin * radius_scale * hmax, adapted between skin_min and skin_max
    double skin_max = 0.1;      // env B200SPH_SKIN (also what a halo exchange must cover)
    double skin_min = 0.02;
    bool skin_adapt = true;     // env B200SPH_SKIN_ADAPT=0 switches the controller off
    int64_t evals_since_build = 0;  // light updates served by the current build
    double skin_next = -1.0;        // set by retire_build: the skin of the next build (else the geometric rule)
    double S_abs = 0.0;         // absolute skin of the current build
    double cell_int = 1.0;      // internal cell size (cell_size + S)
    GridDev G;                  // frozen device grid of the current build
    float4 *A0 = nullptr;       // packed positions at build time
    uint32_t *lst = nullptr;    // transposed lists: [n/32][capg][32]
    int64_t lst_cap = 0;        // entries allocated
    uint32_t *cnt = nullptr;    // [n] list length per destination
    int capg = 0;               // entries reserved per destination
    bool lists_valid = false;
    bool topo_dirty = true;     // particle set / h pushed: a light update is not enough
    bool drift_ok = false;      // set by nnps_drift when its caller took the (collective) decision
    // deferred drift check (b200sph_nnps_update_deferred / b200sph_nnps_confirm)
    bool defer_check = false;   // the running nnps_update may leave its drift check pending
    bool check_pending = false; // a light update ran on the assumption that the lists are valid
    unsigned *drift_host = nullptr;
    cudaEvent_t drift_evt = nullptr;
    int64_t n_deferred_failed = 0;
    // proactive rebuild: the used-up fraction of the skin at the last two confirmed deferred
    // checks of the current build; when their extrapolation says the NEXT evaluation would
    // fail its check, the lists are rebuilt before it instead of after a wasted evaluation
    double drift_hist[2] = {-1.0, -1.0};
    bool proactive = true;      // env B200SPH_PROACTIVE=0
    int64_t n_proactive = 0;
    // device-resident time control block: [0] dt, [1] t, [2] proposed dt, [3] h_minimum
    double *tc = nullptr;
    bool tc_owned = false;
    double *tc_host = nullptr;          // pinned: 2 snapshot slots x 2 doubles
    double t_final = INFINITY, t_eps = 0.0;  // b200sph_time_final: the last dt lands on t_final
    // asynchronous output snapshot (b200sph_snapshot_*): one in flight
    double *snap_buf = nullptr;         // device staging, 8-byte slots
    int64_t snap_cap = 0;               // in doubles
    std::vector<int64_t> snap_off, snap_len;   // per segment: offset (doubles) / elements
    std::vector<int> snap_u32;          // per segment: 1 = 4-byte integers
    cudaStream_t snap_stream = nullptr; // the D2H copies run here, beside the time loop
    cudaEvent_t snap_ready = nullptr, snap_done = nullptr;
    std::atomic<bool> snap_open{false};   // taken by the time loop, released by the output thread
    cudaEvent_t tc_evt[2] = {nullptr, nullptr};
    bool h_dirty = true;        // h changed since the last update_domain reduction
    // the 32-byte-record list kernel (k_pair_list<..., R32>, env B200SPH_PAIR_R32): allowed by the
    // caller (b200sph_set_hm_static), and the per-array h / m extrema it needs, re-reduced when
    // h or m may have changed (uni_dirty)
    bool pair_r32 = true;
    bool hm_static = false;
    bool uni_dirty = true;
    double uni_h[B200SPH_MAX_ARRAYS][2], uni_m[B200SPH_MAX_ARRAYS][2];   // (min, max) over the real particles
    long long *uni_red = nullptr;   // device scratch of k_uni_minmax
    unsigned r32_cls = 0;       // bit a: array a is source class 1 in R (what the state packers write)
    int64_t n_pair_r32 = 0;     // pair passes that ran it (since reset_stats)
    unsigned *red_u32 = nullptr, *red_u32_host = nullptr;
    int64_t n_full_builds = 0, n_light_updates = 0, n_list_builds = 0;

    // scratch
    long long *red = nullptr;     // 16 ordered-int64 slots
    long long *red_host = nullptr;  // pinned
    unsigned long long *counter = nullptr;  // pair counter + misc
    unsigned long long *counter_host = nullptr;
    double *stage_buf = nullptr;  // host<->device staging for f32 props
    int64_t stage_cap = 0;
    uint32_t *flag_a = nullptr, *flag_b = nullptr;  // [pool+1] scan scratch
    int64_t flag_cap = 0;

    // persistent halo: pool-relative indices of the real particles sent to neighbour `slot`
    uint32_t *halo_idx[B200SPH_MAX_ARRAYS][2] = {{nullptr}};
    int64_t halo_cnt[B200SPH_MAX_ARRAYS][2] = {{0}}, halo_cap[B200SPH_MAX_ARRAYS][2] = {{0}};

    EosTab eos_pending;
    bool eos_any = false;
    // ---- peer protocol (b200sph_peer_*) + interior / boundary split of the list consumer --
    int peer_rank = -1, peer_world = 0;
    struct PeerBox *peer_box = nullptr;          // this rank's mailbox
    struct PeerBox *peer_boxes[B200SPH_MAX_RANKS] = {nullptr};   // every rank's (own: the local one)
    bool peer_connected = false;
    unsigned long long peer_epoch = 0, peer_dt_epoch = 0;
    unsigned *peer_done = nullptr;               // "blocks finished" counters of k_peer_push, one per direction
    double *peer_dec_dev = nullptr;
    struct PeerDecision *peer_dec_host = nullptr, *peer_dec_hostdev = nullptr;   // pinned + its device alias
    cudaStream_t comm_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // profiling of the overlapped evaluation (b200sph_set_profiling != 0): per pair pass an event
    // triple {fork of the communication stream, scatter done, boundary launch done}
    struct HaloEvents { cudaEvent_t fork, chain, end, sent, reduced; };
    std::vector<HaloEvents> halo_pending;
    cudaEvent_t halo_ev_fork = nullptr, halo_ev_chain = nullptr, halo_ev_sent = nullptr, halo_ev_reduced = nullptr;
    bool comm_pending = false;                   // work on comm_stream that the main stream has not waited for
    // The scalar agreement runs on its own stream: a rank's ghosts only need its two neighbours,
    // the decision needs every rank, and the boundary launch must not wait for the slowest one.
    cudaStream_t red_stream = nullptr;
    // generic-equation fallback: user properties (fp64, pool-wide) and run-time compiled modules
    double *user_f64[B200SPH_MAX_USER] = {nullptr};
    std::vector<void *> gen_modules;             // CUmodule (or, emulated, a dlopen handle)
    // Group(start_idx, stop_idx): one-shot destination ranges of the next pair pass
    int64_t dst_lo[B200SPH_MAX_ARRAYS] = {0}, dst_hi[B200SPH_MAX_ARRAYS] = {0};
    bool dst_ranged = false;
    int push_first = 0;                          // B200SPH_PUSH_FIRST (measured: profiles/r02k_chain.md)
    cudaEvent_t ev_pushed = nullptr, ev_red = nullptr;
    // peer_publish / peer_send / peer_recv only RECORD: the launches are merged into one
    // k_peer_push (at peer_reduce) and one k_peer_pull (at peer_end)
    struct PeerPending *pend = nullptr;
    uint8_t *sflag = nullptr;                    // [sorted] 1 = ghost
    uint8_t *stype = nullptr;                    // [sorted] particle type byte (array id | ghost bit), written by k_pack_pos
    unsigned long long list_mask[B200SPH_MAX_ARRAYS] = {0};   // the equation mask the current lists were filtered with
    uint32_t *chunk_boundary = nullptr, *chunk_interior = nullptr;
    int64_t n_chunk_boundary = 0, n_chunk_interior = 0, chunk_cap = 0;
    bool chunks_valid = false;
    int64_t n_overlapped = 0;
    // ---- fused stage kernel (k_stage_pack) bookkeeping ---------------------------------
    bool fuse = true;            // env B200SPH_FUSE=0: the unfused kernels only
    EosTab eos_last;             // the equation-of-state calls of the last evaluation ...
    bool eos_last_valid = false;
    bool spec_records = false;   // ... were applied to the packed records speculatively
    unsigned spec_confirmed = 0; // arrays whose b200sph_eos call has matched the speculation
    bool drift_measured = false; // red_u32 holds the drift of the CURRENT packed positions
    bool red_armed = false;      // red[9,11,12] hold their neutral values
    bool dt_reduced = false;     // ... hold the factors of the last evaluation (fused stage2)
    bool dt_adaptive_seen = false;  // a dt proposal followed the last stage2: reduce in the next one
    int64_t n_fused = 0;

    // stats
    b200sph_stats stats;
    int profiling = 0;          // 0 off, 1 every phase, 2 the pair kernels only
    bool async_copies = false;  // push/pull return without waiting (pinned host buffers)
    std::vector<PendingEvent> pending;
    std::vector<cudaEvent_t> ev_pool;
};

struct PhaseTimer;
static int set_err(b200sph_ctx *c, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (c) {
        std::lock_guard<std::mutex> lk(c->err_mu);
        c->err = buf;
    }
    return -1;
}

#define CU(call)                                                                    \
    do {                                                                            \
        cudaError_t _e = (call);                                                    \
        if (_e != cudaSuccess)                                                      \
            return set_err(ctx, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), \
                           __FILE__, __LINE__);                                     \
    } while (0)

#define LAUNCH_CHECK()                                                              \
    do {                                                                            \
        ctx->stats.kernel_launches++;                                               \
        cudaError_t _e = cudaGetLastError();                                        \
        if (_e != cudaSuccess)                                                      \
            return set_err(ctx, "kernel launch failed: %s (%s:%d)",                 \
                           cudaGetErrorString(_e), __FILE__, __LINE__);             \
    } while (0)

// ordered-int64 image of a double so atomicMin/Max(long long) order like doubles
__host__ __device__ static inline long long d2o(double d)
{
    long long b;
#ifdef __CUDA_ARCH__
    b = __double_as_longlong(d);
#else
    memcpy(&b, &d, 8);
#endif
    return b ^ ((b >> 63) & 0x7fffffffffffffffLL);
}
__host__ __device__ static inline double o2d(long long o)
{
    long long b = o ^ ((o >> 63) & 0x7fffffffffffffffLL);
#ifdef __CUDA_ARCH__
    return __longlong_as_double(b);
#else
    double d;
    memcpy(&d, &b, 8);
    return d;
#endif
}

__device__ __forceinline__ float frcp(float x)
{
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float frsqrt(float x)
{
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// A float4 table in shared memory read through an opaque 32-bit shared address: the
// compiler otherwise re-derives the CTA's shared window base (three uniform instructions)
// at every use inside the pair loops.  (The host emulation of the tests supplies its own.)
#ifndef B200SPH_HOST_EMULATION
typedef uint32_t smem_tab_t;
__device__ __forceinline__ smem_tab_t smem_tab(const float4 *table)
{
    uint32_t a = (uint32_t)__cvta_generic_to_shared(table);
    asm volatile("" : "+r"(a));
    return a;
}
__device__ __forceinline__ float4 lds_T(const smem_tab_t t, const uint32_t index)
{
    float4 v;
    asm("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(t + (index << 4)));
    return v;
}
// nanosecond clock shared by every SM (bounds the spin waits of the peer protocol)
__device__ __forceinline__ unsigned long long peer_now_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#endif

#include "generic_args.h"
#include "pool_kernels.cuh"
#include "scan.cuh"
#include "nnps_kernels.cuh"
#include "sph_kernels.cuh"
#include "pair_kernel.cuh"
#include "pair_list.cuh"
#include "tvf_kernels.cuh"
#include "solid_kernels.cuh"
#include "halo_kernels.cuh"

// --------------------------------------------------------------------------
// host side
// --------------------------------------------------------------------------
static int is_solid_prop(int p) { return p >= B200SPH_S00 && p < B200SPH_SOLID_PROPS_END; }
static int is_user_prop(int p) { return p >= B200SPH_USER0 && p < B200SPH_USER0 + B200SPH_MAX_USER; }
static int is_f64_prop(int p)
{
    return (p >= 0 && p < N_F64) || (p >= B200SPH_UHAT && p <= B200SPH_PF0) || (p >= B200SPH_S00 && p <= B200SPH_S220) ||
           is_user_prop(p);
}
static int is_f32_prop(int p)
{
    return (p >= N_F64 && p < N_F64 + N_F32) || (p >= B200SPH_VOL && p <= B200SPH_AP) || (p >= B200SPH_V00 && p <= B200SPH_AS22);
}
static double *f64_ptr(b200sph_ctx *ctx, int p)
{
    if (is_user_prop(p)) return ctx->user_f64[p - B200SPH_USER0];
    return p < N_F64 ? ctx->f64[p] : (p < B200SPH_S00 ? ctx->f64x[p - B200SPH_UHAT] : ctx->f64s[p - B200SPH_S00]);
}
static float *f32_ptr(b200sph_ctx *ctx, int p)
{
    return p < N_F64 + N_F32 ? ctx->f32[p - N_F64] : (p < B200SPH_V00 ? ctx->f32x[p - B200SPH_VOL] : ctx->f32s[p - B200SPH_V00]);
}
static int u32_index(int p) { return (p >= B200SPH_GID && p <= B200SPH_PID) ? p - B200SPH_GID : -1; }

// (re)build the pool so that every array owns [off, off+cap); moves existing data.
static int pool_layout(b200sph_ctx *ctx, const int64_t *new_cap)
{
    int64_t new_off[B200SPH_MAX_ARRAYS], total = 0;
    for (int a = 0; a < ctx->narr; a++) {
        new_off[a] = total;
        total += (new_cap[a] + 31) / 32 * 32;
    }
    const int64_t alloc = std::max<int64_t>(total, 32);
    // allocate new buffers and move array by array
    const int NB = N_F64 + N_F32 + N_U32;
    for (int k = 0; k < NB + N_F64X + N_F32X; k++) {
        const size_t esz = (k < N_F64 || (k >= NB && k < NB + N_F64X)) ? 8 : 4;
        void *old = k < N_F64 ? (void *)ctx->f64[k]
                  : k < N_F64 + N_F32 ? (void *)ctx->f32[k - N_F64]
                  : k < NB ? (void *)ctx->u32[k - N_F64 - N_F32]
                  : k < NB + N_F64X ? (void *)ctx->f64x[k - NB]
                                    : (void *)ctx->f32x[k - NB - N_F64X];
        void *nw = nullptr;
        CU(cudaMalloc(&nw, esz * (size_t)alloc));
        CU(cudaMemsetAsync(nw, 0, esz * (size_t)alloc, ctx->stream));
        if (old) {
            for (int a = 0; a < ctx->narr; a++) {
                if (ctx->arr[a].n > 0 && ctx->arr[a].cap > 0)
                    CU(cudaMemcpyAsync((char *)nw + esz * (size_t)new_off[a],
                                       (char *)old + esz * (size_t)ctx->arr[a].off,
                                       esz * (size_t)ctx->arr[a].n, cudaMemcpyDeviceToDevice,
                                       ctx->stream));
            }
            CU(cudaStreamSynchronize(ctx->stream));
            CU(cudaFree(old));
        }
        if (k < N_F64) ctx->f64[k] = (double *)nw;
        else if (k < N_F64 + N_F32) ctx->f32[k - N_F64] = (float *)nw;
        else if (k < NB) ctx->u32[k - N_F64 - N_F32] = (uint32_t *)nw;
        else if (k < NB + N_F64X) ctx->f64x[k - NB] = (double *)nw;
        else ctx->f32x[k - NB - N_F64X] = (float *)nw;
    }
    if (ctx->solid_alloc) {   // the elastic-dynamics arrays move with the pool
        for (int k = 0; k < 12 + 21; k++) {
            const size_t esz = k < 12 ? 8 : 4;
            void *old = k < 12 ? (void *)ctx->f64s[k] : (void *)ctx->f32s[k - 12];
            void *nw = nullptr;
            CU(cudaMalloc(&nw, esz * (size_t)alloc));
            CU(cudaMemsetAsync(nw, 0, esz * (size_t)alloc, ctx->stream));
            if (old) {
                for (int a = 0; a < ctx->narr; a++)
                    if (ctx->arr[a].n > 0 && ctx->arr[a].cap > 0)
                        CU(cudaMemcpyAsync((char *)nw + esz * (size_t)new_off[a], (char *)old + esz * (size_t)ctx->arr[a].off,
                                           esz * (size_t)ctx->arr[a].n, cudaMemcpyDeviceToDevice, ctx->stream));
                CU(cudaStreamSynchronize(ctx->stream));
                CU(cudaFree(old));
            }
            if (k < 12) ctx->f64s[k] = (double *)nw;
            else ctx->f32s[k - 12] = (float *)nw;
        }
        for (float4 **r : {&ctx->T01, &ctx->T2R, &ctx->R2}) {
            if (*r) CU(cudaFree(*r));
            CU(cudaMalloc((void **)r, 16 * (size_t)alloc));
        }
    }
    for (int k = 0; k < B200SPH_MAX_USER; k++) {   // user properties move with the pool too
        if (!ctx->user_f64[k]) continue;
        double *old = ctx->user_f64[k], *nw = nullptr;
        CU(cudaMalloc((void **)&nw, 8 * (size_t)alloc));
        CU(cudaMemsetAsync(nw, 0, 8 * (size_t)alloc, ctx->stream));
        for (int a = 0; a < ctx->narr; a++)
            if (ctx->arr[a].n > 0 && ctx->arr[a].cap > 0)
                CU(cudaMemcpyAsync(nw + new_off[a], old + ctx->arr[a].off, 8 * (size_t)ctx->arr[a].n, cudaMemcpyDeviceToDevice, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        CU(cudaFree(old));
        ctx->user_f64[k] = nw;
    }
    if (ctx->ptype) CU(cudaFree(ctx->ptype));
    CU(cudaMalloc((void **)&ctx->ptype, (size_t)alloc));
    for (int a = 0; a < ctx->narr; a++) {
        ctx->arr[a].off = new_off[a];
        ctx->arr[a].cap = new_cap[a];
    }
    ctx->pool_cap = alloc;
    ctx->pool_end = total;
    ctx->ptype_dirty = true;
    ctx->grid_valid = false, ctx->packed_valid = false;
    // per-particle work buffers
    if (ctx->key_of) cudaFree(ctx->key_of);
    if (ctx->off_in) cudaFree(ctx->off_in);
    if (ctx->perm_tmp) cudaFree(ctx->perm_tmp);
    if (ctx->perm) cudaFree(ctx->perm);
    if (ctx->skey) cudaFree(ctx->skey);
    if (ctx->rank) cudaFree(ctx->rank);
    if (ctx->A) cudaFree(ctx->A);
    if (ctx->B) cudaFree(ctx->B);
    if (ctx->C) cudaFree(ctx->C);
    if (ctx->AB) cudaFree(ctx->AB);
    if (ctx->R) cudaFree(ctx->R);
    if (ctx->A0) cudaFree(ctx->A0);
    if (ctx->Dv) cudaFree(ctx->Dv);
    if (ctx->PT) cudaFree(ctx->PT);
    if (ctx->cnt) cudaFree(ctx->cnt);
    if (ctx->flag_a) cudaFree(ctx->flag_a);
    if (ctx->flag_b) cudaFree(ctx->flag_b);
    CU(cudaMalloc((void **)&ctx->key_of, 4 * (size_t)alloc));
    CU(cudaMalloc((void **)&ctx->off_in, 4 * (size_t)alloc));
    CU(cudaMalloc((void **)&ctx->perm_tmp, 4 * (size_t)alloc));
    CU(cudaMalloc((void **)&ctx->perm, 4 * (size_t)alloc));
    CU(cudaMalloc((void **)&ctx->skey, 4 * (size_t)alloc));
    CU(cudaMalloc((void **)&ctx->rank, 4 * (size_t)alloc));
    CU(cudaMalloc((void **)&ctx->A, 16 * (size_t)alloc));
    CU(cudaMalloc((void **)&ctx->B, 16 * (size_t)alloc));
    CU(cudaMalloc((void **)&ctx->C, 16 * (size_t)alloc));
    CU(cudaMalloc((void **)&ctx->AB, 32 * (size_t)alloc));
    CU(cudaMalloc((void **)&ctx->R, 32 * (size_t)alloc));
    CU(cudaMalloc((void **)&ctx->A0, 16 * (size_t)alloc));
    CU(cudaMalloc((void **)&ctx->Dv, 16 * (size_t)alloc));
    CU(cudaMalloc((void **)&ctx->PT, 8 * (size_t)alloc));
    CU(cudaMalloc((void **)&ctx->cnt, 4 * (size_t)alloc));
    if (ctx->stype) cudaFree(ctx->stype);
    CU(cudaMalloc((void **)&ctx->stype, (size_t)alloc));
    ctx->lists_valid = false;
    ctx->topo_dirty = true;
    ctx->h_dirty = ctx->uni_dirty = true;
    CU(cudaMalloc((void **)&ctx->flag_a, 4 * (size_t)(alloc + 1)));
    CU(cudaMalloc((void **)&ctx->flag_b, 4 * (size_t)(alloc + 1)));
    ctx->flag_cap = alloc + 1;
    ctx->sort_cap = alloc;
    return 0;
}

static int ensure_capacity(b200sph_ctx *ctx, int arr, int64_t need)
{
    if (need <= ctx->arr[arr].cap && ctx->pool_cap > 0) return 0;
    int64_t caps[B200SPH_MAX_ARRAYS];
    for (int a = 0; a < ctx->narr; a++) caps[a] = ctx->arr[a].cap;
    if (need > caps[arr]) caps[arr] = need + need / 4 + 1024;
    return pool_layout(ctx, caps);
}

static int refresh_ptype(b200sph_ctx *ctx)
{
    if (!ctx->ptype_dirty) return 0;
    PoolLayout L;
    L.narr = ctx->narr;
    for (int a = 0; a < ctx->narr; a++) {
        L.off[a] = ctx->arr[a].off;
        L.n[a] = ctx->arr[a].n;
        L.n_real[a] = ctx->arr[a].n_real;
    }
    if (ctx->pool_end > 0) {
        k_fill_ptype<<<(unsigned)cdiv(ctx->pool_end, 256), 256, 0, ctx->stream>>>(ctx->ptype,
                                                                                  ctx->pool_end, L);
        LAUNCH_CHECK();
    }
    ctx->ptype_dirty = false;
    return 0;
}

// the main stream waits for what the peer protocol left running on the communication stream
static int sync_comm(b200sph_ctx *ctx)
{
    if (!ctx->comm_pending) return 0;
    ctx->comm_pending = false;
    CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_join, 0));
    CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_red, 0));
    return 0;
}

static int ensure_pool(b200sph_ctx *ctx, bool join = true)
{
    if (join) {
        int rc0 = sync_comm(ctx);
        if (rc0) return rc0;
    }
    if (ctx->pool_cap == 0) {
        int64_t caps[B200SPH_MAX_ARRAYS];
        for (int a = 0; a < ctx->narr; a++) caps[a] = std::max(ctx->arr[a].cap, ctx->arr[a].n);
        int rc = pool_layout(ctx, caps);
        if (rc) return rc;
    }
    return refresh_ptype(ctx);
}

static int device_scan(b200sph_ctx *ctx, const uint32_t *in, uint32_t *out, int64_t n)
{
    const int64_t nb = cdiv(n, SCAN_TILE);
    if (nb > ctx->blk_cap) {
        if (ctx->blk_sums) CU(cudaFree(ctx->blk_sums));
        CU(cudaMalloc((void **)&ctx->blk_sums, 4 * (size_t)(nb + 1024)));
        ctx->blk_cap = nb + 1024;
    }
    k_scan_tiles<<<(unsigned)nb, SCAN_THREADS, 0, ctx->stream>>>(in, out, n, ctx->blk_sums);
    LAUNCH_CHECK();
    if (nb > 1) {
        k_scan_sums<<<1, SCAN_THREADS, 0, ctx->stream>>>(ctx->blk_sums, nb);
        LAUNCH_CHECK();
        k_scan_add<<<(unsigned)nb, SCAN_THREADS, 0, ctx->stream>>>(out, n, ctx->blk_sums);
        LAUNCH_CHECK();
    }
    return 0;
}

// Per-phase device timing without host syncs: event pairs are recorded on the
// context's stream and only resolved (cudaEventElapsedTime) in get_stats.
struct PhaseTimer {
    b200sph_ctx *ctx;
    int slot;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    PhaseTimer(b200sph_ctx *c, int s);
    ~PhaseTimer();
};


PhaseTimer::PhaseTimer(b200sph_ctx *c, int s) : ctx(c), slot(s)
{
    if (!ctx->profiling || (ctx->profiling == 2 && slot != 1)) return;
    for (cudaEvent_t *e : {&e0, &e1}) {
        if (!ctx->ev_pool.empty()) {
            *e = ctx->ev_pool.back();
            ctx->ev_pool.pop_back();
        } else {
            cudaEventCreate(e);
        }
    }
    cudaEventRecord(e0, ctx->stream);
}
PhaseTimer::~PhaseTimer()
{
    if (!e0) return;
    cudaEventRecord(e1, ctx->stream);
    ctx->pending.push_back({e0, e1, slot});
}

template <int K> static void launch_pair_dim(int dim, unsigned nb, cudaStream_t st, const PairArgs &pa)
{
    if (dim == 1) k_pair<K, 1><<<nb, PAIR_WARPS * 32, 0, st>>>(pa);
    else if (dim == 2) k_pair<K, 2><<<nb, PAIR_WARPS * 32, 0, st>>>(pa);
    else k_pair<K, 3><<<nb, PAIR_WARPS * 32, 0, st>>>(pa);
}

static double kernel_fac(int kernel, int dim)
{
    const double pi = 3.14159265358979323846;
    switch (kernel) {
    case 0: return dim == 3 ? 1.0 / pi : (dim == 2 ? 10.0 / (7.0 * pi) : 2.0 / 3.0);  // kernels.py:57-65
    case 1: return dim == 2 ? 7.0 / (4.0 * pi) : 21.0 / (16.0 * pi);                  // kernels.py:291-299
    case 2: return dim == 1 ? 1.0 / 120.0 : (dim == 2 ? 7.0 / (478.0 * pi) : 1.0 / (120.0 * pi));  // kernels.py:1071-1079
    default: return std::pow(1.0 / std::sqrt(pi), dim);                                // kernels.py:852-858
    }
}
static double kernel_deltap(int kernel)
{
    switch (kernel) {
    case 0: return 2. / 3;
    case 1: return 0.5;
    case 2: return 0.759298480738450;
    default: return 0.70710678118654746;
    }
}

extern "C" {

static int eos_flush(b200sph_ctx *ctx, cudaStream_t on_comm_stream = nullptr);
static void free_peer_pending(b200sph_ctx *ctx);
static void generic_unload_all(b200sph_ctx *ctx);

int b200sph_abi_version(void) { return B200SPH_ABI_VERSION; }

int b200sph_create(int device, b200sph_ctx **out)
{
    if (!out) return -1;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device >= ndev) {
        fprintf(stderr, "b200sph_create: no usable CUDA device %d (found %d) -- this library has "
                        "no CPU fallback\n", device, ndev);
        return -2;
    }
    b200sph_ctx *ctx = new b200sph_ctx();
    ctx->device = device;
    memset(&ctx->grid, 0, sizeof(ctx->grid));
    memset(&ctx->eos_pending, 0, sizeof(ctx->eos_pending));
    memset(&ctx->eos_last, 0, sizeof(ctx->eos_last));
    memset(&ctx->stats, 0, sizeof(ctx->stats));
    *out = ctx;
    CU(cudaSetDevice(device));
    CU(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    ctx->own_stream = true;
    if (const char *e = getenv("B200SPH_PAIR_KERNEL")) {
        if (!strcmp(e, "warp")) ctx->force_kernel = 1;
        else if (strcmp(e, "list") && e[0]) {
            fprintf(stderr, "b200sph: B200SPH_PAIR_KERNEL must be list or warp\n");
            delete ctx;
            *out = nullptr;
            return -3;
        }
    }
    if (const char *e = getenv("B200SPH_PAIR_MINB")) ctx->pair_minb = ctx->pair_minb_r32 = atoi(e);
    if (const char *e = getenv("B200SPH_FUSE")) ctx->fuse = atoi(e) != 0;
    if (const char *e = getenv("B200SPH_PAIR_SPEC")) ctx->pair_spec = atoi(e) != 0;
    if (const char *e = getenv("B200SPH_PAIR_R32")) ctx->pair_r32 = atoi(e) != 0;
    if (const char *e = getenv("B200SPH_ZORDER")) ctx->zorder = atoi(e) != 0;
    if (const char *e = getenv("B200SPH_PROACTIVE")) ctx->proactive = atoi(e) != 0;
    if (const char *e = getenv("B200SPH_PUSH_FIRST")) ctx->push_first = atoi(e) != 0;
    if (const char *e = getenv("B200SPH_SKIN")) ctx->skin = ctx->skin_max = std::max(0.0, atof(e));
    if (const char *e = getenv("B200SPH_SKIN_ADAPT")) ctx->skin_adapt = atoi(e) != 0;
    ctx->skin_min = std::min(ctx->skin_min, ctx->skin_max);
    CU(cudaMalloc((void **)&ctx->red_u32, 4 * sizeof(unsigned)));
    CU(cudaMallocHost((void **)&ctx->red_u32_host, 4 * sizeof(unsigned)));
    CU(cudaMallocHost((void **)&ctx->drift_host, 4 * sizeof(unsigned)));
    CU(cudaEventCreateWithFlags(&ctx->drift_evt, cudaEventDisableTiming));
    CU(cudaMalloc((void **)&ctx->red, 16 * sizeof(long long)));
    CU(cudaMallocHost((void **)&ctx->red_host, 16 * sizeof(long long)));
    CU(cudaMalloc((void **)&ctx->counter, 8 * sizeof(unsigned long long)));
    CU(cudaMallocHost((void **)&ctx->counter_host, 8 * sizeof(unsigned long long)));
    return 0;
}

int b200sph_destroy(b200sph_ctx *ctx)
{
    if (!ctx) return 0;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (int k = 0; k < N_F64; k++) cudaFree(ctx->f64[k]);
    for (int k = 0; k < N_F32; k++) cudaFree(ctx->f32[k]);
    for (int k = 0; k < N_U32; k++) cudaFree(ctx->u32[k]);
    for (int k = 0; k < N_F64X; k++) cudaFree(ctx->f64x[k]);
    for (int k = 0; k < B200SPH_MAX_USER; k++) cudaFree(ctx->user_f64[k]);
    generic_unload_all(ctx);
    for (int k = 0; k < N_F32X; k++) cudaFree(ctx->f32x[k]);
    cudaFree(ctx->Dv); cudaFree(ctx->PT);
    for (auto &sg : ctx->mirror_segs) cudaFree(sg.idx);
    for (int k = 0; k < 12; k++) cudaFree(ctx->f64s[k]);
    for (int k = 0; k < 21; k++) cudaFree(ctx->f32s[k]);
    cudaFree(ctx->T01); cudaFree(ctx->T2R); cudaFree(ctx->R2);
    cudaFree(ctx->ptype);
    cudaFree(ctx->key_of); cudaFree(ctx->off_in); cudaFree(ctx->cell_cnt); cudaFree(ctx->cell_start);
    cudaFree(ctx->blk_sums); cudaFree(ctx->perm_tmp); cudaFree(ctx->perm); cudaFree(ctx->skey);
    cudaFree(ctx->rank); cudaFree(ctx->A); cudaFree(ctx->B); cudaFree(ctx->C); cudaFree(ctx->AB); cudaFree(ctx->R); cudaFree(ctx->uni_red);
    cudaFree(ctx->red); cudaFreeHost(ctx->red_host); cudaFree(ctx->counter);
    cudaFreeHost(ctx->counter_host); cudaFree(ctx->stage_buf); cudaFree(ctx->flag_a);
    cudaFree(ctx->flag_b); cudaFree(ctx->A0); cudaFree(ctx->lst); cudaFree(ctx->cnt);
    cudaFree(ctx->red_u32); cudaFreeHost(ctx->red_u32_host);
    cudaFreeHost(ctx->drift_host);
    if (ctx->tc_owned) cudaFree(ctx->tc);
    if (ctx->tc_host) cudaFreeHost(ctx->tc_host);
    for (int i = 0; i < 2; i++)
        if (ctx->tc_evt[i]) cudaEventDestroy(ctx->tc_evt[i]);
    if (ctx->drift_evt) cudaEventDestroy(ctx->drift_evt);
    for (auto &pe : ctx->pending) { cudaEventDestroy(pe.e0); cudaEventDestroy(pe.e1); }
    for (auto e : ctx->ev_pool) cudaEventDestroy(e);
    if (ctx->snap_stream) { cudaStreamSynchronize(ctx->snap_stream); cudaStreamDestroy(ctx->snap_stream); }
    if (ctx->snap_ready) cudaEventDestroy(ctx->snap_ready);
    if (ctx->snap_done) cudaEventDestroy(ctx->snap_done);
    cudaFree(ctx->snap_buf);
    for (int r = 0; r < ctx->peer_world; r++)
        if (r != ctx->peer_rank && ctx->peer_boxes[r]) cudaIpcCloseMemHandle(ctx->peer_boxes[r]);
    cudaFree(ctx->peer_box); cudaFree(ctx->peer_done); cudaFree(ctx->peer_dec_dev);
    if (ctx->peer_dec_host) cudaFreeHost(ctx->peer_dec_host);
    if (ctx->comm_stream) { cudaStreamSynchronize(ctx->comm_stream); cudaStreamDestroy(ctx->comm_stream); }
    if (ctx->red_stream) { cudaStreamSynchronize(ctx->red_stream); cudaStreamDestroy(ctx->red_stream); }
    if (ctx->ev_pushed) cudaEventDestroy(ctx->ev_pushed);
    if (ctx->ev_red) cudaEventDestroy(ctx->ev_red);
    free_peer_pending(ctx);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    cudaFree(ctx->sflag); cudaFree(ctx->stype); cudaFree(ctx->chunk_boundary); cudaFree(ctx->chunk_interior);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return 0;
}

const char *b200sph_last_error(b200sph_ctx *ctx)
{
    if (!ctx) return "null context";
    std::lock_guard<std::mutex> lk(ctx->err_mu);
    ctx->err_out = ctx->err;     // a stable copy: another thread may be writing the next message
    return ctx->err_out.c_str();
}

int b200sph_set_stream(b200sph_ctx *ctx, void *s)
{
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    if (ctx->own_stream) CU(cudaStreamDestroy(ctx->stream));
    if (s) {
        ctx->stream = (cudaStream_t)s;
        ctx->own_stream = false;
    } else {
        CU(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        ctx->own_stream = true;
    }
    return 0;
}

int b200sph_synchronize(b200sph_ctx *ctx)
{
    CU(cudaSetDevice(ctx->device));
    if (int rcj = sync_comm(ctx)) return rcj;
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int b200sph_add_array(b200sph_ctx *ctx, const char *name, int64_t n, int64_t n_real, int64_t capacity)
{
    if (ctx->narr >= B200SPH_MAX_ARRAYS) return set_err(ctx, "too many particle arrays (max %d)", B200SPH_MAX_ARRAYS);
    if (n < 0 || n_real < 0 || n_real > n) return set_err(ctx, "add_array: bad sizes n=%lld n_real=%lld", (long long)n, (long long)n_real);
    CU(cudaSetDevice(ctx->device));
    const int a = ctx->narr;
    ctx->arr[a].name = name ? name : "";
    ctx->arr[a].n = n;
    ctx->arr[a].n_real = n_real;
    ctx->arr[a].cap = std::max<int64_t>(capacity, n);
    ctx->arr[a].off = 0;
    ctx->narr++;
    if (ctx->pool_cap > 0) {  // pool already built: re-layout, preserving data of older arrays
        int64_t caps[B200SPH_MAX_ARRAYS];
        const int64_t n_new = ctx->arr[a].n;
        ctx->arr[a].n = 0;  // nothing to move for the new array
        for (int k = 0; k < ctx->narr; k++) caps[k] = ctx->arr[k].cap;
        int rc = pool_layout(ctx, caps);
        ctx->arr[a].n = n_new;
        if (rc) return rc;
    }
    ctx->ptype_dirty = true;
    ctx->grid_valid = false, ctx->packed_valid = false;
    ctx->topo_dirty = true;
    ctx->h_dirty = ctx->uni_dirty = true;
    return a;
}

int b200sph_resize_array(b200sph_ctx *ctx, int arr, int64_t n, int64_t n_real)
{
    if (arr < 0 || arr >= ctx->narr) return set_err(ctx, "resize_array: bad array %d", arr);
    if (n < 0 || n_real < 0 || n_real > n) return set_err(ctx, "resize_array: bad sizes");
    CU(cudaSetDevice(ctx->device));
    { int rc0 = eos_flush(ctx); if (rc0) return rc0; }
    if (ctx->pool_cap == 0) {
        ctx->arr[arr].cap = std::max(ctx->arr[arr].cap, n);
    } else {
        int rc = ensure_capacity(ctx, arr, n);
        if (rc) return rc;
    }
    ctx->arr[arr].n = n;
    ctx->arr[arr].n_real = n_real;
    ctx->ptype_dirty = true;
    ctx->grid_valid = false, ctx->packed_valid = false;
    ctx->topo_dirty = true;
    ctx->h_dirty = ctx->uni_dirty = true;
    return 0;
}

int b200sph_get_array_size(b200sph_ctx *ctx, int arr, int64_t *n, int64_t *n_real)
{
    if (arr < 0 || arr >= ctx->narr) return set_err(ctx, "get_array_size: bad array %d", arr);
    if (n) *n = ctx->arr[arr].n;
    if (n_real) *n_real = ctx->arr[arr].n_real;
    return 0;
}

static int check_range(b200sph_ctx *ctx, int arr, int64_t start, int64_t count)
{
    if (arr < 0 || arr >= ctx->narr) return set_err(ctx, "bad array index %d", arr);
    if (start < 0 || count < 0 || start + count > ctx->arr[arr].n)
        return set_err(ctx, "range [%lld, %lld) outside array '%s' of %lld particles", (long long)start,
                       (long long)(start + count), ctx->arr[arr].name.c_str(), (long long)ctx->arr[arr].n);
    return 0;
}

static int ensure_stage(b200sph_ctx *ctx, int64_t count)
{
    if (count > ctx->stage_cap) {
        if (ctx->stage_buf) CU(cudaFree(ctx->stage_buf));
        CU(cudaMalloc((void **)&ctx->stage_buf, 8 * (size_t)(count + 1024)));
        ctx->stage_cap = count + 1024;
    }
    return 0;
}

// user properties of the generic-equation fallback: allocated (zeroed) when first named
static int ensure_user(b200sph_ctx *ctx, int prop)
{
    if (!is_user_prop(prop)) return 0;
    double *&p = ctx->user_f64[prop - B200SPH_USER0];
    if (p) return 0;
    const size_t alloc = (size_t)std::max<int64_t>(ctx->pool_cap, 32);
    CU(cudaMalloc((void **)&p, 8 * alloc));
    CU(cudaMemsetAsync(p, 0, 8 * alloc, ctx->stream));
    return 0;
}

// elastic-dynamics property arrays: allocated (zeroed) the first time anything names them
static int ensure_solid(b200sph_ctx *ctx)
{
    if (ctx->solid_alloc) return 0;
    const size_t alloc = (size_t)std::max<int64_t>(ctx->pool_cap, 32);
    for (int k = 0; k < 12; k++) {
        CU(cudaMalloc((void **)&ctx->f64s[k], 8 * alloc));
        CU(cudaMemsetAsync(ctx->f64s[k], 0, 8 * alloc, ctx->stream));
    }
    for (int k = 0; k < 21; k++) {
        CU(cudaMalloc((void **)&ctx->f32s[k], 4 * alloc));
        CU(cudaMemsetAsync(ctx->f32s[k], 0, 4 * alloc, ctx->stream));
    }
    for (float4 **r : {&ctx->T01, &ctx->T2R, &ctx->R2}) CU(cudaMalloc((void **)r, 16 * alloc));
    ctx->solid_alloc = true;
    return 0;
}

int b200sph_push_f64(b200sph_ctx *ctx, int arr, int prop, const double *host, int64_t start, int64_t count)
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if ((rc = check_range(ctx, arr, start, count))) return rc;
    // naming an elastic-dynamics property allocates that pool even for an empty array: every
    // rank of a slab decomposition must agree on the message layout (b200sph_halo_layout)
    if (is_solid_prop(prop) && (rc = ensure_solid(ctx))) return rc;
    if ((rc = ensure_user(ctx, prop))) return rc;
    if (count == 0) return 0;
    const int64_t o = ctx->arr[arr].off + start;
    if (is_f64_prop(prop)) {
        CU(cudaMemcpyAsync(f64_ptr(ctx, prop) + o, host, 8 * (size_t)count, cudaMemcpyHostToDevice, ctx->stream));
    } else if (is_f32_prop(prop)) {
        if ((rc = ensure_stage(ctx, count))) return rc;
        CU(cudaMemcpyAsync(ctx->stage_buf, host, 8 * (size_t)count, cudaMemcpyHostToDevice, ctx->stream));
        k_f64_to_f32<<<(unsigned)cdiv(count, 256), 256, 0, ctx->stream>>>(ctx->stage_buf, f32_ptr(ctx, prop) + o, count);
        LAUNCH_CHECK();
    } else {
        return set_err(ctx, "push_f64: property id %d is not a floating point property", prop);
    }
    // the host buffer is borrowed only for this call
    if (!ctx->async_copies) CU(cudaStreamSynchronize(ctx->stream));
    // new positions / smoothing lengths for the SAME particles: the next nnps_update
    // measures the drift against the current neighbour build and reuses it if it can
    if (prop == B200SPH_H) { ctx->domain_valid = false; ctx->h_dirty = ctx->uni_dirty = true; }
    if (prop == B200SPH_M) ctx->uni_dirty = true;
    if (prop <= B200SPH_Z || prop == B200SPH_H) ctx->grid_valid = false, ctx->packed_valid = false;
    ctx->state_packed = false;
    return 0;
}

static int require_confirmed(b200sph_ctx *ctx, const char *who);
int b200sph_pull_f64(b200sph_ctx *ctx, int arr, int prop, double *host, int64_t start, int64_t count)
{
    if (int rcc = require_confirmed(ctx, "pull_f64")) return rcc;
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if ((rc = eos_flush(ctx))) return rc;
    if ((rc = check_range(ctx, arr, start, count))) return rc;
    if (count == 0) return 0;
    const int64_t o = ctx->arr[arr].off + start;
    if (is_solid_prop(prop) && (rc = ensure_solid(ctx))) return rc;
    if ((rc = ensure_user(ctx, prop))) return rc;
    if (is_f64_prop(prop)) {
        CU(cudaMemcpyAsync(host, f64_ptr(ctx, prop) + o, 8 * (size_t)count, cudaMemcpyDeviceToHost, ctx->stream));
    } else if (is_f32_prop(prop)) {
        if ((rc = ensure_stage(ctx, count))) return rc;
        k_f32_to_f64<<<(unsigned)cdiv(count, 256), 256, 0, ctx->stream>>>(f32_ptr(ctx, prop) + o, ctx->stage_buf, count);
        LAUNCH_CHECK();
        CU(cudaMemcpyAsync(host, ctx->stage_buf, 8 * (size_t)count, cudaMemcpyDeviceToHost, ctx->stream));
    } else {
        return set_err(ctx, "pull_f64: property id %d is not a floating point property", prop);
    }
    if (!ctx->async_copies) CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int b200sph_push_u32(b200sph_ctx *ctx, int arr, int prop, const uint32_t *host, int64_t start, int64_t count)
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if ((rc = check_range(ctx, arr, start, count))) return rc;
    const int k = u32_index(prop);
    if (k < 0) return set_err(ctx, "push_u32: property id %d is not an integer property", prop);
    if (count == 0) return 0;
    CU(cudaMemcpyAsync(ctx->u32[k] + ctx->arr[arr].off + start, host, 4 * (size_t)count, cudaMemcpyHostToDevice, ctx->stream));
    if (!ctx->async_copies) CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int b200sph_pull_u32(b200sph_ctx *ctx, int arr, int prop, uint32_t *host, int64_t start, int64_t count)
{
    if (int rcc = require_confirmed(ctx, "pull_u32")) return rcc;
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if ((rc = check_range(ctx, arr, start, count))) return rc;
    const int k = u32_index(prop);
    if (k < 0) return set_err(ctx, "pull_u32: property id %d is not an integer property", prop);
    if (count == 0) return 0;
    CU(cudaMemcpyAsync(host, ctx->u32[k] + ctx->arr[arr].off + start, 4 * (size_t)count, cudaMemcpyDeviceToHost, ctx->stream));
    if (!ctx->async_copies) CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int b200sph_device_ptr(b200sph_ctx *ctx, int arr, int prop, void **out)
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if (arr < 0 || arr >= ctx->narr) return set_err(ctx, "device_ptr: bad array %d", arr);
    const int64_t o = ctx->arr[arr].off;
    if (is_solid_prop(prop) && (rc = ensure_solid(ctx))) return rc;
    if ((rc = ensure_user(ctx, prop))) return rc;
    if (is_f64_prop(prop)) *out = f64_ptr(ctx, prop) + o;
    else if (is_f32_prop(prop)) *out = f32_ptr(ctx, prop) + o;
    else if (u32_index(prop) >= 0) *out = ctx->u32[u32_index(prop)] + o;
    else return set_err(ctx, "device_ptr: bad property %d", prop);
    return 0;
}

// ---- asynchronous output snapshot ---------------------------------------------------
// take: device-to-device copies (fp32 properties widened) into a private buffer, in stream
// order -- the time loop goes on at once; fetch: device-to-host on a second stream, from
// any host thread; release: lets the next take overwrite the buffer.
int b200sph_snapshot_take(b200sph_ctx *ctx, int nseg, const int *arr, const int *prop, const int64_t *count)
{
    if (int rcc = require_confirmed(ctx, "snapshot_take")) return rcc;
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if ((rc = eos_flush(ctx))) return rc;
    if (ctx->snap_open) return set_err(ctx, "snapshot_take: the previous snapshot was not released");
    if (nseg < 1) return set_err(ctx, "snapshot_take: no segments");
    if (!ctx->snap_stream) {
        CU(cudaStreamCreateWithFlags(&ctx->snap_stream, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&ctx->snap_ready, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&ctx->snap_done, cudaEventDisableTiming));
    } else {
        // the copies of the previous snapshot must have left the buffer
        CU(cudaStreamWaitEvent(ctx->stream, ctx->snap_done, 0));
    }
    int64_t total = 0;
    for (int i = 0; i < nseg; i++) {
        if (arr[i] == -1) {  // the time-control block {dt, t, ...}
            if (!ctx->tc) return set_err(ctx, "snapshot_take: no time-control block");
            if (count[i] < 1 || count[i] > 8) return set_err(ctx, "snapshot_take: the time-control block has 8 doubles");
        } else if ((rc = check_range(ctx, arr[i], 0, count[i]))) return rc;
        total += std::max<int64_t>(count[i], 1);
    }
    if (total > ctx->snap_cap) {
        if (ctx->snap_buf) CU(cudaFree(ctx->snap_buf));
        CU(cudaMalloc((void **)&ctx->snap_buf, 8 * (size_t)(total + total / 8 + 1024)));
        ctx->snap_cap = total + total / 8 + 1024;
    }
    ctx->snap_off.assign(nseg, 0), ctx->snap_len.assign(nseg, 0), ctx->snap_u32.assign(nseg, 0);
    int64_t at = 0;
    for (int i = 0; i < nseg; i++) {
        const int64_t n = count[i];
        ctx->snap_off[i] = at, ctx->snap_len[i] = n;
        double *dst = ctx->snap_buf + at;
        at += std::max<int64_t>(n, 1);
        if (n == 0) continue;
        if (arr[i] == -1) {
            CU(cudaMemcpyAsync(dst, ctx->tc, 8 * (size_t)n, cudaMemcpyDeviceToDevice, ctx->stream));
            continue;
        }
        const int64_t o = ctx->arr[arr[i]].off;
        const int pr = prop[i];
        if (is_solid_prop(pr) && (rc = ensure_solid(ctx))) return rc;
        if (is_f64_prop(pr)) {
            CU(cudaMemcpyAsync(dst, f64_ptr(ctx, pr) + o, 8 * (size_t)n, cudaMemcpyDeviceToDevice, ctx->stream));
        } else if (is_f32_prop(pr)) {
            k_f32_to_f64<<<(unsigned)cdiv(n, 256), 256, 0, ctx->stream>>>(f32_ptr(ctx, pr) + o, dst, n);
            LAUNCH_CHECK();
        } else if (u32_index(pr) >= 0) {
            ctx->snap_u32[i] = 1;
            CU(cudaMemcpyAsync(dst, ctx->u32[u32_index(pr)] + o, 4 * (size_t)n, cudaMemcpyDeviceToDevice, ctx->stream));
        } else {
            return set_err(ctx, "snapshot_take: bad property %d", pr);
        }
    }
    CU(cudaEventRecord(ctx->snap_ready, ctx->stream));
    ctx->snap_open = true;
    return 0;
}

int b200sph_snapshot_fetch(b200sph_ctx *ctx, int seg, void *host, int64_t count)
{
    CU(cudaSetDevice(ctx->device));
    if (!ctx->snap_open) return set_err(ctx, "snapshot_fetch: no snapshot");
    if (seg < 0 || seg >= (int)ctx->snap_len.size() || count != ctx->snap_len[seg])
        return set_err(ctx, "snapshot_fetch: segment %d does not hold %lld elements", seg, (long long)count);
    if (count == 0) return 0;
    CU(cudaStreamWaitEvent(ctx->snap_stream, ctx->snap_ready, 0));
    CU(cudaMemcpyAsync(host, ctx->snap_buf + ctx->snap_off[seg], (ctx->snap_u32[seg] ? 4 : 8) * (size_t)count,
                       cudaMemcpyDeviceToHost, ctx->snap_stream));
    CU(cudaStreamSynchronize(ctx->snap_stream));
    return 0;
}

int b200sph_snapshot_release(b200sph_ctx *ctx)
{
    CU(cudaSetDevice(ctx->device));
    if (!ctx->snap_open) return 0;
    CU(cudaEventRecord(ctx->snap_done, ctx->snap_stream));
    ctx->snap_open = false;
    return 0;
}

int b200sph_set_kernel(b200sph_ctx *ctx, int kernel, int dim)
{
    if (kernel < 0 || kernel > 3) return set_err(ctx, "set_kernel: unknown kernel id %d", kernel);
    if (dim < 1 || dim > 3) return set_err(ctx, "set_kernel: dim must be 1, 2 or 3");
    if (kernel == B200SPH_KERNEL_WENDLAND_QUINTIC && dim == 1)
        return set_err(ctx, "WendlandQuintic: Dim 1 not supported");  // kernels.py:289-290
    ctx->kernel = kernel;
    ctx->dim = dim;
    ctx->radius_scale = (kernel == B200SPH_KERNEL_QUINTIC_SPLINE || kernel == B200SPH_KERNEL_GAUSSIAN) ? 3.0 : 2.0;
    ctx->domain_valid = false;
    ctx->grid_valid = false, ctx->packed_valid = false;
    ctx->topo_dirty = true;
    ctx->h_dirty = ctx->uni_dirty = true;
    return 0;
}

static int run_minmax(b200sph_ctx *ctx, int do_xyz, int do_h)
{
    k_red_init<<<1, 32, 0, ctx->stream>>>(ctx->red);
    LAUNCH_CHECK();
    ctx->red_armed = true;   // (slots 9, 11, 12 are not touched by k_reduce_minmax)
    ctx->dt_reduced = false;
    if (ctx->pool_end > 0) {
        const unsigned nb = (unsigned)std::min<int64_t>(cdiv(ctx->pool_end, 256), 148 * 8);
        k_reduce_minmax<<<nb, 256, 0, ctx->stream>>>(ctx->f64[B200SPH_X], ctx->f64[B200SPH_Y], ctx->f64[B200SPH_Z],
                                                     ctx->f64[B200SPH_H], ctx->ptype, ctx->pool_end, do_xyz, do_h, ctx->red);
        LAUNCH_CHECK();
    }
    CU(cudaMemcpyAsync(ctx->red_host, ctx->red, 16 * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int b200sph_set_domain(b200sph_ctx *ctx, const double lo[3], const double hi[3], const int periodic[3])
{
    if ((periodic[0] || periodic[1] || periodic[2]) && (ctx->mirror[0] || ctx->mirror[1] || ctx->mirror[2]))
        return set_err(ctx, "set_domain: mirror planes in a periodic domain are not supported");
    for (int d = 0; d < 3; d++) {
        if (periodic[d] && !(hi[d] > lo[d])) return set_err(ctx, "Invalid domain limits!");  // nnps_base.pyx:352-355
        ctx->periodic[d] = periodic[d] != 0;
        ctx->dom_lo[d] = lo[d];
        ctx->dom_hi[d] = hi[d];
    }
    ctx->grid_valid = false, ctx->packed_valid = false;
    ctx->topo_dirty = true;
    return 0;
}

static inline bool mirror_any(const b200sph_ctx *ctx) { return ctx->mirror[0] || ctx->mirror[1] || ctx->mirror[2]; }
static int mirror_create(b200sph_ctx *ctx);
static int mirror_refresh(b200sph_ctx *ctx);

int b200sph_set_mirror(b200sph_ctx *ctx, const int mirror[3], double n_layers)
{
    if (!(n_layers >= 1.0)) return set_err(ctx, "set_mirror: n_layers must be >= 1 (the images must cover one kernel support)");
    for (int d = 0; d < 3; d++) {
        if (mirror[d] && !(ctx->dom_hi[d] > ctx->dom_lo[d])) return set_err(ctx, "Invalid domain limits!");
    }
    // the reference mirrors the periodic ghosts it has just created as well (nnps_base.pyx:471-480);
    // here periodic images are never materialised, so the combination is refused
    if ((mirror[0] || mirror[1] || mirror[2]) && (ctx->periodic[0] || ctx->periodic[1] || ctx->periodic[2]))
        return set_err(ctx, "set_mirror: mirror planes in a periodic domain are not supported");
    for (int d = 0; d < 3; d++) ctx->mirror[d] = mirror[d] != 0;
    ctx->mirror_layers = n_layers;
    ctx->mirror_built = false;
    ctx->grid_valid = false, ctx->packed_valid = false;
    ctx->topo_dirty = true;
    return 0;
}

int b200sph_update_domain(b200sph_ctx *ctx)
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if (ctx->periodic[0] || ctx->periodic[1] || ctx->periodic[2]) {
        // _box_wrap_periodic, nnps_base.pyx:699-743 (part of DomainManager.update)
        if ((rc = eos_flush(ctx))) return rc;
        GridDev D;
        for (int d = 0; d < 3; d++) {
            D.xmin[d] = ctx->dom_lo[d];
            D.cell[d] = ctx->dom_hi[d] - ctx->dom_lo[d];
            D.nc[d] = 1;
            D.periodic[d] = ctx->periodic[d];
        }
        D.zorder = 0;
        if (ctx->pool_end > 0) {
            k_box_wrap<<<(unsigned)cdiv(ctx->pool_end, 256), 256, 0, ctx->stream>>>(ctx->f64[B200SPH_X], ctx->f64[B200SPH_Y], ctx->f64[B200SPH_Z],
                                                                                   ctx->ptype, ctx->pool_end, D);
            LAUNCH_CHECK();
        }
        ctx->grid_valid = false, ctx->packed_valid = false;
        ctx->state_packed = false;
    }
    if (ctx->domain_valid && !ctx->h_dirty) return 0;  // h untouched since the last reduction
    PhaseTimer pt(ctx, 2);
    if ((rc = run_minmax(ctx, 0, 1))) return rc;
    // nnps_base.pyx:942-978
    double hmin = o2d(ctx->red_host[6]), hmax = o2d(ctx->red_host[7]);
    int64_t ntot = 0;
    for (int a = 0; a < ctx->narr; a++) ntot += ctx->arr[a].n;
    if (ntot == 0) { hmax = -1.0; hmin = 1.7976931348623157e308; }
    double cell = ctx->radius_scale * hmax;
    ctx->hmin_scaled = ctx->radius_scale * hmin;
    if (cell < 1e-6) cell = 1.0;
    if (cell != ctx->cell_size) ctx->grid_valid = false, ctx->packed_valid = false;
    ctx->cell_size = cell;
    ctx->domain_valid = true;
    ctx->h_dirty = false;
    return 0;
}

// 2 |dx|max + k dh <= S, with a 2 % safety margin for the fp32 measurement
static bool drift_within_skin(b200sph_ctx *ctx, const unsigned *raw)
{
    float d2, dh;
    memcpy(&d2, &raw[0], 4);
    memcpy(&dh, &raw[1], 4);
    const double need = 2.0 * std::sqrt((double)d2) + ctx->radius_scale * (double)dh;
    return need <= 0.98 * ctx->S_abs;
}

// Skin controller, part 2 (part 1 adapts the skin geometrically from the lifetime of the build
// that has just ended, see nnps_update).  A build is RETIRED -- rebuilt although it is valid --
//  * when it has lived 3 L* evaluations with more than the minimum skin (a quiet flow must
//    converge to the minimum skin), or
//  * early, after SKIN_PROBE evaluations, when the drift measured so far says the skin is far too
//    generous: with d = drift per evaluation, a skin s lives L(s) = 0.98 s cell / d evaluations,
//    and L(s) = L*(s) = kappa / s gives s* = sqrt(kappa d / (0.98 cell)).  s* < 0.7 s: rebuild
//    now with s* (a rebuild costs ~3 evaluations' worth of the list entries it removes per
//    evaluation; the first build of a run is always made blind, with the maximum skin).
#define SKIN_PROBE 6
static bool retire_build(b200sph_ctx *ctx)
{
    if (!ctx->skin_adapt || !(ctx->skin > ctx->skin_min)) return false;
    if (ctx->evals_since_build >= 3.0 * SKIN_KAPPA / ctx->skin) return true;
    if (ctx->evals_since_build == SKIN_PROBE && ctx->drift_hist[1] >= 0.0 && ctx->cell_size > 0.0) {
        const double d = ctx->drift_hist[1] * ctx->S_abs / (double)SKIN_PROBE;
        const double s_opt = std::min(ctx->skin_max, std::max(ctx->skin_min, std::sqrt(SKIN_KAPPA * d / (0.98 * ctx->cell_size))));
        if (s_opt < 0.7 * ctx->skin) {
            ctx->skin_next = s_opt;
            return true;
        }
    }
    return false;
}

// light path of nnps_update: same sorted order, same cell frames, fresh positions;
// returns 1 if the persistent lists are still valid, 0 if a full rebuild is needed
static int nnps_light_update(b200sph_ctx *ctx)
{
    if (ctx->n_sorted <= 0) return 1;
    if (ctx->drift_ok) {
        // the drift was just measured by b200sph_nnps_drift (multi-GPU: the decision to
        // keep the build is collective); only refresh the packed positions, no host sync
        ctx->drift_ok = false;
        ctx->drift_measured = false;
        if (ctx->packed_valid) return 1;   // nnps_drift_device packed them, halo_overwrite_all kept the ghosts current
        k_pack_pos_light<<<(unsigned)cdiv(ctx->n_sorted, 256), 256, 0, ctx->stream>>>(
            ctx->f64[B200SPH_X], ctx->f64[B200SPH_Y], ctx->f64[B200SPH_Z], ctx->f64[B200SPH_H], ctx->perm, ctx->skey,
            ctx->n_sorted, ctx->G, ctx->A0, ctx->A, ctx->AB, ctx->R, ctx->red_u32);
        LAUNCH_CHECK();
        return 1;
    }
    if (!(ctx->packed_valid && ctx->drift_measured)) {   // (the fused stage kernel packs and measures)
        CU(cudaMemsetAsync(ctx->red_u32, 0, 4 * sizeof(unsigned), ctx->stream));
        k_pack_pos_light<<<(unsigned)cdiv(ctx->n_sorted, 256), 256, 0, ctx->stream>>>(
            ctx->f64[B200SPH_X], ctx->f64[B200SPH_Y], ctx->f64[B200SPH_Z], ctx->f64[B200SPH_H], ctx->perm, ctx->skey,
            ctx->n_sorted, ctx->G, ctx->A0, ctx->A, ctx->AB, ctx->R, ctx->red_u32);
        LAUNCH_CHECK();
    }
    ctx->drift_measured = false;
    ctx->packed_valid = true;
    if (ctx->defer_check) {
        // optimistic: carry on as if the lists were valid; b200sph_nnps_confirm reads the
        // measurement after the evaluation has been enqueued (no idle GPU while we wait)
        CU(cudaMemcpyAsync(ctx->drift_host, ctx->red_u32, 2 * sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaEventRecord(ctx->drift_evt, ctx->stream));
        ctx->check_pending = true;
        return 1;
    }
    CU(cudaMemcpyAsync(ctx->red_u32_host, ctx->red_u32, 4 * sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return drift_within_skin(ctx, ctx->red_u32_host) ? 1 : 0;
}

static int confirm_pending(b200sph_ctx *ctx, int *redo)
{
    *redo = 0;
    if (!ctx->check_pending) return 0;
    CU(cudaSetDevice(ctx->device));
    CU(cudaEventSynchronize(ctx->drift_evt));
    ctx->check_pending = false;
    {
        float d2, dh;
        memcpy(&d2, &ctx->drift_host[0], 4);
        memcpy(&dh, &ctx->drift_host[1], 4);
        ctx->drift_hist[0] = ctx->drift_hist[1];
        ctx->drift_hist[1] = ctx->S_abs > 0.0 ? (2.0 * std::sqrt((double)d2) + ctx->radius_scale * (double)dh) / ctx->S_abs : 2.0;
    }
    if (!drift_within_skin(ctx, ctx->drift_host)) {
        // the evaluation that followed used stale lists: force the full rebuild
        ctx->topo_dirty = true;
        ctx->grid_valid = false, ctx->packed_valid = false;
        ctx->n_light_updates--;
        ctx->n_deferred_failed++;
        *redo = 1;
    }
    return 0;
}
// entry points that consume the results of an evaluation must not run on an
// unconfirmed deferred update
static int require_confirmed(b200sph_ctx *ctx, const char *who)
{
    if (!ctx->check_pending) return 0;
    int redo = 0, rc = confirm_pending(ctx, &redo);
    if (rc) return rc;
    if (redo)
        return set_err(ctx, "%s: the deferred drift check of the last nnps_update failed and was never confirmed "
                            "(call b200sph_nnps_confirm after the evaluation and repeat it when asked to)", who);
    return 0;
}

int b200sph_nnps_confirm(b200sph_ctx *ctx, int *redo) { return confirm_pending(ctx, redo); }

int b200sph_nnps_update_deferred(b200sph_ctx *ctx)
{
    ctx->defer_check = true;
    const int rc = b200sph_nnps_update(ctx);
    ctx->defer_check = false;
    return rc;
}

int b200sph_nnps_update(b200sph_ctx *ctx)
{
    CU(cudaSetDevice(ctx->device));
    // with the peer protocol's refresh in flight the only thing this call may do without
    // waiting for it is to accept the build the ranks have (speculatively) agreed to keep
    int rc = ensure_pool(ctx, !(ctx->comm_pending && ctx->drift_ok && ctx->packed_valid && ctx->lists_valid &&
                                !ctx->topo_dirty && !ctx->eos_any && ctx->domain_valid && !ctx->check_pending));
    if (rc) return rc;
    if (ctx->check_pending) {   // update after update without an evaluation in between
        int redo = 0;
        if ((rc = confirm_pending(ctx, &redo))) return rc;
    }
    if ((rc = eos_flush(ctx))) return rc;
    if (!ctx->domain_valid && (rc = b200sph_update_domain(ctx))) return rc;
    PhaseTimer pt(ctx, 0);

    int64_t ntot0 = 0;
    for (int a = 0; a < ctx->narr; a++) ntot0 += ctx->arr[a].n;
    const bool use_lists = ctx->force_kernel == 0 && ntot0 < (1LL << LIST_JBITS);
    // deferred check + a build whose drift, extrapolated by its last increment, would exceed
    // the skin at THIS evaluation: rebuild now rather than after an evaluation on stale lists
    bool expiring = false;
    if (ctx->proactive && ctx->defer_check && !ctx->drift_ok && ctx->drift_hist[1] >= 0.0) {
        const double r1 = ctx->drift_hist[1], r0 = ctx->drift_hist[0];
        const double step = r0 >= 0.0 ? std::max(r1 - r0, 0.0) : r1;
        expiring = r1 + step > 0.98;
        if (expiring && use_lists && ctx->lists_valid && !ctx->topo_dirty) ctx->n_proactive++;
    }
    if (use_lists && ctx->lists_valid && !ctx->topo_dirty && !expiring &&
        !(!ctx->drift_ok && retire_build(ctx))) {
        // mirror images: the same ghosts, current values (the set is re-selected with the lists)
        if (mirror_any(ctx) && ctx->mirror_built && (rc = mirror_refresh(ctx))) return rc;
        rc = nnps_light_update(ctx);
        if (rc < 0) return rc;
        if (rc == 1) {
            ctx->n_light_updates++;
            ctx->evals_since_build++;
            ctx->grid_valid = true;   // (state_packed is left alone: whatever changed the state cleared it)
            return 0;
        }
    }
    // skin controller (see SKIN_KAPPA): a build that outlived 1.5 L* was built with too
    // generous a skin, one that lasted less than L* / 1.5 with too small a one; builds that
    // reach 3 L* are retired so that a quiet flow converges to the minimum skin
    if (use_lists && ctx->skin_adapt && ctx->lists_valid && ctx->evals_since_build > 0) {
        const double lstar = SKIN_KAPPA / ctx->skin;
        if (ctx->skin_next > 0.0) ctx->skin = ctx->skin_next;     // measured (retire_build)
        else if (ctx->evals_since_build >= 1.5 * lstar) ctx->skin = std::max(ctx->skin_min, ctx->skin * 0.75);
        else if (ctx->evals_since_build < lstar / 1.5) ctx->skin = std::min(ctx->skin_max, ctx->skin * 1.33);
    }
    ctx->skin_next = -1.0;
    ctx->evals_since_build = 0;
    ctx->lists_valid = false;
    ctx->drift_ok = false;
    ctx->drift_hist[0] = ctx->drift_hist[1] = -1.0;
    ctx->n_full_builds++;
    if (mirror_any(ctx)) {
        // _create_ghosts_mirror (nnps_base.pyx:506-689) -- here once per list build, not per update
        if ((rc = mirror_create(ctx))) return rc;
        if (!ctx->domain_valid && (rc = b200sph_update_domain(ctx))) return rc;
    }

    int64_t ntot = 0;
    for (int a = 0; a < ctx->narr; a++) ntot += ctx->arr[a].n;
    if (ntot >= (1LL << 32) - 1) return set_err(ctx, "more than 2^32-2 particles: indices are 32-bit (as in the reference)");

    // _compute_bounds nnps_base.pyx:1520-1575
    if ((rc = run_minmax(ctx, 1, 0))) return rc;
    double mn[3], mx[3], l[3];
    for (int d = 0; d < 3; d++) {
        mn[d] = ntot ? o2d(ctx->red_host[2 * d]) : 1e100;
        mx[d] = ntot ? o2d(ctx->red_host[2 * d + 1]) : -1e100;
        l[d] = mx[d] - mn[d];
    }
    for (int d = 0; d < 3; d++) {
        mn[d] -= l[d] * 0.01;
        mx[d] += l[d] * 0.01;
    }
    const double domain_size = std::max(std::max(l[0], l[1]), l[2]);
    if (ctx->last_domain_size > 1e-16 && domain_size > 2.0 * ctx->last_domain_size)
        fprintf(stderr, "b200sph WARNING: Domain size has increased by a large amount. "
                        "Particles are probably diverging, please check your code!\n");
    ctx->last_domain_size = domain_size;
    if (std::fabs(mx[0] - mn[0]) < 1e-12 && std::fabs(mx[1] - mn[1]) < 1e-12 && std::fabs(mx[2] - mn[2]) < 1e-12)
        for (int d = 0; d < 3; d++) {
            mn[d] -= 0.5;
            mx[d] += 0.5;
        }
    // the reference's grid: _get_number_of_cells / _count_occupied_cells
    // linked_list_nnps.pyx:293-343 (reported by get_grid; the 2^28 guard is honoured)
    int nc_ref[3];
    {
        const double cs1 = 1. / ctx->cell_size;
        for (int d = 0; d < 3; d++) {
            const double v = std::ceil(cs1 * (mx[d] - mn[d]));
            if (!(v < 2147483647.0)) return set_err(ctx, "ERROR: LinkedListNNPS requires too many cells along axis %d", d);
            nc_ref[d] = (int)v;
            if (nc_ref[d] < 0) return set_err(ctx, "LinkedListNNPS: Number of cells is negative");
            if (nc_ref[d] == 0) nc_ref[d] = 1;
        }
        const double ncells_d = (double)nc_ref[0] * (double)nc_ref[1] * (double)nc_ref[2];
        if (ncells_d > (double)(1LL << 28))
            return set_err(ctx, "ERROR: LinkedListNNPS requires too many cells (%.0f).", ncells_d);
    }
    b200sph_grid_info &gi = ctx->grid;
    gi.cell_size = ctx->cell_size;
    gi.hmin = ctx->hmin_scaled;
    for (int d = 0; d < 3; d++) {
        gi.xmin[d] = mn[d];
        gi.xmax[d] = mx[d];
        gi.ncells[d] = nc_ref[d];
    }
    gi.n_cells = (int64_t)nc_ref[0] * nc_ref[1] * nc_ref[2];
    gi.n_particles = ntot;

    // the internal grid: cells widened by the skin when the persistent lists are used
    ctx->S_abs = use_lists ? ctx->skin * ctx->cell_size : 0.0;
    ctx->cell_int = ctx->cell_size + ctx->S_abs;
    int nc[3];
    double cellv[3];
    for (int d = 0; d < 3; d++) {
        if (ctx->periodic[d]) {
            // a periodic axis is tiled EXACTLY by cells not smaller than the cut-off, so
            // that the image shift of a wrapped neighbour cell is a whole number of cells
            const double L = ctx->dom_hi[d] - ctx->dom_lo[d];
            if (!(L >= ctx->cell_int))
                return set_err(ctx, "periodic axis %d: the domain (%g) is smaller than the interaction range + skin (%g)", d, L, ctx->cell_int);
            mn[d] = ctx->dom_lo[d];
            mx[d] = ctx->dom_hi[d];
            nc[d] = std::max(1, (int)std::floor(L / ctx->cell_int));
            cellv[d] = L / nc[d];
        } else {
            nc[d] = (int)std::ceil((mx[d] - mn[d]) / ctx->cell_int);
            if (nc[d] <= 0) nc[d] = 1;
            cellv[d] = ctx->cell_int;
        }
    }
    int64_t ncells = (int64_t)nc[0] * nc[1] * nc[2];
    if (ncells > (1LL << 28)) return set_err(ctx, "ERROR: LinkedListNNPS requires too many cells (%lld).", (long long)ncells);
    // Z-curve over the cell rows: the row table is padded to a power of two per axis (the
    // unused rows are empty cells); a grid whose padding would be excessive stays row-major
    int zorder = 0;
    if (ctx->zorder) {
        int bits = 0;
        while ((1 << bits) < std::max(nc[1], nc[2])) bits++;
        const int64_t padded = ((int64_t)1 << (2 * bits)) * nc[0];
        if (bits <= 15 && padded <= (1LL << 27) && padded <= 8 * ncells + (1 << 20)) {
            zorder = 1;
            ncells = padded;
        }
    }

    if (ncells + 2 > ctx->cell_cap) {
        if (ctx->cell_cnt) CU(cudaFree(ctx->cell_cnt));
        if (ctx->cell_start) CU(cudaFree(ctx->cell_start));
        const int64_t cap = ncells + ncells / 2 + 1024;
        CU(cudaMalloc((void **)&ctx->cell_cnt, 4 * (size_t)cap));
        CU(cudaMalloc((void **)&ctx->cell_start, 4 * (size_t)cap));
        ctx->cell_cap = cap;
    }
    GridDev &G = ctx->G;
    for (int d = 0; d < 3; d++) {
        G.xmin[d] = mn[d];
        G.nc[d] = nc[d];
    }
    for (int d = 0; d < 3; d++) {
        G.cell[d] = cellv[d];
        G.periodic[d] = ctx->periodic[d] ? 1 : 0;
    }
    G.zorder = zorder;

    CU(cudaMemsetAsync(ctx->cell_cnt, 0, 4 * (size_t)(ncells + 1), ctx->stream));
    ctx->n_sorted = ntot;
    if (ctx->pool_end > 0) {
        const unsigned nb = (unsigned)cdiv(ctx->pool_end, 256);
        k_cell_count<<<nb, 256, 0, ctx->stream>>>(ctx->f64[B200SPH_X], ctx->f64[B200SPH_Y], ctx->f64[B200SPH_Z],
                                                  ctx->ptype, ctx->pool_end, G, ctx->key_of, ctx->off_in, ctx->cell_cnt);
        LAUNCH_CHECK();
    }
    if ((rc = device_scan(ctx, ctx->cell_cnt, ctx->cell_start, ncells + 1))) return rc;
    if (ctx->pool_end > 0 && ntot > 0) {
        const unsigned nb = (unsigned)cdiv(ctx->pool_end, 256);
        k_scatter<<<nb, 256, 0, ctx->stream>>>(ctx->key_of, ctx->off_in, ctx->ptype, ctx->pool_end, ctx->cell_start, ctx->perm_tmp);
        LAUNCH_CHECK();
        const unsigned ns = (unsigned)cdiv(ntot, 256);
        k_canon<<<ns, 256, 0, ctx->stream>>>(ctx->perm_tmp, ctx->key_of, ctx->cell_start, ntot, ctx->perm, ctx->skey, ctx->rank);
        LAUNCH_CHECK();
        k_pack_pos<<<ns, 256, 0, ctx->stream>>>(ctx->f64[B200SPH_X], ctx->f64[B200SPH_Y], ctx->f64[B200SPH_Z], ctx->f64[B200SPH_H],
                                                ctx->perm, ctx->skey, ntot, G, ctx->A, ctx->AB, ctx->ptype, ctx->stype, ctx->R);
        LAUNCH_CHECK();
        if (use_lists)
            CU(cudaMemcpyAsync(ctx->A0, ctx->A, 16 * (size_t)ntot, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    ctx->topo_dirty = false;
    ctx->grid_valid = true;
    ctx->state_packed = false;
    return 0;
}

// With ghosts in the build (slab decomposition) the CTAs of the list consumers are split
// into the ones that do not depend on a ghost -- they may run while the halo of the
// evaluation is still in flight -- and the rest (k_chunk_classify).
static int split_chunks(b200sph_ctx *ctx)
{
    ctx->chunks_valid = false;
    int64_t nghost = 0;
    for (int a = 0; a < ctx->narr; a++) nghost += ctx->arr[a].n - ctx->arr[a].n_real;
    const int64_t n = ctx->n_sorted, nchunks = cdiv(n, LIST_NT);
    if (nghost == 0 || n <= 0 || nchunks + 1 > ctx->flag_cap) return 0;
    if (nchunks > ctx->chunk_cap) {
        if (ctx->chunk_boundary) CU(cudaFree(ctx->chunk_boundary));
        if (ctx->chunk_interior) CU(cudaFree(ctx->chunk_interior));
        if (ctx->sflag) CU(cudaFree(ctx->sflag));
        ctx->chunk_cap = nchunks + nchunks / 4 + 64;
        CU(cudaMalloc((void **)&ctx->chunk_boundary, 4 * (size_t)ctx->chunk_cap));
        CU(cudaMalloc((void **)&ctx->chunk_interior, 4 * (size_t)ctx->chunk_cap));
        CU(cudaMalloc((void **)&ctx->sflag, (size_t)ctx->chunk_cap * LIST_NT));
    }
    int rc = refresh_ptype(ctx);
    if (rc) return rc;
    k_sorted_ghost_flag<<<(unsigned)cdiv(n, 256), 256, 0, ctx->stream>>>(ctx->ptype, ctx->perm, n, ctx->sflag);
    LAUNCH_CHECK();
    k_chunk_classify<<<(unsigned)nchunks, LIST_NT, 0, ctx->stream>>>(ctx->cnt, ctx->lst, ctx->capg, ctx->sflag, n, ctx->flag_a);
    LAUNCH_CHECK();
    if ((rc = device_scan(ctx, ctx->flag_a, ctx->flag_b, nchunks + 1))) return rc;
    uint32_t nb = 0;
    CU(cudaMemcpyAsync(&nb, ctx->flag_b + nchunks, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    k_chunk_split<<<(unsigned)cdiv(nchunks, 256), 256, 0, ctx->stream>>>(nchunks, ctx->flag_a, ctx->flag_b, ctx->chunk_boundary, ctx->chunk_interior);
    LAUNCH_CHECK();
    ctx->n_chunk_boundary = nb;
    ctx->n_chunk_interior = nchunks - nb;
    ctx->chunks_valid = true;
    return 0;
}

// (re)build the persistent neighbour lists for the current build.  want[d] (8 bits per source
// type; null: everything) = the (destination, source) type pairs the caller has equations for:
// the lists are filtered with the union of what has been asked for since the particle set last
// changed, so that e.g. a wall particle's wall neighbours -- for which the WCSPH Group has no
// equation -- are never stored, gathered or tested (they were a quarter of the list entries of
// a wall-heavy slab).
static bool lists_cover(const b200sph_ctx *ctx, const unsigned long long *want)
{
    for (int d = 0; d < B200SPH_MAX_ARRAYS; d++) {
        const unsigned long long w = want ? want[d] : ~0ull;
        for (int sx = 0; sx < B200SPH_MAX_ARRAYS; sx++)
            if (((w >> (8 * sx)) & 0xFFull) && !((ctx->list_mask[d] >> (8 * sx)) & 0xFFull)) return false;
    }
    return true;
}
static int build_lists(b200sph_ctx *ctx, const unsigned long long *want)
{
    ctx->chunks_valid = false;
    for (int d = 0; d < B200SPH_MAX_ARRAYS; d++) {
        const unsigned long long w = want ? want[d] : ~0ull;
        for (int sx = 0; sx < B200SPH_MAX_ARRAYS; sx++)
            if ((w >> (8 * sx)) & 0xFFull) ctx->list_mask[d] |= 0xFFull << (8 * sx);
    }
    const int64_t n = ctx->n_sorted;
    ListBuildArgs la;
    la.A = ctx->A; la.cell_start = ctx->cell_start; la.skey = ctx->skey;
    la.n = n;
    la.ncx = ctx->G.nc[0]; la.ncy = ctx->G.nc[1]; la.ncz = ctx->G.nc[2];
    la.cellx = (float)ctx->G.cell[0]; la.celly = (float)ctx->G.cell[1]; la.cellz = (float)ctx->G.cell[2];
    la.zorder = ctx->G.zorder;
    la.px = ctx->G.periodic[0]; la.py = ctx->G.periodic[1]; la.pz = ctx->G.periodic[2];
    const bool per = la.px || la.py || la.pz;
    la.kr = (float)ctx->radius_scale;
    la.S = (float)ctx->S_abs;
    la.cnt = ctx->cnt;
    la.max_count = ctx->red_u32 + 2;
    for (int d = 0; d < B200SPH_MAX_ARRAYS; d++) la.emask[d] = ctx->list_mask[d];
    la.stype = ctx->stype;
    const unsigned nb = (unsigned)cdiv(n, LB_WARPS * 32);
    const int64_t nblk = cdiv(n, 32);
    for (int attempt = 0; attempt < 4; attempt++) {
        const bool count_only = ctx->capg == 0;
        if (!count_only) {
            const int64_t need = nblk * ctx->capg * 32;
            if (need > ctx->lst_cap) {
                if (ctx->lst) CU(cudaFree(ctx->lst));
                ctx->lst = nullptr;
                const int64_t cap = need + need / 8;
                cudaError_t e = cudaMalloc((void **)&ctx->lst, 4 * (size_t)cap);
                if (e != cudaSuccess) return set_err(ctx, "cannot allocate %.1f GB of neighbour lists: %s", 4e-9 * cap, cudaGetErrorString(e));
                ctx->lst_cap = cap;
            }
        }
        la.lst = count_only ? nullptr : ctx->lst;
        la.capg = ctx->capg;
        CU(cudaMemsetAsync(ctx->red_u32 + 2, 0, sizeof(unsigned), ctx->stream));
        if (per) k_list_build<true><<<nb, LB_WARPS * 32, 0, ctx->stream>>>(la);
        else k_list_build<false><<<nb, LB_WARPS * 32, 0, ctx->stream>>>(la);
        LAUNCH_CHECK();
        CU(cudaMemcpyAsync(ctx->red_u32_host + 2, ctx->red_u32 + 2, sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        const int maxc = (int)ctx->red_u32_host[2];
        if (!count_only && maxc <= ctx->capg) {
            ctx->lists_valid = true;
            ctx->n_list_builds++;
            return split_chunks(ctx);
        }
        // (re)size: a little head-room so that later rebuilds usually fit in one pass
        ctx->capg = ((int)(maxc * 1.15) + 8 + 7) / 8 * 8;
    }
    return set_err(ctx, "neighbour list build did not converge");
}

int b200sph_get_grid(b200sph_ctx *ctx, b200sph_grid_info *out)
{
    if (!ctx->grid_valid) return set_err(ctx, "get_grid: the NNPS has not been updated");
    *out = ctx->grid;
    return 0;
}

// run the pending equation-of-state calls stand-alone (something needs rho/p/cs now, or the
// packed records already hold them: the pool side of a speculated EOS) -- one launch
static int eos_flush(b200sph_ctx *ctx, cudaStream_t on_comm_stream)
{
    if (!ctx->eos_any) return 0;
    // ghost rho may be in the middle of a refresh: wait for it -- unless the caller puts
    // this launch on the communication stream itself, behind the scatter
    if (!on_comm_stream)
        if (int rcj = sync_comm(ctx)) return rcj;
    EosTab &E = ctx->eos_pending;
    if (ctx->pool_end > 0) {
        k_eos_tab<<<(unsigned)cdiv(ctx->pool_end, 256), 256, 0, on_comm_stream ? on_comm_stream : ctx->stream>>>(
            ctx->f64[B200SPH_RHO], ctx->f32[B200SPH_P - N_F64], ctx->f32[B200SPH_CS - N_F64], ctx->ptype, ctx->pool_end, E);
        LAUNCH_CHECK();
    }
    memset(E.on, 0, sizeof(E.on));
    ctx->eos_any = false;
    return 0;
}

static int pack_state(b200sph_ctx *ctx)
{
    if (ctx->n_sorted > 0) {
        k_pack_state<<<(unsigned)cdiv(ctx->n_sorted, 256), 256, 0, ctx->stream>>>(
            ctx->f64[B200SPH_U], ctx->f64[B200SPH_V], ctx->f64[B200SPH_W], ctx->f64[B200SPH_M], ctx->f64[B200SPH_RHO],
            ctx->f32[B200SPH_P - N_F64], ctx->f32[B200SPH_CS - N_F64], ctx->ptype, ctx->perm, ctx->n_sorted, ctx->B, ctx->C, ctx->AB,
            ctx->eos_pending, ctx->eos_any ? 1 : 0, ctx->R, ctx->r32_cls);
        LAUNCH_CHECK();
        memset(ctx->eos_pending.on, 0, sizeof(ctx->eos_pending.on));
        ctx->eos_any = false;
    }
    ctx->state_packed = true;
    ctx->spec_records = false;
    return 0;
}

int64_t b200sph_get_neighbors(b200sph_ctx *ctx, int dst_arr, int src_arr, int64_t d_idx, uint32_t *out, int64_t cap)
{
    if (int rcc = require_confirmed(ctx, "get_neighbors")) return rcc;
    CU(cudaSetDevice(ctx->device));
    if (!ctx->grid_valid) return set_err(ctx, "get_neighbors: call nnps_update first");
    if (dst_arr < 0 || dst_arr >= ctx->narr || src_arr < 0 || src_arr >= ctx->narr) return set_err(ctx, "get_neighbors: bad array index");
    if (d_idx < 0 || d_idx >= ctx->arr[dst_arr].n) return set_err(ctx, "get_neighbors: d_idx out of range");
    int rc;
    if (!ctx->state_packed && (rc = pack_state(ctx))) return rc;
    uint32_t s32 = 0;
    CU(cudaMemcpyAsync(&s32, ctx->rank + ctx->arr[dst_arr].off + d_idx, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    const int64_t dcap = std::max<int64_t>(cap, 1);
    uint32_t *dout = nullptr;
    CU(cudaMalloc((void **)&dout, 4 * (size_t)dcap));
    k_neighbors<<<1, 32, 0, ctx->stream>>>(ctx->AB, ctx->C, ctx->cell_start, ctx->skey, ctx->perm, (long long)s32, src_arr,
                                           (long long)ctx->arr[src_arr].off, ctx->G, (float)(ctx->radius_scale * ctx->radius_scale),
                                           dout, cap, ctx->counter + 1);
    ctx->stats.kernel_launches++;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { cudaFree(dout); return set_err(ctx, "k_neighbors launch failed: %s", cudaGetErrorString(e)); }
    CU(cudaMemcpyAsync(ctx->counter_host + 1, ctx->counter + 1, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    const int64_t n = (int64_t)ctx->counter_host[1];
    const int64_t ncopy = std::min(n, cap);
    if (ncopy > 0) {
        CU(cudaMemcpy(out, dout, 4 * (size_t)ncopy, cudaMemcpyDeviceToHost));
        std::sort(out, out + ncopy);
    }
    cudaFree(dout);
    return n;
}

static int arr_range(b200sph_ctx *ctx, int arr, int real_only, int64_t *lo, int64_t *hi)
{
    if (arr < 0 || arr >= ctx->narr) return set_err(ctx, "bad array index %d", arr);
    *lo = ctx->arr[arr].off;
    *hi = ctx->arr[arr].off + (real_only ? ctx->arr[arr].n_real : ctx->arr[arr].n);
    return 0;
}

int b200sph_eos(b200sph_ctx *ctx, int arr, int hg, double rho0, double c0, double gamma, double p0, int real_only)
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx, false);   // only book-keeping here: a halo in flight stays in flight
    if (rc) return rc;
    if (arr < 0 || arr >= ctx->narr) return set_err(ctx, "bad array index %d", arr);
    EosTab &E = ctx->eos_pending;
    // a second call for the same array before the first was applied, or a build that
    // is not valid (no sorted order to pack): run what is pending now
    if ((E.on[arr] || !ctx->grid_valid) && (rc = eos_flush(ctx))) return rc;
    E.on[arr] = 1; E.hg[arr] = hg; E.real_only[arr] = real_only;
    E.rho0[arr] = rho0; E.c0[arr] = c0; E.gamma[arr] = gamma; E.p0[arr] = p0;
    ctx->eos_any = true;
    if (!ctx->grid_valid && (rc = eos_flush(ctx))) return rc;
    // the fused stage kernel may have applied exactly this call to the packed records
    // already (it repeats the last evaluation's calls); pair_pass checks that ALL of them
    // were confirmed before it trusts the records
    const EosTab &L = ctx->eos_last;
    if (ctx->spec_records && ctx->state_packed && ctx->eos_last_valid && L.on[arr] && L.hg[arr] == hg &&
        L.real_only[arr] == real_only && L.rho0[arr] == rho0 && L.c0[arr] == c0 && L.gamma[arr] == gamma && L.p0[arr] == p0) {
        ctx->spec_confirmed |= 1u << arr;
    } else {
        ctx->state_packed = false;
        ctx->spec_records = false;
    }
    return 0;
}

int b200sph_ferrari_h(b200sph_ctx *ctx, int arr, double hdx, int dim, int real_only)
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if ((rc = eos_flush(ctx))) return rc;
    int64_t lo, hi;
    if ((rc = arr_range(ctx, arr, real_only, &lo, &hi))) return rc;
    PhaseTimer pt(ctx, 2);
    if (hi > lo) {
        k_ferrari<<<(unsigned)cdiv(hi - lo, 256), 256, 0, ctx->stream>>>(ctx->f64[B200SPH_H], ctx->f64[B200SPH_M], ctx->f64[B200SPH_RHO], lo, hi, hdx, 1.0 / dim);
        LAUNCH_CHECK();
    }
    ctx->domain_valid = false;  // h changed: the next update_domain must re-reduce it
    ctx->h_dirty = ctx->uni_dirty = true;
    ctx->hm_static = false;     // and keeps changing: no uniform-h kernel from here on
    ctx->grid_valid = false, ctx->packed_valid = false;
    return 0;
}

// ---- generic-equation fallback (pysph_b200/codegen.py; SURVEY.md 8f-4) ---------------------
// Kernels generated from user Equation bodies and compiled by NVRTC are loaded through the
// driver API, which is looked up at first use (the library itself links the runtime only, so
// that it loads -- and fails loudly at the first CUDA call -- on a box without a driver).
#include <dlfcn.h>
#ifndef B200SPH_HOST_EMULATION
struct DriverApi {
    void *lib = nullptr;
    int (*ModuleLoadData)(void **, const void *) = nullptr;
    int (*ModuleGetFunction)(void **, void *, const char *) = nullptr;
    int (*ModuleUnload)(void *) = nullptr;
    int (*LaunchKernel)(void *, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, void *, void **, void **) = nullptr;
    int (*GetErrorString)(int, const char **) = nullptr;
};
static DriverApi g_drv;
static int driver_api(b200sph_ctx *ctx)
{
    if (g_drv.lib) return 0;
    void *lib = dlopen("libcuda.so.1", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) return set_err(ctx, "generic equations: cannot load libcuda.so.1 (%s)", dlerror());
    DriverApi d;
    d.ModuleLoadData = (int (*)(void **, const void *))dlsym(lib, "cuModuleLoadData");
    d.ModuleGetFunction = (int (*)(void **, void *, const char *))dlsym(lib, "cuModuleGetFunction");
    d.ModuleUnload = (int (*)(void *))dlsym(lib, "cuModuleUnload");
    d.LaunchKernel = (int (*)(void *, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, void *, void **, void **))dlsym(lib, "cuLaunchKernel");
    d.GetErrorString = (int (*)(int, const char **))dlsym(lib, "cuGetErrorString");
    if (!d.ModuleLoadData || !d.ModuleGetFunction || !d.ModuleUnload || !d.LaunchKernel)
        return set_err(ctx, "generic equations: libcuda.so.1 lacks the module API");
    d.lib = lib;
    g_drv = d;
    return 0;
}
static const char *drv_err(int e)
{
    const char *m = nullptr;
    if (g_drv.GetErrorString) g_drv.GetErrorString(e, &m);
    return m ? m : "unknown driver error";
}
#endif

static void generic_unload_all(b200sph_ctx *ctx)
{
    for (void *m : ctx->gen_modules) {
        if (!m) continue;
#ifdef B200SPH_HOST_EMULATION
        dlclose(m);
#else
        if (g_drv.ModuleUnload) g_drv.ModuleUnload(m);
#endif
    }
    ctx->gen_modules.clear();
}

int b200sph_user_property(b200sph_ctx *ctx, int prop)
{
    CU(cudaSetDevice(ctx->device));
    if (!is_user_prop(prop)) return set_err(ctx, "user_property: ids %d..%d", B200SPH_USER0, B200SPH_USER0 + B200SPH_MAX_USER - 1);
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    return ensure_user(ctx, prop);
}

int b200sph_generic_load(b200sph_ctx *ctx, const void *image, int64_t size)
{
    CU(cudaSetDevice(ctx->device));
    if (!image || size <= 0) return set_err(ctx, "generic_load: empty image");
    void *mod = nullptr;
#ifdef B200SPH_HOST_EMULATION
    // the emulated library runs kernels that a TEST compiled for the host: the "image" is the
    // path of that shared object
    mod = dlopen((const char *)image, RTLD_NOW | RTLD_LOCAL);
    if (!mod) return set_err(ctx, "generic_load: %s", dlerror());
#else
    int rc = driver_api(ctx);
    if (rc) return rc;
    CU(cudaFree(0));   // the runtime's primary context is current on this thread from here on
    const int e = g_drv.ModuleLoadData(&mod, image);
    if (e) return set_err(ctx, "generic_load: cuModuleLoadData: %s", drv_err(e));
#endif
    ctx->gen_modules.push_back(mod);
    return (int)ctx->gen_modules.size() - 1;
}

// One phase (0 initialize, 1 loop, 2 post_loop) of one destination array of a generated Group
// kernel.  src_mask: the source arrays of its loop bodies; writes: bit 0 a body stores to
// x / y / z / h, bit 1 to any other property the packed records are made from.
int b200sph_generic_launch(b200sph_ctx *ctx, int module, const char *kernel, int dest_arr, int phase, unsigned src_mask,
                           int real_only, double t, double dt, int writes)
{
    if (int rcc = require_confirmed(ctx, "generic_launch")) return rcc;
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if (module < 0 || module >= (int)ctx->gen_modules.size()) return set_err(ctx, "generic_launch: bad module handle %d", module);
    if (dest_arr < 0 || dest_arr >= ctx->narr || phase < 0 || phase > 2) return set_err(ctx, "generic_launch: bad destination / phase");
    if (ctx->peer_box || ctx->comm_pending) return set_err(ctx, "generic equations run on one GPU (no slab decomposition)");
    if (!ctx->grid_valid) return set_err(ctx, "generic_launch: the NNPS is stale (particles were pushed/resized); call nnps_update first");
    if ((rc = eos_flush(ctx))) return rc;
    const bool ranged = ctx->dst_ranged;   // one-shot, as for pair_pass: every launch names its own
    ctx->dst_ranged = false;
    const bool use_lists = ctx->force_kernel == 0 && ctx->n_sorted > 0 && ctx->n_sorted < (1LL << LIST_JBITS);
    if (ctx->n_sorted > 0 && !use_lists) return set_err(ctx, "generic equations need the neighbour-list path");
    if (phase == 1 && use_lists) {
        unsigned long long want[B200SPH_MAX_ARRAYS];
        for (int d = 0; d < B200SPH_MAX_ARRAYS; d++) want[d] = 0;
        for (int sx = 0; sx < ctx->narr; sx++)
            if ((src_mask >> sx) & 1u) want[dest_arr] |= 0xFFull << (8 * sx);
        if (ctx->lists_valid && !lists_cover(ctx, want)) ctx->lists_valid = false;
        if (!ctx->lists_valid) {
            PhaseTimer pt_build(ctx, 0);
            if ((rc = build_lists(ctx, want))) return rc;
        }
    }
    b200sph_generic_args ga;
    memset(&ga, 0, sizeof(ga));
    for (int k = 0; k < N_F64; k++) ga.f64[k] = ctx->f64[k];
    for (int k = 0; k < N_F32; k++) ga.f32[k] = ctx->f32[k];
    for (int k = 0; k < N_U32; k++) ga.u32[k] = ctx->u32[k];
    for (int k = 0; k < B200SPH_MAX_USER; k++) ga.user[k] = ctx->user_f64[k];
    ga.AB = ctx->AB; ga.stype = ctx->stype; ga.perm = ctx->perm;
    ga.cnt = ctx->cnt; ga.lst = ctx->lst; ga.capg = ctx->capg;
    ga.n = ctx->n_sorted;
    ga.cellx = (float)ctx->G.cell[0]; ga.celly = (float)ctx->G.cell[1]; ga.cellz = (float)ctx->G.cell[2];
    ga.k2 = (float)(ctx->radius_scale * ctx->radius_scale);
    ga.dest_type = dest_arr; ga.real_only = real_only; ga.phase = phase; ga.src_mask = src_mask;
    ga.t = t; ga.dt = dt;
    ga.doff = ctx->arr[dest_arr].off;
    ga.dlo = ranged ? ctx->dst_lo[dest_arr] : 0;
    ga.dhi = ranged && ctx->dst_hi[dest_arr] >= 0 ? ctx->dst_hi[dest_arr] : (int64_t)1 << 62;
    if (ctx->n_sorted > 0) {
        PhaseTimer pt(ctx, phase == 1 ? 1 : 2);
        const unsigned nb = (unsigned)cdiv(ctx->n_sorted, 128);
#ifdef B200SPH_HOST_EMULATION
        void (*fn)(b200sph_generic_args) = (void (*)(b200sph_generic_args))dlsym(ctx->gen_modules[module], kernel);
        if (!fn) return set_err(ctx, "generic_launch: no kernel '%s' in the module", kernel);
        emu::launch(nb, 128, emu::SEQ, [&] { fn(ga); });
#else
        void *fn = nullptr;
        int e = g_drv.ModuleGetFunction(&fn, ctx->gen_modules[module], kernel);
        if (e) return set_err(ctx, "generic_launch: no kernel '%s' in the module: %s", kernel, drv_err(e));
        void *params[1] = {&ga};
        e = g_drv.LaunchKernel(fn, nb, 1, 1, 128, 1, 1, 0, (void *)ctx->stream, params, nullptr);
        if (e) return set_err(ctx, "generic_launch: cuLaunchKernel(%s): %s", kernel, drv_err(e));
#endif
        ctx->stats.kernel_launches++;
    }
    // what was derived from the properties the bodies stored to is stale
    if (writes & 1) {
        ctx->grid_valid = false, ctx->packed_valid = false;
        ctx->domain_valid = false, ctx->h_dirty = ctx->uni_dirty = true;
        ctx->hm_static = false;
    }
    if (writes & 2) ctx->state_packed = false, ctx->spec_records = false;
    return 0;
}

int b200sph_set_dest_range(b200sph_ctx *ctx, int arr, int64_t start, int64_t stop)
{
    if (arr < 0 || arr >= ctx->narr) return set_err(ctx, "set_dest_range: bad array index %d", arr);
    if (start < 0 || stop < -1) return set_err(ctx, "set_dest_range: start >= 0 and stop >= 0 (or -1: no limit), got [%lld, %lld)", (long long)start, (long long)stop);
    if (!ctx->dst_ranged)
        for (int d = 0; d < B200SPH_MAX_ARRAYS; d++) ctx->dst_lo[d] = 0, ctx->dst_hi[d] = -1;
    ctx->dst_lo[arr] = start;
    ctx->dst_hi[arr] = stop;
    ctx->dst_ranged = true;
    return 0;
}

int b200sph_set_hm_static(b200sph_ctx *ctx, int on)
{
    ctx->hm_static = on != 0;
    return 0;
}

// Whether the WCSPH Group `prog` may run the R32 list kernel, and with what: the sources split
// into at most two classes of equal equation-mask columns (over the destinations), every class
// that has an equation for some destination has one m and one Tait EOS (gamma = 7, same rho0
// and c0, pending for this evaluation: its cs went into the records), one h for every particle,
// no ghosts.  `lm` is the filter the lists hold entries for; a source the lists can hold is
// classified even if this Group has no equation for it (its class then has none either).
// Returns 1 and fills `pa`, 0 to fall back, < 0 on error.  Only a change of h or m costs a device
// reduction (uni_dirty); the rest is a few loops over the 8 x 8 equation masks per pass.
struct R32Plan {
    unsigned cls;       // bit a: array a is source class 1
    int rep[2];         // PairArgs.r32_*
    float m[2], coef[2];
};
static int r32_plan(b200sph_ctx *ctx, const b200sph_pair_program *prog, const unsigned long long *lm, R32Plan &pa)
{
    bool dest[B200SPH_MAX_ARRAYS];
    for (int d = 0; d < ctx->narr; d++) {
        dest[d] = false;
        for (int sx = 0; sx < ctx->narr; sx++)
            if (prog->eqmask[d][sx]) dest[d] = true;
    }
    if (!ctx->pair_r32 || !ctx->hm_static || !ctx->eos_any) return 0;
    if (ctx->mirror[0] || ctx->mirror[1] || ctx->mirror[2] || ctx->peer_connected) return 0;
    for (int a = 0; a < ctx->narr; a++)
        if (ctx->arr[a].n != ctx->arr[a].n_real) return 0;
    if (ctx->uni_dirty) {
        if (!ctx->uni_red) CU(cudaMalloc((void **)&ctx->uni_red, 4 * B200SPH_MAX_ARRAYS * sizeof(long long)));
        long long init[4 * B200SPH_MAX_ARRAYS];
        for (int k = 0; k < 4 * B200SPH_MAX_ARRAYS; k++) init[k] = d2o(1e300);
        CU(cudaMemcpyAsync(ctx->uni_red, init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
        if (ctx->pool_end > 0) {
            k_uni_minmax<<<(unsigned)cdiv(ctx->pool_end, 256), 256, 0, ctx->stream>>>(
                ctx->f64[B200SPH_H], ctx->f64[B200SPH_M], ctx->ptype, ctx->pool_end, ctx->uni_red);
            LAUNCH_CHECK();
        }
        CU(cudaMemcpyAsync(init, ctx->uni_red, sizeof(init), cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        for (int a = 0; a < B200SPH_MAX_ARRAYS; a++) {
            ctx->uni_h[a][0] = o2d(init[4 * a]); ctx->uni_h[a][1] = -o2d(init[4 * a + 1]);
            ctx->uni_m[a][0] = o2d(init[4 * a + 2]); ctx->uni_m[a][1] = -o2d(init[4 * a + 3]);
        }
        ctx->uni_dirty = false;
    }
    double h = 0.0;
    bool have_h = false;
    for (int a = 0; a < ctx->narr; a++) {
        if (ctx->arr[a].n == 0) continue;
        if (ctx->uni_h[a][0] != ctx->uni_h[a][1] || (have_h && ctx->uni_h[a][0] != h)) return 0;
        h = ctx->uni_h[a][0];
        have_h = true;
    }
    // classes: arrays the lists can hold as sources, by their column of equation bits
    int rep[2] = {-1, -1}, cl[B200SPH_MAX_ARRAYS];
    bool used[2] = {false, false};
    unsigned c1 = 0;
    for (int sx = 0; sx < ctx->narr; sx++) {
        cl[sx] = -1;
        bool listed = false, any = false;
        for (int d = 0; d < ctx->narr; d++) {
            if (!dest[d]) continue;   // not a destination of this Group
            if ((lm[d] >> (8 * sx)) & 0xFFull) listed = true;
            if (prog->eqmask[d][sx]) any = true;
        }
        if (!listed) continue;
        int c = -1;
        for (int k = 0; k < 2 && c < 0; k++) {
            if (rep[k] < 0) { rep[k] = sx; c = k; break; }
            bool same = true;
            for (int d = 0; d < ctx->narr; d++)
                if (dest[d] && prog->eqmask[d][sx] != prog->eqmask[d][rep[k]]) same = false;
            if (same) c = k;
        }
        if (c < 0) return 0;              // a third class
        if (c == 1) c1 |= 1u << sx;
        cl[sx] = c;
        if (!any) continue;               // no equation: m and the EOS do not matter
        const EosTab &E = ctx->eos_pending;
        if (!E.on[sx] || E.gamma[sx] != 7.0) return 0;
        if (ctx->arr[sx].n > 0 && ctx->uni_m[sx][0] != ctx->uni_m[sx][1]) return 0;
        const float m = (float)ctx->uni_m[sx][0];
        const float coef = (float)(E.c0[sx] / (E.rho0[sx] * E.rho0[sx] * E.rho0[sx]));
        if (used[c] && pa.m[c] != m) return 0;
        // the members of a class share their column, so all of them have equations here
        for (int t = 0; t < sx; t++)
            if (cl[t] == c && (E.rho0[t] != E.rho0[sx] || E.c0[t] != E.c0[sx])) return 0;
        pa.m[c] = m;
        pa.coef[c] = coef;
        used[c] = true;
    }
    for (int c = 0; c < 2; c++)
        if (!used[c]) pa.m[c] = pa.coef[c] = 0.f;
    pa.rep[0] = rep[0] < 0 ? 0 : rep[0];
    pa.rep[1] = rep[1] < 0 ? pa.rep[0] : rep[1];
    pa.cls = c1;
    return 1;
}

int b200sph_pair_pass(b200sph_ctx *ctx, const b200sph_pair_program *prog, int64_t *pairs_out)
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx, false);   // a halo in flight is waited for below, as late as possible
    if (rc) return rc;
    if (!ctx->grid_valid) return set_err(ctx, "pair_pass: the NNPS is stale (particles were pushed/resized); call nnps_update first");
    if (ctx->spec_records && ctx->state_packed) {
        // records packed by the fused stage kernel: valid only if this evaluation issued
        // exactly the equation-of-state calls that were applied speculatively
        unsigned want = 0, pending = 0;
        for (int a = 0; a < ctx->narr; a++) {
            if (ctx->eos_last_valid && ctx->eos_last.on[a]) want |= 1u << a;
            if (ctx->eos_any && ctx->eos_pending.on[a]) pending |= 1u << a;
        }
        if (pending != want || ctx->spec_confirmed != want) ctx->state_packed = false;
    }
    ctx->spec_records = false;
    ctx->spec_confirmed = 0;
    ctx->dt_reduced = false;   // this pass writes new dt_cfl / dt_force
    if (ctx->eos_any) {
        ctx->eos_last = ctx->eos_pending;
        ctx->eos_last_valid = true;
    } else {
        ctx->eos_last_valid = false;
    }
    // lists hold 26-bit sorted indices: larger particle counts use the warp kernel
    const bool use_lists = ctx->force_kernel == 0 && ctx->n_sorted > 0 && ctx->n_sorted < (1LL << LIST_JBITS);
    const bool ranged = ctx->dst_ranged;
    ctx->dst_ranged = false;
    if (ranged && !use_lists && ctx->n_sorted > 0)
        return set_err(ctx, "pair_pass: destination ranges (Group start_idx / stop_idx) need the neighbour-list path");
    // the (destination, source) type pairs this Group has equations for; lists that were
    // filtered with a narrower set are rebuilt with the union
    unsigned long long want[B200SPH_MAX_ARRAYS];
    for (int d = 0; d < B200SPH_MAX_ARRAYS; d++) {
        want[d] = 0;
        for (int sx = 0; sx < B200SPH_MAX_ARRAYS; sx++)
            if (d < ctx->narr && sx < ctx->narr && prog->eqmask[d][sx]) want[d] |= 0xFFull << (8 * sx);
    }
    if (use_lists && ctx->lists_valid && !lists_cover(ctx, want)) ctx->lists_valid = false;
    // the WCSPH scheme's Group (continuity + momentum + XSPH, no tensile correction) has a
    // leaner kernel variant (B200SPH_PAIR_SPEC=0: always the generic one) ...
    unsigned prog_bits = 0;
    for (int d = 0; d < ctx->narr; d++)
        for (int sx = 0; sx < ctx->narr; sx++) prog_bits |= prog->eqmask[d][sx];
    const bool wcsph_only = ctx->pair_spec && !(prog_bits & ~(unsigned)PAIR_EQS_WCSPH) && !prog->tensile_correction;
    // ... and that one a 32-byte-record form (r32_plan); a new class split re-packs the state
    // records (the sign of rho in R)
    R32Plan r32p;
    int r32 = 0;
    if (use_lists && !ranged && wcsph_only) {
        unsigned long long lm[B200SPH_MAX_ARRAYS];
        for (int d = 0; d < B200SPH_MAX_ARRAYS; d++) lm[d] = ctx->list_mask[d] | want[d];   // what build_lists keeps
        if ((r32 = r32_plan(ctx, prog, lm, r32p)) < 0) return r32;
        if (r32 && r32p.cls != ctx->r32_cls) {
            ctx->r32_cls = r32p.cls;
            ctx->state_packed = false;
        }
    }
    // the peer protocol's refresh is still in flight and every record a ghost-free CTA
    // reads is in place: those CTAs go first, the main stream waits for the halo only then
    const bool overlap = ctx->comm_pending && use_lists && ctx->lists_valid && ctx->chunks_valid && ctx->state_packed &&
                         ctx->n_chunk_interior > 0 && !pairs_out && !ranged;
    if (!overlap && (rc = sync_comm(ctx))) return rc;
    if (!ctx->state_packed) {
        if ((rc = pack_state(ctx))) return rc;
    } else if (!overlap && (rc = eos_flush(ctx))) {   // the records have them; now the pool's rho / p / cs
        return rc;
    }
    if (!use_lists && (ctx->periodic[0] || ctx->periodic[1] || ctx->periodic[2]))
        return set_err(ctx, "periodic domains need the neighbour-list path (B200SPH_PAIR_KERNEL=list, < 2^26 particles)");
    if (use_lists && !ctx->lists_valid) {
        PhaseTimer pt_build(ctx, 0);  // list builds are part of the neighbour search time
        if ((rc = build_lists(ctx, want))) return rc;
    }
    PhaseTimer pt(ctx, 1);

    PairArgs pa;
    memset(&pa, 0, sizeof(pa));
    pa.A = ctx->A; pa.B = ctx->B; pa.C = ctx->C; pa.AB = ctx->AB;
    pa.cell_start = ctx->cell_start; pa.skey = ctx->skey; pa.perm = ctx->perm;
    pa.arho = ctx->f32[B200SPH_ARHO - N_F64];
    pa.au = ctx->f32[B200SPH_AU - N_F64]; pa.av = ctx->f32[B200SPH_AV - N_F64]; pa.aw = ctx->f32[B200SPH_AW - N_F64];
    pa.ax = ctx->f32[B200SPH_AX - N_F64]; pa.ay = ctx->f32[B200SPH_AY - N_F64]; pa.az = ctx->f32[B200SPH_AZ - N_F64];
    pa.dt_cfl = ctx->f32[B200SPH_DT_CFL - N_F64]; pa.dt_force = ctx->f32[B200SPH_DT_FORCE - N_F64];
    pa.rho = ctx->f64[B200SPH_RHO];
    pa.n = ctx->n_sorted;
    pa.ncx = ctx->G.nc[0]; pa.ncy = ctx->G.nc[1]; pa.ncz = ctx->G.nc[2];
    pa.zorder = ctx->G.zorder;
    pa.cellx = (float)ctx->G.cell[0]; pa.celly = (float)ctx->G.cell[1]; pa.cellz = (float)ctx->G.cell[2];
    pa.k2 = (float)(ctx->radius_scale * ctx->radius_scale);
    pa.kfac = (float)kernel_fac(ctx->kernel, ctx->dim);
    pa.deltap = (float)kernel_deltap(ctx->kernel);
    bool sumdens = false;
    for (int d = 0; d < B200SPH_MAX_ARRAYS; d++) {
        unsigned long long m = 0;
        for (int s = 0; s < B200SPH_MAX_ARRAYS; s++) {
            const uint32_t b = (d < ctx->narr && s < ctx->narr) ? prog->eqmask[d][s] : 0u;
            if (b > 0xFFu) return set_err(ctx, "pair_pass: unknown equation bits 0x%x", b);
            m |= (unsigned long long)b << (8 * s);
            if (b & B200SPH_EQ_SUMMATION_DENSITY) sumdens = true;
        }
        pa.emask[d] = m;
    }
    pa.c0 = (float)prog->c0; pa.alpha = (float)prog->alpha; pa.beta = (float)prog->beta;
    pa.gx = (float)prog->gx; pa.gy = (float)prog->gy; pa.gz = (float)prog->gz;
    pa.eps_xsph = (float)prog->eps_xsph;
    pa.nu4 = (float)(4.0 * prog->nu); pa.eta = (float)prog->eta;
    pa.tensile = prog->tensile_correction;
    pa.real_only = prog->real_only;
    if (r32) {
        pa.R = ctx->R;
        for (int c = 0; c < 2; c++) pa.r32_rep[c] = r32p.rep[c], pa.r32_m[c] = r32p.m[c], pa.r32_coef[c] = r32p.coef[c];
    }
    if (ranged)
        for (int d = 0; d < ctx->narr; d++) {
            pa.doff[d] = ctx->arr[d].off;
            pa.dlo[d] = ctx->dst_lo[d];
            pa.dhi[d] = ctx->dst_hi[d] < 0 ? (int64_t)1 << 62 : ctx->dst_hi[d];
        }
    pa.pair_counter = nullptr;
    if (pairs_out) {
        CU(cudaMemsetAsync(ctx->counter, 0, 8, ctx->stream));
        pa.pair_counter = ctx->counter;
    }
    if (use_lists) {
        // phase 0: every CTA, or (overlap) the ghost-free CTAs on the main stream; phase 1: the
        // others on the COMMUNICATION stream, in order behind the halo scatter -- the two
        // launches run side by side, the boundary CTAs (higher stream priority) take the SM
        // slots the interior CTAs free, and there is one tail instead of two.  The main
        // stream joins when the next entry point needs the results (sync_comm).
        for (int phase = 0; phase < (overlap ? 2 : 1); phase++) {
            const uint32_t *ids = !overlap ? nullptr : (phase == 0 ? ctx->chunk_interior : ctx->chunk_boundary);
            const unsigned nb = (unsigned)(!overlap ? cdiv(ctx->n_sorted, LIST_NT) : (phase == 0 ? ctx->n_chunk_interior : ctx->n_chunk_boundary));
            cudaStream_t lst_stream = ctx->stream;
            if (phase == 1) {
                lst_stream = ctx->comm_stream;
                if ((rc = eos_flush(ctx, ctx->comm_stream))) return rc;   // pool side of the speculated EOS, ghosts included
                ctx->n_overlapped++;
            }
            if (nb == 0) continue;
            // The interior CTAs of the first wave hold every SM slot for a whole CTA lifetime
            // (~50 us): the outgoing messages go first, and the receiving CTAs (next on the
            // communication stream, higher priority) get their slots before the wave does.
            if (overlap && phase == 0 && ctx->push_first) CU(cudaStreamWaitEvent(ctx->stream, ctx->ev_pushed, 0));
            switch (ctx->kernel * 4 + ctx->dim) {
#define LIST_LAUNCH(K, D, M, Q) k_pair_list<K, D, M, Q><<<nb, LIST_NT, 0, lst_stream>>>(pa, ctx->cnt, ctx->lst, ctx->capg, ids)
#define LIST_LAUNCH_R32(K, D, M) k_pair_list<K, D, M, PAIR_EQS_WCSPH, false, true><<<nb, LIST_NT, 0, lst_stream>>>(pa, ctx->cnt, ctx->lst, ctx->capg, ids)
#define LIST_CASE(K, D)                                                          \
    case K * 4 + D:                                                              \
        if (ranged) k_pair_list<K, D, 6, PAIR_EQS_ALL, true><<<nb, LIST_NT, 0, lst_stream>>>(pa, ctx->cnt, ctx->lst, ctx->capg, ids); \
        else if (r32 && ctx->pair_minb_r32 >= 8) LIST_LAUNCH_R32(K, D, 8);          \
        else if (r32) LIST_LAUNCH_R32(K, D, 7);                                    \
        else if (wcsph_only && ctx->pair_minb >= 8) LIST_LAUNCH(K, D, 8, PAIR_EQS_WCSPH); \
        else if (wcsph_only && ctx->pair_minb == 7) LIST_LAUNCH(K, D, 7, PAIR_EQS_WCSPH); \
        else if (ctx->pair_minb >= 7) LIST_LAUNCH(K, D, 7, PAIR_EQS_ALL);          \
        else LIST_LAUNCH(K, D, 6, PAIR_EQS_ALL);                                  \
        break;
                LIST_CASE(0, 1) LIST_CASE(0, 2) LIST_CASE(0, 3) LIST_CASE(1, 2) LIST_CASE(1, 3)
                LIST_CASE(2, 1) LIST_CASE(2, 2) LIST_CASE(2, 3) LIST_CASE(3, 1) LIST_CASE(3, 2) LIST_CASE(3, 3)
#undef LIST_LAUNCH
#undef LIST_LAUNCH_R32
#undef LIST_CASE
            default: return set_err(ctx, "pair_pass: unsupported kernel/dim combination");
            }
            LAUNCH_CHECK();
        }
        if (overlap) {   // the join point moves behind the boundary launch
            CU(cudaEventRecord(ctx->ev_join, ctx->comm_stream));
            ctx->comm_pending = true;
            if (ctx->profiling && ctx->halo_ev_fork && ctx->halo_ev_chain) {
                cudaEvent_t e_end = nullptr;
                if (!ctx->ev_pool.empty()) { e_end = ctx->ev_pool.back(); ctx->ev_pool.pop_back(); }
                else CU(cudaEventCreate(&e_end));
                CU(cudaEventRecord(e_end, ctx->comm_stream));
                ctx->halo_pending.push_back({ctx->halo_ev_fork, ctx->halo_ev_chain, e_end, ctx->halo_ev_sent, ctx->halo_ev_reduced});
                ctx->halo_ev_fork = ctx->halo_ev_chain = ctx->halo_ev_sent = ctx->halo_ev_reduced = nullptr;
            }
        }
        ctx->stats.pair_launches++;
        if (r32) ctx->n_pair_r32++;
    } else if (ctx->n_sorted > 0) {
        const unsigned nb = (unsigned)cdiv(ctx->n_sorted, PAIR_WARPS * PAIR_CHUNK);
        switch (ctx->kernel) {
        case 0: launch_pair_dim<0>(ctx->dim, nb, ctx->stream, pa); break;
        case 1: launch_pair_dim<1>(ctx->dim, nb, ctx->stream, pa); break;
        case 2: launch_pair_dim<2>(ctx->dim, nb, ctx->stream, pa); break;
        default: launch_pair_dim<3>(ctx->dim, nb, ctx->stream, pa); break;
        }
        LAUNCH_CHECK();
        ctx->stats.pair_launches++;
    }
    if (pairs_out) {
        CU(cudaMemcpyAsync(ctx->counter_host, ctx->counter, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        *pairs_out = (int64_t)ctx->counter_host[0];
        ctx->stats.pairs += *pairs_out;
    }
    if (sumdens) ctx->state_packed = false;  // rho changed
    return 0;
}

int b200sph_tvf_pass(b200sph_ctx *ctx, const b200sph_tvf_program *prog, int64_t *pairs_out)
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if ((rc = eos_flush(ctx))) return rc;
    if (!ctx->grid_valid) return set_err(ctx, "tvf_pass: the NNPS is stale (particles were pushed/resized); call nnps_update first");
    if (!(prog->passes & 7)) return set_err(ctx, "tvf_pass: passes must select group 1, the average-pressure group and/or group 2");
    if (prog->eqbits > 255u) return set_err(ctx, "tvf_pass: unknown equation bits 0x%x", prog->eqbits);
    const bool ext = (prog->eqbits & (B200SPH_TVF_MOM | B200SPH_TVF_XSPH)) != 0;
    if (ext && (prog->eqbits & (B200SPH_TVF_PGRAD | B200SPH_TVF_ASTRESS)))
        return set_err(ctx, "tvf_pass: equations of the internal-flow (transport velocity) and of the external-flow branch in one Group");
    if (prog->clamp_p && !prog->solid_mask) return set_err(ctx, "tvf_pass: ClampWallPressure without a solid wall");
    if (prog->fluid_mask == 0 || prog->fluid_mask >= (1u << ctx->narr)) return set_err(ctx, "tvf_pass: bad fluid mask 0x%x", prog->fluid_mask);
    const unsigned solid_mask = prog->solid_mask;
    if (solid_mask >= (1u << ctx->narr) || (solid_mask & prog->fluid_mask))
        return set_err(ctx, "tvf_pass: bad solid mask 0x%x (fluids 0x%x)", solid_mask, prog->fluid_mask);
    if ((prog->eqbits & B200SPH_TVF_NOSLIP) && !solid_mask) return set_err(ctx, "tvf_pass: SolidWallNoSlipBC without a solid wall");
    if ((prog->passes & 4) && ext) return set_err(ctx, "tvf_pass: the external-flow branch has no average pressure");
    if ((prog->passes & 4) && !solid_mask) return set_err(ctx, "tvf_pass: the average pressure has a Group of its own only with solid walls");
    if ((prog->passes & 1) && solid_mask && prog->bql)
        return set_err(ctx, "tvf_pass: with solid walls the average pressure is computed after the wall pressure (passes bit 2), not in group 1");
    if (solid_mask && (ctx->peer_box || ctx->comm_pending)) return set_err(ctx, "tvf_pass: EDAC with solid walls runs on one GPU");
    const bool use_lists = ctx->force_kernel == 0 && ctx->n_sorted > 0 && ctx->n_sorted < (1LL << LIST_JBITS);
    if (ctx->n_sorted == 0) return 0;
    if (!use_lists) return set_err(ctx, "tvf_pass: the EDAC kernels need the neighbour-list path (B200SPH_PAIR_KERNEL=list, < 2^26 particles)");
    if (ctx->lists_valid && !lists_cover(ctx, nullptr)) ctx->lists_valid = false;   // (these passes take unfiltered lists)
    if (!ctx->lists_valid) {
        PhaseTimer pt_build(ctx, 0);
        if ((rc = build_lists(ctx, nullptr))) return rc;
    }
    // timing slots: pack + group 1 count as "other", group 2 (the dominant kernel) as "pair"
    std::unique_ptr<PhaseTimer> pt(new PhaseTimer(ctx, 2));
    const unsigned nbp = (unsigned)cdiv(ctx->n_sorted, 256);
    k_pack_tvf<<<nbp, 256, 0, ctx->stream>>>(ctx->f64[B200SPH_U], ctx->f64[B200SPH_V], ctx->f64[B200SPH_W], ctx->f64[B200SPH_M],
                                             ctx->f64x[B200SPH_UHAT - B200SPH_UHAT], ctx->f64x[B200SPH_VHAT - B200SPH_UHAT],
                                             ctx->f64x[B200SPH_WHAT - B200SPH_UHAT], ctx->f64x[B200SPH_PF - B200SPH_UHAT],
                                             ctx->f32x[B200SPH_PAVG - B200SPH_VOL], ctx->ptype, ctx->perm, ctx->n_sorted,
                                             ctx->B, ctx->AB, ctx->C, ctx->Dv, ctx->PT, ctx->f64[B200SPH_RHO], solid_mask);
    LAUNCH_CHECK();
    ctx->state_packed = false;   // B / C no longer hold the WCSPH records

    TvfArgs ta;
    memset(&ta, 0, sizeof(ta));
    ta.AB = ctx->AB; ta.C2 = ctx->C; ta.Dv = ctx->Dv; ta.PT = ctx->PT; ta.perm = ctx->perm;
    ta.rho = ctx->f64[B200SPH_RHO];
    ta.V = ctx->f32x[B200SPH_VOL - B200SPH_VOL]; ta.pavg = ctx->f32x[B200SPH_PAVG - B200SPH_VOL];
    ta.au = ctx->f32[B200SPH_AU - N_F64]; ta.av = ctx->f32[B200SPH_AV - N_F64]; ta.aw = ctx->f32[B200SPH_AW - N_F64];
    ta.auhat = ctx->f32x[B200SPH_AUHAT - B200SPH_VOL]; ta.avhat = ctx->f32x[B200SPH_AVHAT - B200SPH_VOL];
    ta.awhat = ctx->f32x[B200SPH_AWHAT - B200SPH_VOL]; ta.ap = ctx->f32x[B200SPH_AP - B200SPH_VOL];
    ta.n = ctx->n_sorted;
    ta.cellx = (float)ctx->G.cell[0]; ta.celly = (float)ctx->G.cell[1]; ta.cellz = (float)ctx->G.cell[2];
    ta.k2 = (float)(ctx->radius_scale * ctx->radius_scale);
    ta.kfac = (float)kernel_fac(ctx->kernel, ctx->dim);
    ta.fluid_mask = prog->fluid_mask;
    ta.solid_mask = solid_mask;
    ta.src_mask = prog->fluid_mask | solid_mask;
    ta.eqbits = prog->eqbits;
    ta.bql = prog->bql;
    ta.wgx = (float)prog->gx; ta.wgy = (float)prog->gy; ta.wgz = (float)prog->gz;
    ta.eps_xsph = (float)prog->eps_xsph;
    ta.clamp_p = prog->clamp_p;
    ta.ax = ctx->f32[B200SPH_AX - N_F64]; ta.ay = ctx->f32[B200SPH_AY - N_F64]; ta.az = ctx->f32[B200SPH_AZ - N_F64];
    ta.p32 = ctx->f32[B200SPH_P - N_F64];
    ta.ug = ctx->f64x[B200SPH_UHAT - B200SPH_UHAT]; ta.vg = ctx->f64x[B200SPH_VHAT - B200SPH_UHAT];
    ta.wg = ctx->f64x[B200SPH_WHAT - B200SPH_UHAT];
    ta.pb = (float)prog->pb; ta.nu = (float)prog->nu; ta.edac_nu = (float)prog->edac_nu;
    ta.c0 = (float)prog->c0; ta.alpha = (float)prog->alpha;
    double damp = 1.0;   // wc/edac.py:483-488
    if (prog->t < prog->tdamp) damp = 0.5 * (std::sin((-0.5 + prog->t / prog->tdamp) * 3.14159265358979323846) + 1.0);
    ta.gx = (float)(prog->gx * damp); ta.gy = (float)(prog->gy * damp); ta.gz = (float)(prog->gz * damp);
    if (pairs_out) {
        CU(cudaMemsetAsync(ctx->counter, 0, 8, ctx->stream));
        ta.pair_counter = ctx->counter;
    }
    const unsigned nb = (unsigned)cdiv(ctx->n_sorted, LIST_NT);
    // stages: 1 group 1 (fluids), 2 group 1 (wall arrays), 3 the average-pressure group, 4 group 2
    for (int stage = 1; stage <= 4; stage++) {
        const int pass = stage == 4 ? 2 : 1;
        if (stage == 4) {
            pt.reset();
            pt.reset(new PhaseTimer(ctx, 1));
        }
        if (stage == 1 && !(prog->passes & 1)) continue;
        if (stage == 2 && !((prog->passes & 1) && solid_mask)) continue;
        if (stage == 3 && !(prog->passes & 4)) continue;
        if (stage == 4 && !(prog->passes & 2)) continue;
        ta.avg_only = stage == 3 ? 1 : 0;
        if (stage == 3) ta.bql = 1;
        switch (ctx->kernel * 4 + ctx->dim) {
#define TVF_CASE(K, D)                                                                                   \
    case K * 4 + D:                                                                                      \
        if (stage == 2) k_tvf_wall<K, D><<<nb, LIST_NT, 0, ctx->stream>>>(ta, ctx->cnt, ctx->lst, ctx->capg); \
        else if (pass == 1) k_tvf_pass1<K, D><<<nb, LIST_NT, 0, ctx->stream>>>(ta, ctx->cnt, ctx->lst, ctx->capg); \
        else if (ext) k_tvf_pass2<K, D, true, true><<<nb, LIST_NT, 0, ctx->stream>>>(ta, ctx->cnt, ctx->lst, ctx->capg); \
        else if (solid_mask) k_tvf_pass2<K, D, true><<<nb, LIST_NT, 0, ctx->stream>>>(ta, ctx->cnt, ctx->lst, ctx->capg); \
        else k_tvf_pass2<K, D><<<nb, LIST_NT, 0, ctx->stream>>>(ta, ctx->cnt, ctx->lst, ctx->capg);            \
        break;
            TVF_CASE(0, 1) TVF_CASE(0, 2) TVF_CASE(0, 3) TVF_CASE(1, 2) TVF_CASE(1, 3)
            TVF_CASE(2, 1) TVF_CASE(2, 2) TVF_CASE(2, 3) TVF_CASE(3, 1) TVF_CASE(3, 2) TVF_CASE(3, 3)
#undef TVF_CASE
        default: return set_err(ctx, "tvf_pass: unsupported kernel/dim combination");
        }
        LAUNCH_CHECK();
        if (stage == 3) ta.bql = prog->bql;
        if (pass == 2) ctx->stats.pair_launches++;
    }
    pt.reset();
    if (pairs_out) {
        CU(cudaMemcpyAsync(ctx->counter_host, ctx->counter, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        *pairs_out = (int64_t)ctx->counter_host[0];
        ctx->stats.pairs += *pairs_out;
    }
    return 0;
}

int b200sph_solid_pass(b200sph_ctx *ctx, const b200sph_solid_program *prog, int64_t *pairs_out)
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if ((rc = eos_flush(ctx))) return rc;
    if ((rc = ensure_solid(ctx))) return rc;
    if (!ctx->grid_valid) return set_err(ctx, "solid_pass: the NNPS is stale (particles were pushed/resized); call nnps_update first");
    if (!(prog->passes & 3)) return set_err(ctx, "solid_pass: passes must select group 1 and/or group 2");
    if (prog->elastic_mask == 0 || prog->elastic_mask >= (1u << ctx->narr)) return set_err(ctx, "solid_pass: bad elastic mask 0x%x", prog->elastic_mask);
    if (ctx->n_sorted == 0) return 0;
    const bool use_lists = ctx->force_kernel == 0 && ctx->n_sorted < (1LL << LIST_JBITS);
    if (!use_lists) return set_err(ctx, "solid_pass: the elastic-dynamics kernels need the neighbour-list path");
    if (ctx->lists_valid && !lists_cover(ctx, nullptr)) ctx->lists_valid = false;   // (these passes take unfiltered lists)
    if (!ctx->lists_valid) {
        PhaseTimer pt_build(ctx, 0);
        if ((rc = build_lists(ctx, nullptr))) return rc;
    }
    SolidArgs sa;
    memset(&sa, 0, sizeof(sa));
    sa.AB = ctx->AB; sa.C3 = ctx->C; sa.T01 = ctx->T01; sa.T2R = ctx->T2R; sa.R2 = ctx->R2; sa.perm = ctx->perm;
    sa.rho = ctx->f64[B200SPH_RHO];
    for (int k = 0; k < 6; k++) {
        sa.s[k] = ctx->f64s[k];
        sa.r[k] = ctx->f32s[9 + k];
        sa.as[k] = ctx->f32s[15 + k];
    }
    for (int k = 0; k < 9; k++) sa.vg[k] = ctx->f32s[k];
    sa.p = ctx->f32[B200SPH_P - N_F64];
    sa.arho = ctx->f32[B200SPH_ARHO - N_F64];
    sa.au = ctx->f32[B200SPH_AU - N_F64]; sa.av = ctx->f32[B200SPH_AV - N_F64]; sa.aw = ctx->f32[B200SPH_AW - N_F64];
    sa.ax = ctx->f32[B200SPH_AX - N_F64]; sa.ay = ctx->f32[B200SPH_AY - N_F64]; sa.az = ctx->f32[B200SPH_AZ - N_F64];
    sa.n = ctx->n_sorted;
    sa.cellx = (float)ctx->G.cell[0]; sa.celly = (float)ctx->G.cell[1]; sa.cellz = (float)ctx->G.cell[2];
    sa.k2 = (float)(ctx->radius_scale * ctx->radius_scale);
    sa.kfac = (float)kernel_fac(ctx->kernel, ctx->dim);
    sa.elastic_mask = prog->elastic_mask;
    sa.source_mask = prog->source_mask ? prog->source_mask : prog->elastic_mask;
    if ((sa.source_mask & sa.elastic_mask) != sa.elastic_mask) return set_err(ctx, "solid_pass: every elastic array must be a source");
    sa.grad3d = prog->grad3d;
    sa.ghost_group1 = prog->ghost_group1;
    sa.eps = (float)prog->eps; sa.alpha = (float)prog->alpha; sa.beta = (float)prog->beta; sa.eps_xsph = (float)prog->eps_xsph;
    for (int a = 0; a < B200SPH_MAX_ARRAYS; a++) {
        sa.c0_ref[a] = prog->c0_ref[a]; sa.rho_ref[a] = prog->rho_ref[a]; sa.G[a] = prog->G[a];
        sa.wdeltap[a] = (float)prog->wdeltap[a]; sa.nexp[a] = (float)prog->n[a];
    }
    if (pairs_out) {
        CU(cudaMemsetAsync(ctx->counter, 0, 8, ctx->stream));
        sa.pair_counter = ctx->counter;
    }
    std::unique_ptr<PhaseTimer> pt(new PhaseTimer(ctx, 2));
    if (prog->passes & 1) {
        // group 2 alone reuses the records the last group 1 left behind
        k_pack_solid<<<(unsigned)cdiv(ctx->n_sorted, 256), 256, 0, ctx->stream>>>(
            ctx->f64[B200SPH_U], ctx->f64[B200SPH_V], ctx->f64[B200SPH_W], ctx->f64[B200SPH_M], ctx->f64[B200SPH_RHO],
            ctx->f32[B200SPH_P - N_F64], ctx->f32[B200SPH_CS - N_F64], ctx->ptype, ctx->perm, ctx->n_sorted, ctx->B, ctx->AB, ctx->C);
        LAUNCH_CHECK();
        ctx->state_packed = false;
    }
    const unsigned nb = (unsigned)cdiv(ctx->n_sorted, LIST_NT);
    for (int pass = 1; pass <= 2; pass++) {
        if (pass == 2) {
            pt.reset();
            pt.reset(new PhaseTimer(ctx, 1));
        }
        if (!(prog->passes & pass)) continue;
        switch (ctx->kernel * 4 + ctx->dim) {
#define SOLID_CASE(K, D)                                                                                    \
    case K * 4 + D:                                                                                         \
        if (pass == 1) k_solid_pass1<K, D><<<nb, LIST_NT, 0, ctx->stream>>>(sa, ctx->cnt, ctx->lst, ctx->capg); \
        else k_solid_pass2<K, D><<<nb, LIST_NT, 0, ctx->stream>>>(sa, ctx->cnt, ctx->lst, ctx->capg);            \
        break;
            SOLID_CASE(0, 1) SOLID_CASE(0, 2) SOLID_CASE(0, 3) SOLID_CASE(1, 2) SOLID_CASE(1, 3)
            SOLID_CASE(2, 1) SOLID_CASE(2, 2) SOLID_CASE(2, 3) SOLID_CASE(3, 1) SOLID_CASE(3, 2) SOLID_CASE(3, 3)
#undef SOLID_CASE
        default: return set_err(ctx, "solid_pass: unsupported kernel/dim combination");
        }
        LAUNCH_CHECK();
        if (pass == 2) ctx->stats.pair_launches++;
    }
    pt.reset();
    if (pairs_out) {
        CU(cudaMemcpyAsync(ctx->counter_host, ctx->counter, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        *pairs_out = (int64_t)ctx->counter_host[0];
        ctx->stats.pairs += *pairs_out;
    }
    return 0;
}

static int ensure_tc(b200sph_ctx *ctx);
static int stage_solid_impl(b200sph_ctx *ctx, int arr, int which, double dt, bool devdt)
{
    if (int rcc = require_confirmed(ctx, "stage_solid")) return rcc;
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if ((rc = ensure_solid(ctx))) return rc;
    if (arr >= ctx->narr) return set_err(ctx, "stage_solid: bad array %d", arr);
    if (which < 0 || which > 2) return set_err(ctx, "stage_solid: which must be 0 (initialize), 1 (stage1) or 2 (stage2)");
    if (devdt && (rc = ensure_tc(ctx))) return rc;
    PhaseTimer pt(ctx, 2);
    StageSolidArgs sa;
    sa.x = ctx->f64[B200SPH_X]; sa.y = ctx->f64[B200SPH_Y]; sa.z = ctx->f64[B200SPH_Z];
    sa.u = ctx->f64[B200SPH_U]; sa.v = ctx->f64[B200SPH_V]; sa.w = ctx->f64[B200SPH_W]; sa.rho = ctx->f64[B200SPH_RHO];
    sa.x0 = ctx->f64[B200SPH_X0]; sa.y0 = ctx->f64[B200SPH_Y0]; sa.z0 = ctx->f64[B200SPH_Z0];
    sa.u0 = ctx->f64[B200SPH_U0]; sa.v0 = ctx->f64[B200SPH_V0]; sa.w0 = ctx->f64[B200SPH_W0]; sa.rho0 = ctx->f64[B200SPH_RHO0];
    for (int k = 0; k < 6; k++) {
        sa.s[k] = ctx->f64s[k];
        sa.s0[k] = ctx->f64s[6 + k];
        sa.as[k] = ctx->f32s[15 + k];
    }
    sa.au = ctx->f32[B200SPH_AU - N_F64]; sa.av = ctx->f32[B200SPH_AV - N_F64]; sa.aw = ctx->f32[B200SPH_AW - N_F64];
    sa.ax = ctx->f32[B200SPH_AX - N_F64]; sa.ay = ctx->f32[B200SPH_AY - N_F64]; sa.az = ctx->f32[B200SPH_AZ - N_F64];
    sa.arho = ctx->f32[B200SPH_ARHO - N_F64];
    sa.ptype = ctx->ptype;
    sa.pool_end = ctx->pool_end;
    sa.arr = arr;
    sa.which = which;
    sa.f = which == 1 ? 0.5 * dt : dt;
    if (ctx->pool_end > 0) {
        if (devdt) k_stage_solid_devdt<<<(unsigned)cdiv(ctx->pool_end, 256), 256, 0, ctx->stream>>>(sa, ctx->tc);
        else k_stage_solid<<<(unsigned)cdiv(ctx->pool_end, 256), 256, 0, ctx->stream>>>(sa);
        LAUNCH_CHECK();
    }
    if (which != 0) {
        ctx->grid_valid = false, ctx->packed_valid = false;
        ctx->state_packed = false;
    }
    return 0;
}
int b200sph_stage_solid(b200sph_ctx *ctx, int arr, int which, double dt) { return stage_solid_impl(ctx, arr, which, dt, false); }
int b200sph_stage_solid_dev(b200sph_ctx *ctx, int arr, int which) { return stage_solid_impl(ctx, arr, which, 0.0, true); }

static int ensure_tc(b200sph_ctx *ctx);
static int stage_tvf_impl(b200sph_ctx *ctx, int arr, int which, double dt, bool devdt, int ext = 0)
{
    if (int rcc = require_confirmed(ctx, "stage_tvf")) return rcc;
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if (arr >= ctx->narr) return set_err(ctx, "stage_tvf: bad array %d", arr);
    if (which < 0 || which > 2) return set_err(ctx, "stage_tvf: which must be 0 (initialize), 1 (stage1) or 2 (stage2)");
    if (devdt && (rc = ensure_tc(ctx))) return rc;
    PhaseTimer pt(ctx, 2);
    StageTvfArgs sa;
    sa.x = ctx->f64[B200SPH_X]; sa.y = ctx->f64[B200SPH_Y]; sa.z = ctx->f64[B200SPH_Z];
    sa.u = ctx->f64[B200SPH_U]; sa.v = ctx->f64[B200SPH_V]; sa.w = ctx->f64[B200SPH_W];
    sa.x0 = ctx->f64[B200SPH_X0]; sa.y0 = ctx->f64[B200SPH_Y0]; sa.z0 = ctx->f64[B200SPH_Z0];
    sa.u0 = ctx->f64[B200SPH_U0]; sa.v0 = ctx->f64[B200SPH_V0]; sa.w0 = ctx->f64[B200SPH_W0];
    sa.uh = ctx->f64x[B200SPH_UHAT - B200SPH_UHAT]; sa.vh = ctx->f64x[B200SPH_VHAT - B200SPH_UHAT];
    sa.wh = ctx->f64x[B200SPH_WHAT - B200SPH_UHAT];
    sa.pf = ctx->f64x[B200SPH_PF - B200SPH_UHAT]; sa.pf0 = ctx->f64x[B200SPH_PF0 - B200SPH_UHAT];
    sa.au = ctx->f32[B200SPH_AU - N_F64]; sa.av = ctx->f32[B200SPH_AV - N_F64]; sa.aw = ctx->f32[B200SPH_AW - N_F64];
    sa.auh = ctx->f32x[B200SPH_AUHAT - B200SPH_VOL]; sa.avh = ctx->f32x[B200SPH_AVHAT - B200SPH_VOL];
    sa.awh = ctx->f32x[B200SPH_AWHAT - B200SPH_VOL]; sa.ap = ctx->f32x[B200SPH_AP - B200SPH_VOL];
    sa.ptype = ctx->ptype;
    sa.pool_end = ctx->pool_end;
    sa.arr = arr;
    sa.which = which;
    sa.f = which == 1 ? 0.5 * dt : dt;
    sa.ext = ext;
    sa.ax = ctx->f32[B200SPH_AX - N_F64]; sa.ay = ctx->f32[B200SPH_AY - N_F64]; sa.az = ctx->f32[B200SPH_AZ - N_F64];
    if (ctx->pool_end > 0) {
        if (devdt) k_stage_tvf_devdt<<<(unsigned)cdiv(ctx->pool_end, 256), 256, 0, ctx->stream>>>(sa, ctx->tc);
        else k_stage_tvf<<<(unsigned)cdiv(ctx->pool_end, 256), 256, 0, ctx->stream>>>(sa);
        LAUNCH_CHECK();
    }
    if (which != 0) {
        ctx->grid_valid = false, ctx->packed_valid = false;
        ctx->state_packed = false;
    }
    return 0;
}
int b200sph_stage_tvf(b200sph_ctx *ctx, int arr, int which, double dt) { return stage_tvf_impl(ctx, arr, which, dt, false); }
int b200sph_stage_tvf_dev(b200sph_ctx *ctx, int arr, int which) { return stage_tvf_impl(ctx, arr, which, 0.0, true); }
int b200sph_stage_edac(b200sph_ctx *ctx, int arr, int which, double dt) { return stage_tvf_impl(ctx, arr, which, dt, false, 1); }
int b200sph_stage_edac_dev(b200sph_ctx *ctx, int arr, int which) { return stage_tvf_impl(ctx, arr, which, 0.0, true, 1); }

static int ensure_tc(b200sph_ctx *ctx)
{
    if (ctx->tc) return 0;
    CU(cudaMalloc((void **)&ctx->tc, 8 * sizeof(double)));
    ctx->tc_owned = true;
    const double init[8] = {0.0, 0.0, 1e20, -1.0, 0.0, 0.0, 0.0, 0.0};
    CU(cudaMemcpy(ctx->tc, init, sizeof(init), cudaMemcpyHostToDevice));
    return 0;
}

// the fused stage kernel applies when one launch steps every array (arr == -1) and the
// neighbour lists of the current build can be reused: then the records of the next
// evaluation can be written at the particles' frozen sorted slots
static bool can_fuse_stage(const b200sph_ctx *ctx, int arr)
{
    if (!ctx->fuse || arr != -1 || ctx->force_kernel != 0) return false;
    if (!ctx->lists_valid || ctx->topo_dirty || ctx->n_sorted <= 0) return false;
    if (ctx->periodic[0] || ctx->periodic[1] || ctx->periodic[2] || mirror_any(ctx)) return false;
    int64_t ntot = 0;
    for (int a = 0; a < ctx->narr; a++) ntot += ctx->arr[a].n;
    return ntot == ctx->n_sorted && ntot < (1LL << LIST_JBITS);
}

static int stage_impl(b200sph_ctx *ctx, int arr, int which, double dt, bool devdt)
{
    if (int rcc = require_confirmed(ctx, "stage")) return rcc;
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if ((rc = eos_flush(ctx))) return rc;
    if (arr >= ctx->narr) return set_err(ctx, "stage: bad array %d", arr);
    if (which < 0 || which > 2) return set_err(ctx, "stage: which must be 0 (initialize), 1 (stage1) or 2 (stage2)");
    if (devdt && (rc = ensure_tc(ctx))) return rc;
    PhaseTimer pt(ctx, 2);
    StageArgs sa;
    sa.x = ctx->f64[B200SPH_X]; sa.y = ctx->f64[B200SPH_Y]; sa.z = ctx->f64[B200SPH_Z];
    sa.u = ctx->f64[B200SPH_U]; sa.v = ctx->f64[B200SPH_V]; sa.w = ctx->f64[B200SPH_W]; sa.rho = ctx->f64[B200SPH_RHO];
    sa.x0 = ctx->f64[B200SPH_X0]; sa.y0 = ctx->f64[B200SPH_Y0]; sa.z0 = ctx->f64[B200SPH_Z0];
    sa.u0 = ctx->f64[B200SPH_U0]; sa.v0 = ctx->f64[B200SPH_V0]; sa.w0 = ctx->f64[B200SPH_W0]; sa.rho0 = ctx->f64[B200SPH_RHO0];
    sa.au = ctx->f32[B200SPH_AU - N_F64]; sa.av = ctx->f32[B200SPH_AV - N_F64]; sa.aw = ctx->f32[B200SPH_AW - N_F64];
    sa.ax = ctx->f32[B200SPH_AX - N_F64]; sa.ay = ctx->f32[B200SPH_AY - N_F64]; sa.az = ctx->f32[B200SPH_AZ - N_F64];
    sa.arho = ctx->f32[B200SPH_ARHO - N_F64];
    sa.ptype = ctx->ptype;
    sa.pool_end = ctx->pool_end;
    sa.arr = arr;
    sa.which = which;
    sa.f = which == 1 ? 0.5 * dt : dt;
    if (which != 0 && ctx->pool_end > 0 && can_fuse_stage(ctx, arr)) {
        // stage + records of the next evaluation (+ the dt factors after stage2) in one pass
        FusePackArgs q;
        memset(&q, 0, sizeof(q));
        q.h = ctx->f64[B200SPH_H]; q.m = ctx->f64[B200SPH_M];
        q.p = ctx->f32[B200SPH_P - N_F64]; q.cs = ctx->f32[B200SPH_CS - N_F64];
        q.rank = ctx->rank; q.key_of = ctx->key_of;
        q.A0 = ctx->A0; q.AB = ctx->AB; q.C = ctx->C;
        q.R = ctx->R; q.r32_cls = ctx->r32_cls;
        q.G = ctx->G;
        q.red_u32 = ctx->red_u32;
        q.dt_cfl = ctx->f32[B200SPH_DT_CFL - N_F64]; q.dt_force = ctx->f32[B200SPH_DT_FORCE - N_F64];
        q.red = ctx->red;
        q.tc = devdt ? ctx->tc : nullptr;
        q.do_init = 0;
        q.reduce_dt = (which == 2 && ctx->dt_adaptive_seen) ? 1 : 0;
        q.eos_any = ctx->eos_last_valid ? 1 : 0;
        q.E = ctx->eos_last;
        if (q.reduce_dt && !ctx->red_armed) {
            k_red_init<<<1, 32, 0, ctx->stream>>>(ctx->red);
            LAUNCH_CHECK();
        }
        CU(cudaMemsetAsync(ctx->red_u32, 0, 2 * sizeof(unsigned), ctx->stream));
        k_stage_pack<<<(unsigned)cdiv(ctx->pool_end, 256), 256, 0, ctx->stream>>>(sa, q);
        LAUNCH_CHECK();
        ctx->n_fused++;
        if (q.reduce_dt) ctx->red_armed = false;
        if (which == 2) ctx->dt_reduced = q.reduce_dt != 0, ctx->dt_adaptive_seen = false;
        ctx->grid_valid = false;       // particles moved: nnps_update must decide about the lists
        ctx->packed_valid = true;      // ... but their packed positions are current,
        ctx->drift_measured = true;    // the drift of the build is in red_u32,
        ctx->state_packed = true;      // and so is their packed state,
        ctx->spec_records = ctx->eos_last_valid;   // with last evaluation's EOS calls applied
        ctx->spec_confirmed = 0;
        return 0;
    }
    if (ctx->pool_end > 0) {
        if (devdt) k_stage_devdt<<<(unsigned)cdiv(ctx->pool_end, 256), 256, 0, ctx->stream>>>(sa, ctx->tc);
        else k_stage<<<(unsigned)cdiv(ctx->pool_end, 256), 256, 0, ctx->stream>>>(sa);
        LAUNCH_CHECK();
    }
    if (which != 0) {
        ctx->grid_valid = false, ctx->packed_valid = false;  // particles moved: neighbours are stale until nnps_update
        ctx->state_packed = false;
        if (which == 2) ctx->dt_adaptive_seen = false, ctx->dt_reduced = false;
    }
    return 0;
}

int b200sph_stage(b200sph_ctx *ctx, int arr, int which, double dt) { return stage_impl(ctx, arr, which, dt, false); }
int b200sph_stage_dev(b200sph_ctx *ctx, int arr, int which) { return stage_impl(ctx, arr, which, 0.0, true); }

// ---- device-resident time step ------------------------------------------------
int b200sph_time_control(b200sph_ctx *ctx, double *external_block8, double **dev_block)
{
    CU(cudaSetDevice(ctx->device));
    if (external_block8) {
        if (ctx->tc_owned) CU(cudaFree(ctx->tc));
        ctx->tc = external_block8;
        ctx->tc_owned = false;
        const double init[8] = {0.0, 0.0, 1e20, -1.0, 0.0, 0.0, 0.0, 0.0};
        CU(cudaMemcpyAsync(ctx->tc, init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
    } else if (int rc = ensure_tc(ctx)) return rc;
    if (!ctx->tc_host) {
        CU(cudaMallocHost((void **)&ctx->tc_host, 4 * sizeof(double)));
        for (int i = 0; i < 2; i++) CU(cudaEventCreateWithFlags(&ctx->tc_evt[i], cudaEventDisableTiming));
    }
    if (dev_block) *dev_block = ctx->tc;
    return 0;
}

int b200sph_time_set(b200sph_ctx *ctx, double t, double dt)
{
    CU(cudaSetDevice(ctx->device));
    int rc = b200sph_time_control(ctx, nullptr, nullptr);
    if (rc) return rc;
    const double v[2] = {dt, t};
    CU(cudaMemcpyAsync(ctx->tc, v, sizeof(v), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}

// max dt_cfl, max dt_force, min h into red[9,11,12] -- unless the fused stage2 kernel has
// just left them there
static int reduce_dt_factors(b200sph_ctx *ctx)
{
    if (ctx->dt_reduced) return 0;
    k_red_init<<<1, 32, 0, ctx->stream>>>(ctx->red);
    LAUNCH_CHECK();
    if (ctx->pool_end > 0) {
        const unsigned nb = (unsigned)std::min<int64_t>(cdiv(ctx->pool_end, 256), 148 * 8);
        k_reduce_dt<<<nb, 256, 0, ctx->stream>>>(ctx->f32[B200SPH_DT_CFL - N_F64], ctx->f32[B200SPH_DT_FORCE - N_F64], ctx->f64[B200SPH_H],
                                                 ctx->ptype, ctx->pool_end, ctx->red);
        LAUNCH_CHECK();
    }
    ctx->red_armed = false;
    return 0;
}

int b200sph_dt_propose(b200sph_ctx *ctx, double cfl, int fixed_h)
{
    if (int rcc = require_confirmed(ctx, "dt_propose")) return rcc;
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if ((rc = b200sph_time_control(ctx, nullptr, nullptr))) return rc;
    PhaseTimer pt(ctx, 2);
    if ((rc = reduce_dt_factors(ctx))) return rc;
    k_dt_propose<<<1, 1, 0, ctx->stream>>>(ctx->red, ctx->tc, cfl, fixed_h);
    LAUNCH_CHECK();
    ctx->red_armed = true;
    ctx->dt_reduced = false;
    ctx->dt_adaptive_seen = true;
    return 0;
}

int b200sph_dt_advance(b200sph_ctx *ctx, double cfl, int fixed_h, double prev_factor, double new_factor, int adaptive, int advance,
                       int snapshot_slot)
{
    if (int rcc = require_confirmed(ctx, "dt_advance")) return rcc;
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if ((rc = b200sph_time_control(ctx, nullptr, nullptr))) return rc;
    if (!(prev_factor > 0.0) || !(new_factor > 0.0)) return set_err(ctx, "dt_advance: damping factors must be positive");
    if (snapshot_slot > 1) return set_err(ctx, "dt_advance: snapshot slot must be 0 or 1");
    PhaseTimer pt(ctx, 2);
    if (adaptive && (rc = reduce_dt_factors(ctx))) return rc;
    k_dt_advance<<<1, 1, 0, ctx->stream>>>(ctx->red, ctx->tc, cfl, fixed_h, prev_factor, new_factor, adaptive, advance, ctx->t_final, ctx->t_eps);
    LAUNCH_CHECK();
    ctx->red_armed = true;
    ctx->dt_reduced = false;
    ctx->dt_adaptive_seen = adaptive != 0;
    if (snapshot_slot >= 0) {
        CU(cudaMemcpyAsync(ctx->tc_host + 2 * snapshot_slot, ctx->tc, 2 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaEventRecord(ctx->tc_evt[snapshot_slot], ctx->stream));
    }
    return 0;
}

int b200sph_dt_commit(b200sph_ctx *ctx, double prev_factor, double new_factor, int in_parallel, int adaptive, int advance, int snapshot_slot)
{
    CU(cudaSetDevice(ctx->device));
    int rc = b200sph_time_control(ctx, nullptr, nullptr);
    if (rc) return rc;
    if (!(prev_factor > 0.0) || !(new_factor > 0.0)) return set_err(ctx, "dt_commit: damping factors must be positive");
    k_dt_commit<<<1, 1, 0, ctx->stream>>>(ctx->tc, prev_factor, new_factor, in_parallel, adaptive, advance, ctx->t_final, ctx->t_eps);
    LAUNCH_CHECK();
    if (snapshot_slot >= 0) {
        if (snapshot_slot > 1) return set_err(ctx, "dt_commit: snapshot slot must be 0 or 1");
        CU(cudaMemcpyAsync(ctx->tc_host + 2 * snapshot_slot, ctx->tc, 2 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaEventRecord(ctx->tc_evt[snapshot_slot], ctx->stream));
    }
    return 0;
}

int b200sph_time_final(b200sph_ctx *ctx, double t_final, double eps)
{
    if (!(eps >= 0.0) || t_final != t_final) return set_err(ctx, "time_final: bad final time / tolerance");
    ctx->t_final = t_final;
    ctx->t_eps = eps;
    return 0;
}

int b200sph_time_snapshot(b200sph_ctx *ctx, int slot, double out[2])
{
    if (slot < 0 || slot > 1 || !ctx->tc_host) return set_err(ctx, "time_snapshot: no snapshot in slot %d", slot);
    CU(cudaSetDevice(ctx->device));
    CU(cudaEventSynchronize(ctx->tc_evt[slot]));
    out[0] = ctx->tc_host[2 * slot];      // dt of the step that follows the snapshot
    out[1] = ctx->tc_host[2 * slot + 1];  // t at the snapshot
    return 0;
}

int b200sph_time_get(b200sph_ctx *ctx, double out[2])
{
    CU(cudaSetDevice(ctx->device));
    int rc = b200sph_time_control(ctx, nullptr, nullptr);
    if (rc) return rc;
    double v[2];
    CU(cudaMemcpyAsync(v, ctx->tc, sizeof(v), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    out[0] = v[0];
    out[1] = v[1];
    return 0;
}

int b200sph_dt_factors(b200sph_ctx *ctx, double out[3])
{
    if (int rcc = require_confirmed(ctx, "dt_factors")) return rcc;
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    PhaseTimer pt(ctx, 2);
    if ((rc = reduce_dt_factors(ctx))) return rc;
    ctx->dt_adaptive_seen = true;
    CU(cudaMemcpyAsync(ctx->red_host, ctx->red, 16 * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    const double mc = o2d(ctx->red_host[9]), mf = o2d(ctx->red_host[11]), hm = o2d(ctx->red_host[12]);
    out[0] = mc < -1e299 ? -1.0 : mc;  // _my_max of an empty property is -1.0, integrator.py:55-59
    out[1] = mf < -1e299 ? -1.0 : mf;
    out[2] = std::min(1.0, hm);        // compute_h_minimum starts from 1.0, integrator.py:149
    return 0;
}

// ---- halo helpers ------------------------------------------------------------
static const int halo_fields[9] = {B200SPH_X, B200SPH_Y, B200SPH_Z, B200SPH_U, B200SPH_V, B200SPH_W, B200SPH_RHO, B200SPH_H, B200SPH_M};

// with the elastic-dynamics arrays allocated the deviatoric stress travels too: a ghost is a
// source of group 2 (and, with SolidProgram.ghost_group1, a destination of group 1), and a
// migrating particle takes s and its stage copy s0 along
static inline int halo_nf(const b200sph_ctx *ctx) { return ctx->solid_alloc ? B200SPH_HALO_FIELDS_SOLID : B200SPH_HALO_FIELDS; }
static inline int migrate_nf(const b200sph_ctx *ctx) { return ctx->solid_alloc ? B200SPH_MIGRATE_FIELDS_SOLID : B200SPH_MIGRATE_FIELDS; }

static HaloPtrs halo_ptrs(b200sph_ctx *ctx)
{
    HaloPtrs P;
    for (int f = 0; f < B200SPH_HALO_FIELDS; f++) P.p[f] = ctx->f64[halo_fields[f]];
    for (int f = B200SPH_HALO_FIELDS; f < B200SPH_HALO_FIELDS_SOLID - 1; f++) P.p[f] = ctx->f64s[f - B200SPH_HALO_FIELDS];
    P.cs = ctx->f32[B200SPH_CS - N_F64];
    return P;
}

// ---- mirror boundaries ----------------------------------------------------------------
// DomainManager(mirror_in_x ...) nnps_base.pyx:506-689: every particle within n_layers cells
// of a mirror plane gets an image on the other side (position reflected, the normal velocity
// component negated, everything else copied), images of images at the corners: x images
// first, then y images of the real particles AND of the x images, then z images of
// everything.  The reference re-selects at every update_domain; here the selection lives as
// long as the neighbour lists (its width covers the skin) and nnps_update refreshes the
// images' values in creation order before every evaluation.
static int mirror_refresh(b200sph_ctx *ctx)
{
    const HaloPtrs P = halo_ptrs(ctx);
    for (const auto &sg : ctx->mirror_segs) {
        if (sg.count == 0) continue;
        const ArrayInfo &ai = ctx->arr[sg.arr];
        const double plane2 = 2.0 * (sg.side == 0 ? ctx->dom_lo[sg.axis] : ctx->dom_hi[sg.axis]);
        k_mirror_copy<<<(unsigned)cdiv(sg.count, 256), 256, 0, ctx->stream>>>(P, ai.off, sg.idx, sg.count, ai.off + ai.n_real + sg.ghost_first, sg.axis, plane2);
        LAUNCH_CHECK();
    }
    ctx->grid_valid = false, ctx->packed_valid = false;
    ctx->state_packed = false;
    return 0;
}

static int mirror_create(b200sph_ctx *ctx)
{
    int rc;
    if (ctx->solid_alloc) return set_err(ctx, "mirror boundaries: images carry the WCSPH fields only (x y z u v w rho h m), not the elastic-dynamics state");
    if ((rc = eos_flush(ctx))) return rc;
    // the cell size of the REAL particles decides the width (images have their sources' h)
    for (int a = 0; a < ctx->narr; a++) ctx->arr[a].n = ctx->arr[a].n_real;
    ctx->ptype_dirty = true;
    ctx->domain_valid = false;
    ctx->mirror_built = false;
    if ((rc = b200sph_update_domain(ctx))) return rc;
    const double width = ctx->mirror_layers * ctx->cell_size * (1.0 + (ctx->force_kernel == 0 ? ctx->skin : 0.0));
    size_t nseg = 0;
    for (int a = 0; a < ctx->narr; a++) {
        for (int axis = 0; axis < 3; axis++) {
            if (!ctx->mirror[axis]) continue;
            // both sides select from the particles present BEFORE this axis (real + earlier axes' images)
            const int64_t n_sel = ctx->arr[a].n;
            for (int side = 0; side < 2; side++) {
                if (nseg == ctx->mirror_segs.size()) ctx->mirror_segs.emplace_back();
                b200sph_ctx::MirrorSeg &sg = ctx->mirror_segs[nseg++];
                sg.arr = a, sg.axis = axis, sg.side = side, sg.count = 0;
                ArrayInfo &ai = ctx->arr[a];
                sg.ghost_first = ai.n - ai.n_real;
                if (n_sel == 0) continue;
                const unsigned nb = (unsigned)cdiv(n_sel + 1, 256);
                k_flag_mirror<<<nb, 256, 0, ctx->stream>>>(ctx->f64[B200SPH_X + axis], ai.off, n_sel, side == 0 ? ctx->dom_lo[axis] : ctx->dom_hi[axis], width, side, ctx->flag_a);
                LAUNCH_CHECK();
                if ((rc = device_scan(ctx, ctx->flag_a, ctx->flag_b, n_sel + 1))) return rc;
                uint32_t tot = 0;
                CU(cudaMemcpyAsync(&tot, ctx->flag_b + n_sel, 4, cudaMemcpyDeviceToHost, ctx->stream));
                CU(cudaStreamSynchronize(ctx->stream));
                if (tot == 0) continue;
                if ((int64_t)tot > sg.cap) {
                    if (sg.idx) CU(cudaFree(sg.idx));
                    sg.cap = (int64_t)tot + tot / 4 + 256;
                    CU(cudaMalloc((void **)&sg.idx, 4 * (size_t)sg.cap));
                }
                k_save_idx<<<nb, 256, 0, ctx->stream>>>(n_sel, ctx->flag_a, ctx->flag_b, sg.idx);
                LAUNCH_CHECK();
                if ((rc = ensure_capacity(ctx, a, ai.n + tot))) return rc;   // may move the pool
                const int64_t o = ai.off + ai.n;
                const unsigned nbt = (unsigned)cdiv((int64_t)tot, 256);
                k_mirror_copy<<<nbt, 256, 0, ctx->stream>>>(halo_ptrs(ctx), ai.off, sg.idx, (long long)tot, o, axis, 2.0 * (side == 0 ? ctx->dom_lo[axis] : ctx->dom_hi[axis]));
                LAUNCH_CHECK();
                // like halo_append for ghosts: stage copies and derived fields zero, no gid, tag = Ghost (2)
                for (int k = B200SPH_X0; k < N_F64; k++) CU(cudaMemsetAsync(ctx->f64[k] + o, 0, 8 * (size_t)tot, ctx->stream));
                for (int k = 0; k < N_F32; k++) CU(cudaMemsetAsync(ctx->f32[k] + o, 0, 4 * (size_t)tot, ctx->stream));
                k_fill_u32<<<nbt, 256, 0, ctx->stream>>>(ctx->u32[0] + o, tot, 0xFFFFFFFFu);
                LAUNCH_CHECK();
                k_fill_u32<<<nbt, 256, 0, ctx->stream>>>(ctx->u32[1] + o, tot, 2u);
                LAUNCH_CHECK();
                CU(cudaMemsetAsync(ctx->u32[2] + o, 0, 4 * (size_t)tot, ctx->stream));
                sg.count = tot;
                ai.n += tot;
            }
        }
    }
    ctx->mirror_segs.resize(nseg);   // (a shrinking narr never happens; keeps the vector tidy)
    ctx->mirror_built = true;
    ctx->ptype_dirty = true;
    ctx->grid_valid = false, ctx->packed_valid = false;
    ctx->topo_dirty = true;
    ctx->h_dirty = ctx->uni_dirty = true;
    ctx->domain_valid = false;
    ctx->state_packed = false;
    return 0;
}

int b200sph_halo_layout(b200sph_ctx *ctx, int *halo_fields_out, int *migrate_fields_out)
{
    if (halo_fields_out) *halo_fields_out = halo_nf(ctx);
    if (migrate_fields_out) *migrate_fields_out = migrate_nf(ctx);
    return 0;
}

int b200sph_halo_pack(b200sph_ctx *ctx, int arr, int slot, double lo, double hi, double *dev_buf, int64_t cap, int64_t *count)
{
    if (int rcc = require_confirmed(ctx, "halo_pack")) return rcc;
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if ((rc = eos_flush(ctx))) return rc;
    if (arr < 0 || arr >= ctx->narr) return set_err(ctx, "halo_pack: bad array %d", arr);
    const int64_t n = ctx->arr[arr].n_real, off = ctx->arr[arr].off;
    *count = 0;
    if (slot == 0 || slot == 1) ctx->halo_cnt[arr][slot] = 0;
    if (n == 0) return 0;
    const unsigned nb = (unsigned)cdiv(n + 1, 256);
    k_flag_range<<<nb, 256, 0, ctx->stream>>>(ctx->f64[B200SPH_X], off, n, lo, hi, 0, ctx->flag_a);
    LAUNCH_CHECK();
    if ((rc = device_scan(ctx, ctx->flag_a, ctx->flag_b, n + 1))) return rc;
    uint32_t tot = 0;
    CU(cudaMemcpyAsync(&tot, ctx->flag_b + n, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    *count = tot;
    if ((int64_t)tot > cap) return set_err(ctx, "halo_pack: %u particles selected but the buffer holds %lld", tot, (long long)cap);
    if (slot == 0 || slot == 1) {  // remember the selection for halo_pack_selected
        if ((int64_t)tot > ctx->halo_cap[arr][slot]) {
            if (ctx->halo_idx[arr][slot]) CU(cudaFree(ctx->halo_idx[arr][slot]));
            ctx->halo_cap[arr][slot] = (int64_t)tot + tot / 4 + 256;
            CU(cudaMalloc((void **)&ctx->halo_idx[arr][slot], 4 * (size_t)ctx->halo_cap[arr][slot]));
        }
        ctx->halo_cnt[arr][slot] = tot;
        if (tot) {
            k_save_idx<<<nb, 256, 0, ctx->stream>>>(n, ctx->flag_a, ctx->flag_b, ctx->halo_idx[arr][slot]);
            LAUNCH_CHECK();
        }
    } else if (slot != -1) {
        return set_err(ctx, "halo_pack: slot must be -1, 0 or 1");
    }
    if (tot == 0) return 0;
    if (halo_nf(ctx) == B200SPH_HALO_FIELDS) k_halo_gather_flag<B200SPH_HALO_FIELDS><<<nb, 256, 0, ctx->stream>>>(halo_ptrs(ctx), off, n, ctx->flag_a, ctx->flag_b, dev_buf, (long long)tot);
    else k_halo_gather_flag<B200SPH_HALO_FIELDS_SOLID><<<nb, 256, 0, ctx->stream>>>(halo_ptrs(ctx), off, n, ctx->flag_a, ctx->flag_b, dev_buf, (long long)tot);
    LAUNCH_CHECK();
    return 0;
}

int b200sph_halo_append(b200sph_ctx *ctx, int arr, const double *dev_buf, int64_t stride, int64_t n, int nfields, int as_real)
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if ((rc = eos_flush(ctx))) return rc;
    if (arr < 0 || arr >= ctx->narr) return set_err(ctx, "halo_append: bad array %d", arr);
    const int hnf = halo_nf(ctx), mnf = migrate_nf(ctx);
    if (nfields != hnf && nfields != mnf) return set_err(ctx, "halo_append: nfields must be %d or %d", hnf, mnf);
    ArrayInfo &ai = ctx->arr[arr];
    if (as_real && ai.n != ai.n_real) return set_err(ctx, "halo_append(as_real): drop the ghosts of '%s' first (real particles must precede ghosts)", ai.name.c_str());
    if (n <= 0) return 0;
    if ((rc = ensure_capacity(ctx, arr, ai.n + n))) return rc;
    const int64_t o = ai.off + ai.n;
    const unsigned nb = (unsigned)cdiv(n, 256);
    // derived fields of the appended particles start at zero (cs of an elastic array is then
    // filled from the message)
    for (int k = 0; k < N_F32; k++) CU(cudaMemsetAsync(ctx->f32[k] + o, 0, 4 * (size_t)n, ctx->stream));
    if (ctx->solid_alloc)
        for (int k = 0; k < 21; k++) CU(cudaMemsetAsync(ctx->f32s[k] + o, 0, 4 * (size_t)n, ctx->stream));
    if (nfields == hnf) {
        if (hnf == B200SPH_HALO_FIELDS) k_halo_scatter<B200SPH_HALO_FIELDS><<<nb, 256, 0, ctx->stream>>>(halo_ptrs(ctx), o, dev_buf, stride, n);
        else k_halo_scatter<B200SPH_HALO_FIELDS_SOLID><<<nb, 256, 0, ctx->stream>>>(halo_ptrs(ctx), o, dev_buf, stride, n);
        LAUNCH_CHECK();
        for (int k = B200SPH_X0; k < N_F64; k++) CU(cudaMemsetAsync(ctx->f64[k] + o, 0, 8 * (size_t)n, ctx->stream));
        if (ctx->solid_alloc)
            for (int k = 6; k < 12; k++) CU(cudaMemsetAsync(ctx->f64s[k] + o, 0, 8 * (size_t)n, ctx->stream));
        k_fill_u32<<<nb, 256, 0, ctx->stream>>>(ctx->u32[0] + o, n, 0xFFFFFFFFu);
        LAUNCH_CHECK();
    } else {
        for (int k = 0; k < N_F64; k++)
            CU(cudaMemcpyAsync(ctx->f64[k] + o, dev_buf + (size_t)k * stride, 8 * (size_t)n, cudaMemcpyDeviceToDevice, ctx->stream));
        k_f64_to_u32<<<nb, 256, 0, ctx->stream>>>(dev_buf + (size_t)N_F64 * stride, ctx->u32[0] + o, n);
        LAUNCH_CHECK();
        if (ctx->solid_alloc) {  // fields 17..28: s00..s22, s000..s220; field 29: cs
            for (int k = 0; k < 12; k++)
                CU(cudaMemcpyAsync(ctx->f64s[k] + o, dev_buf + (size_t)(B200SPH_MIGRATE_FIELDS + k) * stride, 8 * (size_t)n, cudaMemcpyDeviceToDevice, ctx->stream));
            k_f64_to_f32<<<nb, 256, 0, ctx->stream>>>(dev_buf + (size_t)(B200SPH_MIGRATE_FIELDS + 12) * stride, ctx->f32[B200SPH_CS - N_F64] + o, n);
            LAUNCH_CHECK();
        }
    }
    // tag = Remote (1) for ghosts
    k_fill_u32<<<nb, 256, 0, ctx->stream>>>(ctx->u32[1] + o, n, as_real ? 0u : 1u);
    LAUNCH_CHECK();
    CU(cudaMemsetAsync(ctx->u32[2] + o, 0, 4 * (size_t)n, ctx->stream));
    ai.n += n;
    if (as_real) ai.n_real += n;
    ctx->ptype_dirty = true;
    ctx->grid_valid = false, ctx->packed_valid = false;
    ctx->topo_dirty = true;
    ctx->h_dirty = ctx->uni_dirty = true;
    ctx->domain_valid = false;
    ctx->state_packed = false;
    return 0;
}

int b200sph_halo_pack_selected(b200sph_ctx *ctx, int arr, int slot, double *dev_buf, int64_t cap, int64_t *count)
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if ((rc = eos_flush(ctx))) return rc;
    if (arr < 0 || arr >= ctx->narr || slot < 0 || slot > 1) return set_err(ctx, "halo_pack_selected: bad array / slot");
    const int64_t n = ctx->halo_cnt[arr][slot];
    *count = n;
    if (n > cap) return set_err(ctx, "halo_pack_selected: buffer too small");
    if (n == 0) return 0;
    if (halo_nf(ctx) == B200SPH_HALO_FIELDS) k_halo_gather_idx<B200SPH_HALO_FIELDS><<<(unsigned)cdiv(n, 256), 256, 0, ctx->stream>>>(halo_ptrs(ctx), ctx->arr[arr].off, ctx->halo_idx[arr][slot], n, dev_buf);
    else k_halo_gather_idx<B200SPH_HALO_FIELDS_SOLID><<<(unsigned)cdiv(n, 256), 256, 0, ctx->stream>>>(halo_ptrs(ctx), ctx->arr[arr].off, ctx->halo_idx[arr][slot], n, dev_buf);
    LAUNCH_CHECK();
    return 0;
}

int b200sph_halo_overwrite(b200sph_ctx *ctx, int arr, int64_t ghost_first, const double *dev_buf, int64_t stride, int64_t n)
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if (arr < 0 || arr >= ctx->narr) return set_err(ctx, "halo_overwrite: bad array %d", arr);
    const ArrayInfo &ai = ctx->arr[arr];
    if (ghost_first < 0 || n < 0 || ai.n_real + ghost_first + n > ai.n)
        return set_err(ctx, "halo_overwrite: ghosts [%lld, %lld) outside the %lld ghosts of '%s'", (long long)ghost_first, (long long)(ghost_first + n), (long long)(ai.n - ai.n_real), ai.name.c_str());
    if (n == 0) return 0;
    const int64_t o = ai.off + ai.n_real + ghost_first;
    if (halo_nf(ctx) == B200SPH_HALO_FIELDS) k_halo_scatter<B200SPH_HALO_FIELDS><<<(unsigned)cdiv(n, 256), 256, 0, ctx->stream>>>(halo_ptrs(ctx), o, dev_buf, stride, n);
    else k_halo_scatter<B200SPH_HALO_FIELDS_SOLID><<<(unsigned)cdiv(n, 256), 256, 0, ctx->stream>>>(halo_ptrs(ctx), o, dev_buf, stride, n);
    LAUNCH_CHECK();
    // values moved, the particle set did not: a light nnps_update is enough
    ctx->grid_valid = false, ctx->packed_valid = false;
    ctx->state_packed = false;
    return 0;
}

int b200sph_nnps_drift(b200sph_ctx *ctx, double out[2])
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    out[0] = -1.0;
    out[1] = ctx->S_abs;
    if (ctx->force_kernel != 0 || !ctx->lists_valid || ctx->topo_dirty) return 0;  // no reusable build
    if (retire_build(ctx)) return 0;
    if (ctx->n_sorted <= 0) { out[0] = 0.0; return 0; }
    if (!(ctx->packed_valid && ctx->drift_measured)) {
        CU(cudaMemsetAsync(ctx->red_u32, 0, 2 * sizeof(unsigned), ctx->stream));
        k_pack_pos_light<<<(unsigned)cdiv(ctx->n_sorted, 256), 256, 0, ctx->stream>>>(
            ctx->f64[B200SPH_X], ctx->f64[B200SPH_Y], ctx->f64[B200SPH_Z], ctx->f64[B200SPH_H], ctx->perm, ctx->skey,
            ctx->n_sorted, ctx->G, ctx->A0, ctx->A, ctx->AB, ctx->R, ctx->red_u32);
        LAUNCH_CHECK();
    }
    CU(cudaMemcpyAsync(ctx->red_u32_host, ctx->red_u32, 2 * sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    float d2, dh;
    memcpy(&d2, &ctx->red_u32_host[0], 4);
    memcpy(&dh, &ctx->red_u32_host[1], 4);
    out[0] = 2.0 * std::sqrt((double)d2) + ctx->radius_scale * (double)dh;
    return 0;
}

int b200sph_halo_pack_selected_all(b200sph_ctx *ctx, int slot, double *dev_buf, int64_t cap_doubles, int64_t *ndoubles)
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if ((rc = eos_flush(ctx))) return rc;
    if (slot < 0 || slot > 1) return set_err(ctx, "halo_pack_selected_all: bad slot");
    HaloAllArgs A;
    A.narr = ctx->narr;
    A.prefix[0] = 0;
    for (int a = 0; a < ctx->narr; a++) {
        A.prefix[a + 1] = A.prefix[a] + ctx->halo_cnt[a][slot];
        A.off[a] = ctx->arr[a].off;
        A.idx[a] = ctx->halo_idx[a][slot];
    }
    const int64_t tot = A.prefix[ctx->narr];
    *ndoubles = tot * halo_nf(ctx);
    if (*ndoubles > cap_doubles) return set_err(ctx, "halo_pack_selected_all: buffer too small");
    if (tot == 0) return 0;
    if (halo_nf(ctx) == B200SPH_HALO_FIELDS) k_halo_gather_all<B200SPH_HALO_FIELDS><<<(unsigned)cdiv(tot, 256), 256, 0, ctx->stream>>>(halo_ptrs(ctx), A, dev_buf);
    else k_halo_gather_all<B200SPH_HALO_FIELDS_SOLID><<<(unsigned)cdiv(tot, 256), 256, 0, ctx->stream>>>(halo_ptrs(ctx), A, dev_buf);
    LAUNCH_CHECK();
    return 0;
}

int b200sph_halo_overwrite_all(b200sph_ctx *ctx, const int64_t *ghost_first, const int64_t *counts, const double *dev_buf)
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    HaloAllArgs A;
    A.narr = ctx->narr;
    A.prefix[0] = 0;
    for (int a = 0; a < ctx->narr; a++) {
        const ArrayInfo &ai = ctx->arr[a];
        if (ghost_first[a] < 0 || counts[a] < 0 || ai.n_real + ghost_first[a] + counts[a] > ai.n)
            return set_err(ctx, "halo_overwrite_all: ghosts [%lld, %lld) outside the %lld ghosts of '%s'", (long long)ghost_first[a],
                           (long long)(ghost_first[a] + counts[a]), (long long)(ai.n - ai.n_real), ai.name.c_str());
        A.prefix[a + 1] = A.prefix[a] + counts[a];
        A.off[a] = ai.off + ai.n_real + ghost_first[a];
        A.idx[a] = nullptr;
    }
    const int64_t tot = A.prefix[ctx->narr];
    if (tot == 0) return 0;
    // with a reusable build whose packed positions are current (nnps_drift_device just
    // ran) only the ghosts moved: refresh their packed records here and keep the flag
    const bool repack = ctx->packed_valid && ctx->lists_valid && !ctx->topo_dirty && ctx->force_kernel == 0 && ctx->n_sorted > 0;
    RepackArgs R;
    R.rank = repack ? ctx->rank : nullptr;
    R.skey = ctx->skey;
    R.A = ctx->A;
    R.AB = ctx->AB;
    R.G = ctx->G;
    if (halo_nf(ctx) == B200SPH_HALO_FIELDS) k_halo_scatter_all<B200SPH_HALO_FIELDS><<<(unsigned)cdiv(tot, 256), 256, 0, ctx->stream>>>(halo_ptrs(ctx), A, dev_buf, R);
    else k_halo_scatter_all<B200SPH_HALO_FIELDS_SOLID><<<(unsigned)cdiv(tot, 256), 256, 0, ctx->stream>>>(halo_ptrs(ctx), A, dev_buf, R);
    LAUNCH_CHECK();
    ctx->grid_valid = false;
    ctx->packed_valid = repack;
    ctx->state_packed = false;
    return 0;
}

// ---- peer memory (same node, NVLink): staging buffers a neighbour rank writes into ----
int b200sph_ipc_alloc(b200sph_ctx *ctx, int64_t bytes, void **dev_ptr, void *handle64)
{
    CU(cudaSetDevice(ctx->device));
    void *p = nullptr;
    CU(cudaMalloc(&p, (size_t)std::max<int64_t>(bytes, 256)));
    CU(cudaMemset(p, 0, (size_t)std::max<int64_t>(bytes, 256)));
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) {
        cudaFree(p);
        return set_err(ctx, "cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    memcpy(handle64, &h, 64);
    *dev_ptr = p;
    return 0;
}

int b200sph_ipc_open(b200sph_ctx *ctx, const void *handle64, void **dev_ptr)
{
    CU(cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    cudaError_t e = cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return set_err(ctx, "cudaIpcOpenMemHandle failed: %s", cudaGetErrorString(e));
    return 0;
}

int b200sph_ipc_close(b200sph_ctx *ctx, void *dev_ptr, int owner)
{
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->stream));
    if (owner) CU(cudaFree(dev_ptr));
    else CU(cudaIpcCloseMemHandle(dev_ptr));
    return 0;
}

int b200sph_nnps_drift_device(b200sph_ctx *ctx, double *dev_ratio)
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if (ctx->force_kernel != 0 || !ctx->lists_valid || ctx->topo_dirty) return 1;  // no reusable build
    if (retire_build(ctx)) return 1;
    if (ctx->n_sorted <= 0) {
        CU(cudaMemsetAsync(dev_ratio, 0, sizeof(double), ctx->stream));
        return 0;
    }
    if (!(ctx->packed_valid && ctx->drift_measured)) {   // (the fused stage kernel packs and measures)
        CU(cudaMemsetAsync(ctx->red_u32, 0, 2 * sizeof(unsigned), ctx->stream));
        k_pack_pos_light<<<(unsigned)cdiv(ctx->n_sorted, 256), 256, 0, ctx->stream>>>(
            ctx->f64[B200SPH_X], ctx->f64[B200SPH_Y], ctx->f64[B200SPH_Z], ctx->f64[B200SPH_H], ctx->perm, ctx->skey,
            ctx->n_sorted, ctx->G, ctx->A0, ctx->A, ctx->AB, ctx->R, ctx->red_u32);
        LAUNCH_CHECK();
    }
    k_drift_ratio<<<1, 1, 0, ctx->stream>>>(ctx->red_u32, (float)ctx->radius_scale, (float)ctx->S_abs, dev_ratio);
    LAUNCH_CHECK();
    ctx->packed_valid = true;
    ctx->drift_measured = true;
    return 0;
}

int b200sph_nnps_keep_build(b200sph_ctx *ctx)
{
    if (ctx->force_kernel != 0 || !ctx->lists_valid || ctx->topo_dirty)
        return set_err(ctx, "nnps_keep_build: there is no reusable neighbour build");
    ctx->drift_ok = true;
    return 0;
}

// ---- peer protocol (include/b200sph.h "peer protocol") ---------------------------------
// peer_publish / peer_send / peer_recv only RECORD what the epoch carries; peer_reduce
// launches the outgoing half as one k_peer_push and peer_end the incoming half as one
// k_peer_pull (seven dependent launches on a busy GPU cost 0.1 ms per evaluation, the two
// merged ones a third of that: profiles/r02k_chain.md).
struct PeerPending {
    struct Dir { HaloAllArgs A; double *buf; unsigned long long *flag; long long tot; };
    Dir send[2], recv[2];
    int n_send = 0, n_recv = 0;
    int have_build = 0, with_dt = 0;
    bool publish = false;
    GhostPackArgs pack;
};
static void free_peer_pending(b200sph_ctx *ctx)
{
    delete ctx->pend;
    ctx->pend = nullptr;
}
static int peer_streams(b200sph_ctx *ctx)
{
    if (ctx->comm_stream) return 0;
    int lo = 0, hi = 0;
    CU(cudaDeviceGetStreamPriorityRange(&lo, &hi));   // hi = the numerically lowest = highest priority
    CU(cudaStreamCreateWithPriority(&ctx->comm_stream, cudaStreamNonBlocking, hi));
    CU(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
    CU(cudaStreamCreateWithPriority(&ctx->red_stream, cudaStreamNonBlocking, hi));
    CU(cudaEventCreateWithFlags(&ctx->ev_pushed, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&ctx->ev_red, cudaEventDisableTiming));
    CU(cudaEventRecord(ctx->ev_red, ctx->red_stream));
    ctx->pend = new PeerPending();
    return 0;
}

int b200sph_peer_init(b200sph_ctx *ctx, int rank, int world, void *handle64)
{
    CU(cudaSetDevice(ctx->device));
    if (world < 1 || world > B200SPH_MAX_RANKS || rank < 0 || rank >= world)
        return set_err(ctx, "peer_init: rank %d of %d (at most %d ranks)", rank, world, B200SPH_MAX_RANKS);
    if (ctx->peer_box) return set_err(ctx, "peer_init: already initialised");
    int rc = peer_streams(ctx);
    if (rc) return rc;
    const size_t box_bytes = std::max<size_t>(sizeof(PeerBox), 4096);
    CU(cudaMalloc((void **)&ctx->peer_box, box_bytes));
    CU(cudaMemset(ctx->peer_box, 0, box_bytes));
    CU(cudaMalloc((void **)&ctx->peer_done, 2 * sizeof(unsigned)));
    CU(cudaMemset(ctx->peer_done, 0, 2 * sizeof(unsigned)));
    CU(cudaMalloc((void **)&ctx->peer_dec_dev, sizeof(double)));
    CU(cudaHostAlloc((void **)&ctx->peer_dec_host, sizeof(PeerDecision), cudaHostAllocMapped));
    memset(ctx->peer_dec_host, 0, sizeof(PeerDecision));
    CU(cudaHostGetDevicePointer((void **)&ctx->peer_dec_hostdev, ctx->peer_dec_host, 0));
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, ctx->peer_box);
    if (e != cudaSuccess) return set_err(ctx, "cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
    memcpy(handle64, &h, 64);
    ctx->peer_rank = rank;
    ctx->peer_world = world;
    ctx->peer_boxes[rank] = ctx->peer_box;
    return 0;
}

int b200sph_peer_connect(b200sph_ctx *ctx, const void *handles)
{
    CU(cudaSetDevice(ctx->device));
    if (!ctx->peer_box) return set_err(ctx, "peer_connect: call peer_init first");
    if (ctx->peer_connected) return 0;
    for (int r = 0; r < ctx->peer_world; r++) {
        if (r == ctx->peer_rank) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, (const char *)handles + 64 * (size_t)r, 64);
        void *p = nullptr;
        cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) return set_err(ctx, "peer_connect: cudaIpcOpenMemHandle(rank %d) failed: %s", r, cudaGetErrorString(e));
        ctx->peer_boxes[r] = (PeerBox *)p;
    }
    ctx->peer_connected = true;
    return 0;
}

static PeerPtrs peer_ptrs(const b200sph_ctx *ctx)
{
    PeerPtrs R;
    for (int r = 0; r < B200SPH_MAX_RANKS; r++) R.box[r] = ctx->peer_boxes[r];
    return R;
}

int b200sph_peer_begin(b200sph_ctx *ctx)
{
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if (!ctx->peer_connected) return set_err(ctx, "peer_begin: the mailboxes are not connected");
    if ((rc = eos_flush(ctx))) return rc;
    int no_build = 0;
    if (ctx->force_kernel != 0 || !ctx->lists_valid || ctx->topo_dirty) no_build = 1;
    else if (retire_build(ctx)) no_build = 1;
    if (!no_build && ctx->n_sorted > 0 && !(ctx->packed_valid && ctx->drift_measured)) {
        CU(cudaMemsetAsync(ctx->red_u32, 0, 2 * sizeof(unsigned), ctx->stream));
        k_pack_pos_light<<<(unsigned)cdiv(ctx->n_sorted, 256), 256, 0, ctx->stream>>>(
            ctx->f64[B200SPH_X], ctx->f64[B200SPH_Y], ctx->f64[B200SPH_Z], ctx->f64[B200SPH_H], ctx->perm, ctx->skey,
            ctx->n_sorted, ctx->G, ctx->A0, ctx->A, ctx->AB, ctx->R, ctx->red_u32);
        LAUNCH_CHECK();
    }
    if (!no_build) ctx->packed_valid = true, ctx->drift_measured = true;
    ctx->peer_epoch++;
    CU(cudaEventRecord(ctx->ev_fork, ctx->stream));
    CU(cudaStreamWaitEvent(ctx->comm_stream, ctx->ev_fork, 0));
    if (ctx->profiling) {
        for (cudaEvent_t *e : {&ctx->halo_ev_fork, &ctx->halo_ev_chain, &ctx->halo_ev_sent, &ctx->halo_ev_reduced})
            if (!*e) {
                if (!ctx->ev_pool.empty()) { *e = ctx->ev_pool.back(); ctx->ev_pool.pop_back(); }
                else CU(cudaEventCreate(e));
            }
        CU(cudaEventRecord(ctx->halo_ev_fork, ctx->stream));
    }
    return no_build;
}

int b200sph_peer_publish(b200sph_ctx *ctx, int have_build, int with_dt)
{
    CU(cudaSetDevice(ctx->device));
    if (!ctx->peer_connected) return set_err(ctx, "peer_publish: the mailboxes are not connected");
    if (with_dt && !ctx->tc) return set_err(ctx, "peer_publish: no time-control block");
    ctx->pend->publish = true;
    ctx->pend->have_build = have_build && ctx->n_sorted > 0 ? 1 : (have_build ? 2 : 0);
    ctx->pend->with_dt = with_dt;
    ctx->pend->n_send = ctx->pend->n_recv = 0;
    return 0;
}

int b200sph_peer_send(b200sph_ctx *ctx, int slot, int nb_rank, int side, double *remote_staging, int64_t cap_doubles)
{
    CU(cudaSetDevice(ctx->device));
    if (!ctx->peer_connected) return set_err(ctx, "peer_send: the mailboxes are not connected");
    if (slot < -1 || slot > 1 || side < 0 || side > 1 || nb_rank < 0 || nb_rank >= ctx->peer_world || nb_rank == ctx->peer_rank)
        return set_err(ctx, "peer_send: bad slot / side / neighbour");
    HaloAllArgs A;
    A.narr = ctx->narr;
    A.prefix[0] = 0;
    for (int a = 0; a < ctx->narr; a++) {
        // slot -1: the flag alone (this rank has no reusable build: the neighbour must not wait)
        A.prefix[a + 1] = A.prefix[a] + (slot < 0 ? 0 : ctx->halo_cnt[a][slot]);
        A.off[a] = ctx->arr[a].off;
        A.idx[a] = slot < 0 ? nullptr : ctx->halo_idx[a][slot];
    }
    const int64_t tot = A.prefix[ctx->narr];
    if (tot * halo_nf(ctx) > cap_doubles) return set_err(ctx, "peer_send: staging buffer too small");
    if (!ctx->pend->publish) return set_err(ctx, "peer_send: peer_publish opens the outgoing half of an epoch");
    if (ctx->pend->n_send >= 2) return set_err(ctx, "peer_send: a slab has two neighbours");
    PeerPending::Dir &D = ctx->pend->send[ctx->pend->n_send++];
    D.A = A;
    D.buf = remote_staging;
    D.flag = &ctx->peer_boxes[nb_rank]->data_seq[ctx->peer_epoch & 1][side];
    D.tot = tot;
    return 0;
}

static void peer_dir(PeerDir &d, const PeerPending::Dir &p, unsigned *done)
{
    d.A = p.A;
    d.buf = p.buf;
    d.flag = p.flag;
    d.done = done;
    d.nblocks = (unsigned)cdiv(p.tot, PEER_NT);
}

// the outgoing half of the epoch: scalars + both messages, one launch
static int peer_push(b200sph_ctx *ctx)
{
    PeerPending &Q = *ctx->pend;
    if (!Q.publish) return set_err(ctx, "peer_reduce: nothing was published for this epoch");
    Q.publish = false;
    PeerPushArgs X;
    memset(&X, 0, sizeof(X));
    X.ndir = Q.n_send;
    for (int d = 0; d < Q.n_send; d++) peer_dir(X.d[d], Q.send[d], ctx->peer_done + d);
    X.rank = ctx->peer_rank;
    X.world = ctx->peer_world;
    X.have_build = Q.have_build;
    X.with_dt = Q.with_dt;
    X.kr = (float)ctx->radius_scale;
    X.S = (float)ctx->S_abs;
    X.red_u32 = ctx->red_u32;
    X.tc = ctx->tc;
    const unsigned blocks = 1 + X.d[0].nblocks + X.d[1].nblocks;
    if (halo_nf(ctx) == B200SPH_HALO_FIELDS)
        k_peer_push<B200SPH_HALO_FIELDS><<<blocks, PEER_NT, 0, ctx->comm_stream>>>(halo_ptrs(ctx), X, peer_ptrs(ctx), ctx->peer_epoch);
    else
        k_peer_push<B200SPH_HALO_FIELDS_SOLID><<<blocks, PEER_NT, 0, ctx->comm_stream>>>(halo_ptrs(ctx), X, peer_ptrs(ctx), ctx->peer_epoch);
    LAUNCH_CHECK();
    return 0;
}

// the incoming half: both neighbours' messages scattered (and packed) by one launch
static int peer_pull(b200sph_ctx *ctx)
{
    PeerPending &Q = *ctx->pend;
    if (Q.n_recv == 0) return 0;
    PeerPullArgs X;
    memset(&X, 0, sizeof(X));
    X.ndir = Q.n_recv;
    for (int d = 0; d < Q.n_recv; d++) peer_dir(X.d[d], Q.recv[d], nullptr);
    Q.n_recv = 0;
    const unsigned blocks = X.d[0].nblocks + X.d[1].nblocks;
    if (halo_nf(ctx) == B200SPH_HALO_FIELDS)
        k_peer_pull<B200SPH_HALO_FIELDS><<<blocks, PEER_NT, 0, ctx->comm_stream>>>(halo_ptrs(ctx), X, Q.pack, ctx->peer_epoch, ctx->peer_dec_hostdev);
    else
        k_peer_pull<B200SPH_HALO_FIELDS_SOLID><<<blocks, PEER_NT, 0, ctx->comm_stream>>>(halo_ptrs(ctx), X, Q.pack, ctx->peer_epoch, ctx->peer_dec_hostdev);
    LAUNCH_CHECK();
    return 0;
}

int b200sph_peer_reduce(b200sph_ctx *ctx, int with_dt)
{
    CU(cudaSetDevice(ctx->device));
    if (!ctx->peer_connected) return set_err(ctx, "peer_reduce: the mailboxes are not connected");
    int rc = peer_push(ctx);
    if (rc) return rc;
    if (ctx->profiling && ctx->halo_ev_sent) CU(cudaEventRecord(ctx->halo_ev_sent, ctx->comm_stream));
    CU(cudaEventRecord(ctx->ev_pushed, ctx->comm_stream));
    CU(cudaStreamWaitEvent(ctx->red_stream, ctx->ev_pushed, 0));   // my scalars are out before I wait for the others'
    k_peer_reduce<<<1, 32, 0, ctx->red_stream>>>(ctx->peer_box, ctx->peer_world, ctx->peer_epoch, 0, ctx->peer_dec_dev, ctx->peer_dec_hostdev,
                                                  ctx->tc, with_dt && ctx->tc ? 1 : 0);
    LAUNCH_CHECK();
    if (ctx->profiling && ctx->halo_ev_reduced) CU(cudaEventRecord(ctx->halo_ev_reduced, ctx->red_stream));
    CU(cudaEventRecord(ctx->ev_red, ctx->red_stream));
    return 0;
}

int b200sph_peer_recv(b200sph_ctx *ctx, int side, const int64_t *ghost_first, const int64_t *counts, const double *local_staging)
{
    CU(cudaSetDevice(ctx->device));
    if (!ctx->peer_connected) return set_err(ctx, "peer_recv: the mailboxes are not connected");
    if (side < 0 || side > 1) return set_err(ctx, "peer_recv: bad side");
    HaloAllArgs A;
    A.narr = ctx->narr;
    A.prefix[0] = 0;
    for (int a = 0; a < ctx->narr; a++) {
        const ArrayInfo &ai = ctx->arr[a];
        if (ghost_first[a] < 0 || counts[a] < 0 || ai.n_real + ghost_first[a] + counts[a] > ai.n)
            return set_err(ctx, "peer_recv: ghosts [%lld, %lld) outside the %lld ghosts of '%s'", (long long)ghost_first[a],
                           (long long)(ghost_first[a] + counts[a]), (long long)(ai.n - ai.n_real), ai.name.c_str());
        A.prefix[a + 1] = A.prefix[a] + counts[a];
        A.off[a] = ai.off + ai.n_real + ghost_first[a];
        A.idx[a] = nullptr;
    }
    const int64_t tot = A.prefix[ctx->narr];
    if (tot == 0) return 0;
    int rc = refresh_ptype(ctx);
    if (rc) return rc;
    const bool repack = ctx->packed_valid && ctx->lists_valid && !ctx->topo_dirty && ctx->force_kernel == 0 && ctx->n_sorted > 0;
    // the ghosts' state records too when the real particles' are in place (fused stage kernel)
    const bool records = repack && ctx->state_packed && halo_nf(ctx) == B200SPH_HALO_FIELDS;
    GhostPackArgs R;
    memset(&R, 0, sizeof(R));
    R.rank = repack ? ctx->rank : nullptr;
    R.skey = ctx->skey;
    R.A = ctx->A; R.AB = ctx->AB;
    R.C = records ? ctx->C : nullptr;
    R.G = ctx->G;
    R.ptype = ctx->ptype;
    R.p = ctx->f32[B200SPH_P - N_F64]; R.cs = ctx->f32[B200SPH_CS - N_F64];
    R.eos_any = ctx->spec_records && ctx->eos_last_valid ? 1 : 0;
    R.E = ctx->eos_last;
    if (ctx->pend->n_recv >= 2) return set_err(ctx, "peer_recv: a slab has two neighbours");
    PeerPending::Dir &D = ctx->pend->recv[ctx->pend->n_recv++];
    D.A = A;
    D.buf = const_cast<double *>(local_staging);
    D.flag = &ctx->peer_box->data_seq[ctx->peer_epoch & 1][side];
    D.tot = tot;
    ctx->pend->pack = R;          // the same for both sides: it describes the receiver
    ctx->grid_valid = false;
    ctx->packed_valid = repack;
    if (!records) ctx->state_packed = false;
    return 0;
}

int b200sph_peer_commit_dt(b200sph_ctx *ctx, double prev_factor, double new_factor, int adaptive, int advance, int snapshot_slot)
{
    CU(cudaSetDevice(ctx->device));
    if (!ctx->comm_stream || !ctx->tc) return set_err(ctx, "peer_commit_dt: no epoch in flight / no time-control block");
    if (!(prev_factor > 0.0) || !(new_factor > 0.0)) return set_err(ctx, "peer_commit_dt: damping factors must be positive");
    if (snapshot_slot > 1) return set_err(ctx, "peer_commit_dt: snapshot slot must be 0 or 1");
    // behind the agreement (k_peer_reduce left the MIN in tc[2]), on its stream
    k_dt_commit<<<1, 1, 0, ctx->red_stream>>>(ctx->tc, prev_factor, new_factor, 1, adaptive, advance, ctx->t_final, ctx->t_eps);
    LAUNCH_CHECK();
    if (snapshot_slot >= 0) {
        CU(cudaMemcpyAsync(ctx->tc_host + 2 * snapshot_slot, ctx->tc, 2 * sizeof(double), cudaMemcpyDeviceToHost, ctx->red_stream));
        CU(cudaEventRecord(ctx->tc_evt[snapshot_slot], ctx->red_stream));
    }
    CU(cudaEventRecord(ctx->ev_red, ctx->red_stream));
    return 0;
}

int b200sph_peer_end(b200sph_ctx *ctx)
{
    CU(cudaSetDevice(ctx->device));
    if (!ctx->comm_stream) return set_err(ctx, "peer_end: no epoch in flight");
    if (ctx->pend->publish) return set_err(ctx, "peer_end: peer_reduce closes the outgoing half of an epoch");
    if (int rc = peer_pull(ctx)) return rc;
    if (ctx->profiling && ctx->halo_ev_chain) CU(cudaEventRecord(ctx->halo_ev_chain, ctx->comm_stream));
    CU(cudaEventRecord(ctx->ev_join, ctx->comm_stream));
    ctx->comm_pending = true;
    return 0;
}

int b200sph_peer_decision(b200sph_ctx *ctx, double *ratio_max)
{
    if (!ctx->peer_dec_host) return set_err(ctx, "peer_decision: no peer protocol");
    volatile PeerDecision *d = ctx->peer_dec_host;
    const unsigned long long want = ctx->peer_epoch;
    // the kernel that writes it is on the communication stream and needs no help from the host
    for (long long spin = 0; d->seq != want; spin++) {
        if ((spin & 0xFFFF) == 0xFFFF) {
            // nothing enqueued can be stuck for half a minute unless a peer died
            cudaError_t e = cudaStreamQuery(ctx->red_stream);
            if (e != cudaSuccess && e != cudaErrorNotReady) return set_err(ctx, "peer_decision: %s", cudaGetErrorString(e));
            if (e == cudaSuccess && d->seq != want) return set_err(ctx, "peer_decision: epoch %llu was never decided", want);
        }
    }
    if (d->error == want) return set_err(ctx, "peer protocol: a rank did not answer within %.0f s (epoch %llu)", PEER_TIMEOUT_NS * 1e-9, want);
    *ratio_max = d->value;
    if (d->value <= 1.0) {   // the skin controller's view of the build: the all-rank maximum (the same on every rank)
        ctx->drift_hist[0] = ctx->drift_hist[1];
        ctx->drift_hist[1] = d->value;
    }
    return 0;
}

int b200sph_peer_allreduce_dt(b200sph_ctx *ctx)
{
    CU(cudaSetDevice(ctx->device));
    if (!ctx->peer_connected) return set_err(ctx, "peer_allreduce_dt: the mailboxes are not connected");
    if (!ctx->tc) return set_err(ctx, "peer_allreduce_dt: no time-control block");
    ctx->peer_dt_epoch++;
    k_peer_publish<<<1, 32, 0, ctx->stream>>>(peer_ptrs(ctx), ctx->peer_rank, ctx->peer_world, ctx->peer_dt_epoch, 1, ctx->red_u32, 0.f, 0.f, 0, ctx->tc, 1);
    LAUNCH_CHECK();
    k_peer_reduce<<<1, 32, 0, ctx->stream>>>(ctx->peer_box, ctx->peer_world, ctx->peer_dt_epoch, 1, nullptr, nullptr, ctx->tc, 1);
    LAUNCH_CHECK();
    return 0;
}

int b200sph_drop_ghosts(b200sph_ctx *ctx, int arr)
{
    if (arr < 0 || arr >= ctx->narr) return set_err(ctx, "drop_ghosts: bad array %d", arr);
    if (ctx->arr[arr].n != ctx->arr[arr].n_real) {
        ctx->arr[arr].n = ctx->arr[arr].n_real;
        ctx->ptype_dirty = true;
        ctx->grid_valid = false, ctx->packed_valid = false;
        ctx->topo_dirty = true;
        ctx->h_dirty = ctx->uni_dirty = true;
        ctx->state_packed = false;
    }
    return 0;
}

// Per-column particle counts for the slab re-cut.  Every thread walks COLUMN_RUN
// consecutive particles and merges equal bins before the atomic: particles are stored
// in cell order, so a run mostly stays in one column and the counters see ~n/32 atomics.
#define COLUMN_RUN 32
__global__ void k_column_counts(const double *__restrict__ x, long long off, long long n, double x0, double inv_w, int nbins,
                                unsigned long long *__restrict__ counts)
{
    const long long first = (blockIdx.x * (long long)blockDim.x + threadIdx.x) * COLUMN_RUN;
    if (first >= n) return;
    const long long last = first + COLUMN_RUN < n ? first + COLUMN_RUN : n;
    int cur = -1;
    unsigned long long run = 0;
    for (long long i = first; i < last; i++) {
        int b = (int)floor((x[off + i] - x0) * inv_w);
        b = b < 0 ? 0 : (b >= nbins ? nbins - 1 : b);
        if (b != cur) {
            if (run) atomicAdd(&counts[cur], run);
            cur = b, run = 0;
        }
        run++;
    }
    if (run) atomicAdd(&counts[cur], run);
}

int b200sph_column_counts(b200sph_ctx *ctx, int arr, double x0, double inv_width, int nbins, unsigned long long *dev_counts)
{
    if (int rcc = require_confirmed(ctx, "column_counts")) return rcc;
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if (arr < 0 || arr >= ctx->narr) return set_err(ctx, "column_counts: bad array %d", arr);
    if (nbins < 1 || !(inv_width > 0.0) || !dev_counts) return set_err(ctx, "column_counts: bad bins");
    const ArrayInfo &ai = ctx->arr[arr];
    if (ai.n_real == 0) return 0;
    const unsigned nb = (unsigned)cdiv(cdiv(ai.n_real, COLUMN_RUN), 256);
    k_column_counts<<<nb, 256, 0, ctx->stream>>>(ctx->f64[B200SPH_X], ai.off, ai.n_real, x0, inv_width, nbins, dev_counts);
    LAUNCH_CHECK();
    return 0;
}

int b200sph_migrate_out(b200sph_ctx *ctx, int arr, double lo, double hi, double *dev_buf, int64_t cap, int64_t count[2])
{
    if (int rcc = require_confirmed(ctx, "migrate_out")) return rcc;
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_pool(ctx);
    if (rc) return rc;
    if ((rc = eos_flush(ctx))) return rc;
    if (arr < 0 || arr >= ctx->narr) return set_err(ctx, "migrate_out: bad array %d", arr);
    ArrayInfo &ai = ctx->arr[arr];
    if (ai.n != ai.n_real) return set_err(ctx, "migrate_out: drop the ghosts of '%s' first", ai.name.c_str());
    const int64_t n = ai.n_real, off = ai.off;
    count[0] = count[1] = 0;
    if (n == 0) return 0;
    const unsigned nb = (unsigned)cdiv(n + 1, 256);
    const int mnf = migrate_nf(ctx);
    int64_t base = 0;  // doubles written so far
    for (int side = 0; side < 2; side++) {
        k_flag_range<<<nb, 256, 0, ctx->stream>>>(ctx->f64[B200SPH_X], off, n, lo, hi, side == 0 ? 1 : 2, ctx->flag_a);
        LAUNCH_CHECK();
        if ((rc = device_scan(ctx, ctx->flag_a, ctx->flag_b, n + 1))) return rc;
        uint32_t tot = 0;
        CU(cudaMemcpyAsync(&tot, ctx->flag_b + n, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CU(cudaStreamSynchronize(ctx->stream));
        count[side] = tot;
        if (base + (int64_t)tot * mnf > cap * mnf) return set_err(ctx, "migrate_out: buffer too small");
        if (tot) {
            for (int k = 0; k < N_F64; k++) {
                k_gather_f64<<<nb, 256, 0, ctx->stream>>>(ctx->f64[k], off, n, ctx->flag_a, ctx->flag_b, dev_buf, base + (long long)k * tot);
                LAUNCH_CHECK();
            }
            k_gather_u32_as_f64<<<nb, 256, 0, ctx->stream>>>(ctx->u32[0], off, n, ctx->flag_a, ctx->flag_b, dev_buf, base + (long long)N_F64 * tot);
            LAUNCH_CHECK();
            if (ctx->solid_alloc) {
                for (int k = 0; k < 12; k++) {
                    k_gather_f64<<<nb, 256, 0, ctx->stream>>>(ctx->f64s[k], off, n, ctx->flag_a, ctx->flag_b, dev_buf, base + (long long)(B200SPH_MIGRATE_FIELDS + k) * tot);
                    LAUNCH_CHECK();
                }
                k_gather_f32_as_f64<<<nb, 256, 0, ctx->stream>>>(ctx->f32[B200SPH_CS - N_F64], off, n, ctx->flag_a, ctx->flag_b, dev_buf, base + (long long)(B200SPH_MIGRATE_FIELDS + 12) * tot);
                LAUNCH_CHECK();
            }
        }
        base += (int64_t)tot * mnf;
    }
    if (count[0] + count[1] == 0) return 0;
    // stable compaction of the keepers, property by property, through the staging buffer
    k_flag_range<<<nb, 256, 0, ctx->stream>>>(ctx->f64[B200SPH_X], off, n, lo, hi, 3, ctx->flag_a);
    LAUNCH_CHECK();
    if ((rc = device_scan(ctx, ctx->flag_a, ctx->flag_b, n + 1))) return rc;
    const int64_t keep = n - count[0] - count[1];
    if ((rc = ensure_stage(ctx, n))) return rc;
    // x is the selection key: compact it last
    for (int k = N_F64 - 1; k >= 0; k--) {
        k_gather_f64<<<nb, 256, 0, ctx->stream>>>(ctx->f64[k], off, n, ctx->flag_a, ctx->flag_b, ctx->stage_buf, 0);
        LAUNCH_CHECK();
        if (keep) CU(cudaMemcpyAsync(ctx->f64[k] + off, ctx->stage_buf, 8 * (size_t)keep, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    for (int k = 0; k < N_U32; k++) {
        k_gather_u32<<<nb, 256, 0, ctx->stream>>>(ctx->u32[k], off, n, ctx->flag_a, ctx->flag_b, (uint32_t *)ctx->stage_buf);
        LAUNCH_CHECK();
        if (keep) CU(cudaMemcpyAsync(ctx->u32[k] + off, ctx->stage_buf, 4 * (size_t)keep, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    if (ctx->solid_alloc) {  // the keepers' stress state and cs move with them (the other fp32 fields are recomputed)
        for (int k = 0; k < 12; k++) {
            k_gather_f64<<<nb, 256, 0, ctx->stream>>>(ctx->f64s[k], off, n, ctx->flag_a, ctx->flag_b, ctx->stage_buf, 0);
            LAUNCH_CHECK();
            if (keep) CU(cudaMemcpyAsync(ctx->f64s[k] + off, ctx->stage_buf, 8 * (size_t)keep, cudaMemcpyDeviceToDevice, ctx->stream));
        }
        k_gather_u32<<<nb, 256, 0, ctx->stream>>>((const uint32_t *)ctx->f32[B200SPH_CS - N_F64], off, n, ctx->flag_a, ctx->flag_b, (uint32_t *)ctx->stage_buf);
        LAUNCH_CHECK();
        if (keep) CU(cudaMemcpyAsync(ctx->f32[B200SPH_CS - N_F64] + off, ctx->stage_buf, 4 * (size_t)keep, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    ai.n = ai.n_real = keep;
    ctx->ptype_dirty = true;
    ctx->grid_valid = false, ctx->packed_valid = false;
    ctx->topo_dirty = true;
    ctx->h_dirty = ctx->uni_dirty = true;
    ctx->domain_valid = false;
    ctx->state_packed = false;
    return 0;
}

int b200sph_get_stats(b200sph_ctx *ctx, b200sph_stats *out)
{
    if (!ctx->pending.empty()) {
        CU(cudaSetDevice(ctx->device));
        CU(cudaStreamSynchronize(ctx->stream));
        for (auto &pe : ctx->pending) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, pe.e0, pe.e1);
            if (pe.slot == 0) ctx->stats.ms_nnps += ms;
            else if (pe.slot == 1) ctx->stats.ms_pair += ms;
            else ctx->stats.ms_other += ms;
            ctx->ev_pool.push_back(pe.e0);
            ctx->ev_pool.push_back(pe.e1);
        }
        ctx->pending.clear();
    }
    if (!ctx->halo_pending.empty()) {
        CU(cudaSetDevice(ctx->device));
        CU(cudaStreamSynchronize(ctx->stream));
        if (ctx->comm_stream) CU(cudaStreamSynchronize(ctx->comm_stream));
        if (ctx->red_stream) CU(cudaStreamSynchronize(ctx->red_stream));
        for (auto &h : ctx->halo_pending) {
            float a = 0.f, b = 0.f;
            cudaEventElapsedTime(&a, h.fork, h.chain);
            cudaEventElapsedTime(&b, h.fork, h.end);
            ctx->stats.ms_halo_chain += a;
            ctx->stats.ms_pair_wall += b;
            if (h.sent && h.reduced) {
                float c = 0.f, d = 0.f;
                if (cudaEventElapsedTime(&c, h.fork, h.sent) == cudaSuccess) ctx->stats.ms_halo_sent += c;
                if (cudaEventElapsedTime(&d, h.fork, h.reduced) == cudaSuccess) ctx->stats.ms_halo_reduced += d;
                ctx->ev_pool.push_back(h.sent); ctx->ev_pool.push_back(h.reduced);
            }
            ctx->ev_pool.push_back(h.fork); ctx->ev_pool.push_back(h.chain); ctx->ev_pool.push_back(h.end);
        }
        ctx->halo_pending.clear();
    }
    ctx->stats.full_builds = ctx->n_full_builds;
    ctx->stats.light_updates = ctx->n_light_updates;
    ctx->stats.list_builds = ctx->n_list_builds;
    ctx->stats.list_entries_per_particle = ctx->capg;
    ctx->stats.deferred_failed = ctx->n_deferred_failed;
    ctx->stats.fused_stages = ctx->n_fused;
    ctx->stats.overlapped = ctx->n_overlapped;
    ctx->stats.proactive_builds = ctx->n_proactive;
    ctx->stats.chunks_interior = ctx->chunks_valid ? ctx->n_chunk_interior : 0;
    ctx->stats.chunks_boundary = ctx->chunks_valid ? ctx->n_chunk_boundary : 0;
    *out = ctx->stats;
    return 0;
}
int b200sph_get_pair_r32_launches(b200sph_ctx *ctx, int64_t *out)
{
    *out = ctx->n_pair_r32;
    return 0;
}

int b200sph_reset_stats(b200sph_ctx *ctx)
{
    ctx->n_pair_r32 = 0;
    b200sph_stats tmp;
    b200sph_get_stats(ctx, &tmp);  // drain pending events
    memset(&ctx->stats, 0, sizeof(ctx->stats));
    ctx->n_full_builds = ctx->n_light_updates = ctx->n_list_builds = ctx->n_deferred_failed = ctx->n_fused = ctx->n_overlapped = ctx->n_proactive = 0;
    return 0;
}
int b200sph_set_async_copies(b200sph_ctx *ctx, int on)
{
    ctx->async_copies = on != 0;
    if (!on) CU(cudaStreamSynchronize(ctx->stream));
    return 0;
}
int b200sph_set_profiling(b200sph_ctx *ctx, int on)
{
    ctx->profiling = on < 0 ? 0 : (on > 2 ? 1 : on);
    return 0;
}

}  // extern "C"
