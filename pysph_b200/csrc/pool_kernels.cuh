// pool_kernels.cuh -- elementwise / reduction kernels over the particle pool.
// Part of the single translation unit b200sph.cu (included there, in this order; not a
// stand-alone header).

// --------------------------------------------------------------------------
// elementwise / reduction kernels over the pool
// --------------------------------------------------------------------------
struct PoolLayout {
    int narr;
    long long off[B200SPH_MAX_ARRAYS], n[B200SPH_MAX_ARRAYS], n_real[B200SPH_MAX_ARRAYS];
};

__global__ void k_fill_ptype(uint8_t *ptype, long long pool_end, PoolLayout L)
{
    long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= pool_end) return;
    uint8_t t = PT_INVALID;
    for (int a = 0; a < L.narr; a++) {
        long long i = g - L.off[a];
        if (i >= 0 && i < L.n[a]) t = (uint8_t)(a | (i >= L.n_real[a] ? PT_GHOST : 0));
    }
    ptype[g] = t;
}

__global__ void k_red_init(long long *red)
{
    int i = threadIdx.x;
    if (i < 16) red[i] = (i & 1) ? d2o(-1e300) : d2o(1e300);  // even: min slots, odd: max slots
}

// slots: 0 xmin 1 xmax 2 ymin 3 ymax 4 zmin 5 zmax 6 hmin 7 hmax
__global__ void k_reduce_minmax(const double *__restrict__ x, const double *__restrict__ y,
                                const double *__restrict__ z, const double *__restrict__ h,
                                const uint8_t *__restrict__ ptype, long long pool_end,
                                int do_xyz, int do_h, long long *red)
{
    double mn[4] = {1e300, 1e300, 1e300, 1e300}, mx[4] = {-1e300, -1e300, -1e300, -1e300};
    for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < pool_end;
         g += (long long)gridDim.x * blockDim.x) {
        if (ptype[g] == PT_INVALID) continue;
        if (do_xyz) {
            double v = x[g]; mn[0] = fmin(mn[0], v); mx[0] = fmax(mx[0], v);
            v = y[g]; mn[1] = fmin(mn[1], v); mx[1] = fmax(mx[1], v);
            v = z[g]; mn[2] = fmin(mn[2], v); mx[2] = fmax(mx[2], v);
        }
        if (do_h) {
            double v = h[g]; mn[3] = fmin(mn[3], v); mx[3] = fmax(mx[3], v);
        }
    }
    for (int k = 0; k < 4; k++) {
        for (int o = 16; o > 0; o >>= 1) {
            mn[k] = fmin(mn[k], __shfl_xor_sync(0xffffffffu, mn[k], o));
            mx[k] = fmax(mx[k], __shfl_xor_sync(0xffffffffu, mx[k], o));
        }
    }
    if ((threadIdx.x & 31) == 0) {
        for (int k = 0; k < 4; k++) {
            if ((k < 3 && !do_xyz) || (k == 3 && !do_h)) continue;
            atomicMin(&red[2 * k], d2o(mn[k]));
            atomicMax(&red[2 * k + 1], d2o(mx[k]));
        }
    }
}

// slots: 9 max dt_cfl, 11 max dt_force (real particles), 12 min h (all)
__global__ void k_reduce_dt(const float *__restrict__ dt_cfl, const float *__restrict__ dt_force,
                            const double *__restrict__ h, const uint8_t *__restrict__ ptype,
                            long long pool_end, long long *red)
{
    double mc = -1e300, mf = -1e300, hm = 1e300;
    for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < pool_end;
         g += (long long)gridDim.x * blockDim.x) {
        uint8_t t = ptype[g];
        if (t == PT_INVALID) continue;
        hm = fmin(hm, h[g]);
        if (t & PT_GHOST) continue;
        mc = fmax(mc, (double)dt_cfl[g]);
        mf = fmax(mf, (double)dt_force[g]);
    }
    for (int o = 16; o > 0; o >>= 1) {
        mc = fmax(mc, __shfl_xor_sync(0xffffffffu, mc, o));
        mf = fmax(mf, __shfl_xor_sync(0xffffffffu, mf, o));
        hm = fmin(hm, __shfl_xor_sync(0xffffffffu, hm, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMax(&red[9], d2o(mc));
        atomicMax(&red[11], d2o(mf));
        atomicMin(&red[12], d2o(hm));
    }
}

// Integrator.compute_time_step (integrator.py:161-200) on the reduced factors: the local
// proposal cfl * dt_min, or 1e20 when no factor constrains it (solver.py:655-660)
__global__ void k_dt_propose(long long *__restrict__ red, double *__restrict__ tc, double cfl, int fixed_h)
{
    const double mc = o2d(red[9]), mf = o2d(red[11]);
    const double f_cfl = mc < -1e299 ? -1.0 : mc, f_force = mf < -1e299 ? -1.0 : mf;
    double hmin = fmin(1.0, o2d(red[12]));
    if (!fixed_h || tc[3] < 0.0) tc[3] = hmin;
    hmin = tc[3];
    const double inf = __longlong_as_double(0x7ff0000000000000LL);
    double dt_cfl = inf, dt_force = inf;
    if (f_cfl > 0.0) dt_cfl = hmin / f_cfl;
    if (f_force > 0.0) dt_force = sqrt(hmin / sqrt(f_force));
    const double dt_min = fmin(dt_cfl, dt_force);
    tc[2] = (dt_min <= 0.0 || isinf(dt_min)) ? 1e20 : cfl * dt_min;
    // re-arm the slots for the next reduction (the fused stage kernel adds to them directly)
    red[9] = d2o(-1e300); red[11] = d2o(-1e300); red[12] = d2o(1e300);
}
// Solver loop bookkeeping (solver.py:478-491, :647-688): t += dt; dt = damp(new dt)
// and the last step lands on the final time (solver.py:757-760, :771-773)
__global__ void k_dt_commit(double *__restrict__ tc, double prev_factor, double new_factor, int in_parallel, int adaptive, int advance,
                            double t_final, double t_eps)
{
    const double dt_old = tc[0];
    if (advance) tc[1] += dt_old;
    const double t = tc[1];
    if (fabs(t_final - t) < t_eps) return;  // reached the end: dt stays
    const double undamped = dt_old / prev_factor;
    double dt = undamped;
    if (adaptive) {
        dt = tc[2];
        if (!in_parallel && dt >= 1e20) dt = undamped;
    }
    dt *= new_factor;
    if (t + dt > t_final - t_eps) dt = t_final - t;
    tc[0] = dt;
}
// UpdateSmoothingLengthFerrari.loop wc/basic.py:458-463
__global__ void k_ferrari(double *__restrict__ h, const double *__restrict__ m,
                          const double *__restrict__ rho, long long lo, long long hi, double hdx,
                          double dim1)
{
    long long g = lo + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= hi) return;
    h[g] = hdx * pow(m[g] / rho[g], dim1);
}

struct StageArgs {
    double *x, *y, *z, *u, *v, *w, *rho;
    double *x0, *y0, *z0, *u0, *v0, *w0, *rho0;
    const float *au, *av, *aw, *ax, *ay, *az, *arho;
    const uint8_t *ptype;
    long long pool_end;
    int arr, which;
    double f;
};

// WCSPHStep.initialize / stage1 / stage2 integrator_step.py:51-91 (real particles only,
// integrator_cython.mako:97-111)
__device__ __forceinline__ void stage_body(const StageArgs &a);
__global__ void k_stage(StageArgs a) { stage_body(a); }
__global__ void k_stage_devdt(StageArgs a, const double *__restrict__ tc)
{
    const double dt = tc[0];
    a.f = a.which == 1 ? 0.5 * dt : dt;
    stage_body(a);
}
__device__ __forceinline__ void stage_body(const StageArgs &a)
{
    long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= a.pool_end) return;
    uint8_t t = a.ptype[g];
    if (t == PT_INVALID || (t & PT_GHOST)) return;
    if (a.arr >= 0 && (t & 7) != a.arr) return;
    if (a.which == 0) {
        a.x0[g] = a.x[g]; a.y0[g] = a.y[g]; a.z0[g] = a.z[g];
        a.u0[g] = a.u[g]; a.v0[g] = a.v[g]; a.w0[g] = a.w[g];
        a.rho0[g] = a.rho[g];
    } else {
        const double f = a.f;
        a.u[g] = a.u0[g] + f * (double)a.au[g];
        a.v[g] = a.v0[g] + f * (double)a.av[g];
        a.w[g] = a.w0[g] + f * (double)a.aw[g];
        a.x[g] = a.x0[g] + f * (double)a.ax[g];
        a.y[g] = a.y0[g] + f * (double)a.ay[g];
        a.z[g] = a.z0[g] + f * (double)a.az[g];
        a.rho[g] = a.rho0[g] + f * (double)a.arho[g];
    }
}

// ---------------------------------------------------------------------------
// The fused stage kernel of the WCSPH fast path (every array steps with WCSPHStep, the
// neighbour lists of the current build are reusable): in ONE pass over the pool, per real
// particle,
//   [initialize (integrator_step.py:51-61) when it was deferred to here]
//   stage1 / stage2 (integrator_step.py:63-91), fp64, bitwise what k_stage computes
//   the packed pair records of the NEXT evaluation at the particle's sorted slot:
//     {A, B} = (cell-relative position of the frozen build, h, u, v, w, m)   -- k_pack_pos_light
//     C      = (rho, p / rho^2, cs, type) with the equation-of-state calls of the LAST
//              evaluation applied to the record only (k_pack_state's arithmetic); the pool's
//              rho / p / cs are written when the evaluation really issues those calls
//   the drift of the build (max |x - x_build|^2, max (h - h_build)) into red_u32
//   [stage2: the adaptive-dt factors max dt_cfl, max dt_force, min h into red[9,11,12]]
// It replaces k_stage + k_stage(initialize) + k_pack_pos_light + k_pack_state (+ k_reduce_dt):
// five sweeps over the fp64 state become one.  Ghost particles are not stepped
// (integrator_cython.mako:97-111) and their records are refreshed by the halo scatter.
// ---------------------------------------------------------------------------
struct FusePackArgs {
    const double *h, *m;
    const float *p, *cs;             // pool values, used for arrays without a speculated EOS
    const uint32_t *rank, *key_of;   // pool index -> sorted slot / cell key of the current build
    const float4 *A0;                // packed positions at build time (sorted order)
    float4 *AB, *C;
    float4 *R;                       // the 32-byte source records (PairArgs.R)
    unsigned r32_cls;                // bit a: array a is source class 1
    GridDev G;
    unsigned *red_u32;
    const float *dt_cfl, *dt_force;
    long long *red;
    const double *tc;                // device-resident dt (tc[0]); null: StageArgs.f
    int do_init, reduce_dt, eos_any;
    EosTab E;
};

__global__ void __launch_bounds__(256, 5) k_stage_pack(const StageArgs a, const FusePackArgs q)
{
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    float d2 = 0.f, dh = 0.f;
    double mc = -1e300, mf = -1e300, hm = 1e300;
    const uint8_t t = g < a.pool_end ? a.ptype[g] : (uint8_t)PT_INVALID;
    if (t != PT_INVALID) {
        const double hg = q.h[g];
        hm = hg;
        if (!(t & PT_GHOST)) {
            double f = a.f;
            if (q.tc) {
                const double dt = q.tc[0];
                f = a.which == 1 ? 0.5 * dt : dt;
            }
            double x0, y0, z0, u0, v0, w0, r0;
            if (q.do_init) {
                x0 = a.x[g]; y0 = a.y[g]; z0 = a.z[g];
                u0 = a.u[g]; v0 = a.v[g]; w0 = a.w[g];
                r0 = a.rho[g];
                a.x0[g] = x0; a.y0[g] = y0; a.z0[g] = z0;
                a.u0[g] = u0; a.v0[g] = v0; a.w0[g] = w0;
                a.rho0[g] = r0;
            } else {
                x0 = a.x0[g]; y0 = a.y0[g]; z0 = a.z0[g];
                u0 = a.u0[g]; v0 = a.v0[g]; w0 = a.w0[g];
                r0 = a.rho0[g];
            }
            const double un = u0 + f * (double)a.au[g];
            const double vn = v0 + f * (double)a.av[g];
            const double wn = w0 + f * (double)a.aw[g];
            const double xn = x0 + f * (double)a.ax[g];
            const double yn = y0 + f * (double)a.ay[g];
            const double zn = z0 + f * (double)a.az[g];
            double r = r0 + f * (double)a.arho[g];
            a.u[g] = un; a.v[g] = vn; a.w[g] = wn;
            a.x[g] = xn; a.y[g] = yn; a.z[g] = zn;
            a.rho[g] = r;
            if (q.reduce_dt) {
                mc = (double)q.dt_cfl[g];
                mf = (double)q.dt_force[g];
            }
            // ---- records of the next evaluation ---------------------------------------
            const uint32_t s = q.rank[g];
            const uint32_t key = q.key_of[g];
            uint32_t cx, cy, cz;
            grid_decode(q.G.zorder, (uint32_t)q.G.nc[0], (uint32_t)q.G.nc[1], key, cx, cy, cz);
            float4 A, B, C;
            A.x = (float)(xn - (q.G.xmin[0] + (double)cx * q.G.cell[0]));
            A.y = (float)(yn - (q.G.xmin[1] + (double)cy * q.G.cell[1]));
            A.z = (float)(zn - (q.G.xmin[2] + (double)cz * q.G.cell[2]));
            A.w = (float)hg;
            B.x = (float)un; B.y = (float)vn; B.z = (float)wn; B.w = (float)q.m[g];
            float pg, csg;
            const int ar = t & 7;
            if (q.eos_any && q.E.on[ar]) {   // real particle: real_only does not matter here
                const double rho0 = q.E.rho0[ar];
                if (q.E.hg[ar] && r < rho0) r = rho0;   // the record only: the pool keeps rho
                const double ratio = r * (1.0 / rho0);
                const double Bc = rho0 * q.E.c0[ar] * q.E.c0[ar] / q.E.gamma[ar];
{ double rg_, rh_; tait_powers(ratio, q.E.gamma[ar], rg_, rh_);
                pg = (float)((q.E.hg[ar] ? 0.0 : q.E.p0[ar]) + Bc * (rg_ - 1.0));
                csg = (float)(q.E.c0[ar] * rh_); }
            } else {
                pg = q.p[g];
                csg = q.cs[g];
            }
            C.x = (float)r;
            C.y = (float)((double)pg / (r * r));
            C.z = csg;
            C.w = __int_as_float((int)t);
            q.AB[2 * (size_t)s] = A;
            q.AB[2 * (size_t)s + 1] = B;
            q.C[s] = C;
            q.R[2 * (size_t)s] = make_float4(A.x, A.y, A.z, __uint_as_float((unsigned)__float_as_int(C.x) | (((q.r32_cls >> ar) & 1u) << 31)));
            q.R[2 * (size_t)s + 1] = make_float4(B.x, B.y, B.z, C.y);
            const float4 b0 = q.A0[s];
            const float ex = A.x - b0.x, ey = A.y - b0.y, ez = A.z - b0.z;
            d2 = ex * ex + ey * ey + ez * ez;
            dh = fmaxf(A.w - b0.w, 0.f);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        d2 = fmaxf(d2, __shfl_xor_sync(0xffffffffu, d2, o));
        dh = fmaxf(dh, __shfl_xor_sync(0xffffffffu, dh, o));
    }
    if (q.reduce_dt) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mc = fmax(mc, __shfl_xor_sync(0xffffffffu, mc, o));
            mf = fmax(mf, __shfl_xor_sync(0xffffffffu, mf, o));
            hm = fmin(hm, __shfl_xor_sync(0xffffffffu, hm, o));
        }
    }
    // one atomic per block and quantity
    __shared__ float s_d2[8], s_dh[8];
    __shared__ double s_mc[8], s_mf[8], s_hm[8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) {
        s_d2[warp] = d2; s_dh[warp] = dh;
        s_mc[warp] = mc; s_mf[warp] = mf; s_hm[warp] = hm;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < 8; k++) {
            d2 = fmaxf(d2, s_d2[k]); dh = fmaxf(dh, s_dh[k]);
            mc = fmax(mc, s_mc[k]); mf = fmax(mf, s_mf[k]); hm = fmin(hm, s_hm[k]);
        }
        if (d2 > 0.f) atomicMax(&q.red_u32[0], __float_as_uint(d2));
        if (dh > 0.f) atomicMax(&q.red_u32[1], __float_as_uint(dh));
        if (q.reduce_dt) {
            if (mc > -1e299) atomicMax(&q.red[9], d2o(mc));
            if (mf > -1e299) atomicMax(&q.red[11], d2o(mf));
            if (hm < 1e299) atomicMin(&q.red[12], d2o(hm));
        }
    }
}

// TaitEOS.loop wc/basic.py:60-65 ; TaitEOSHGCorrection.loop wc/basic.py:118-126: the pending
// equation-of-state calls of every array in one launch (pool side: rho clamp of the HG
// variant, p, cs); same arithmetic as k_pack_state
__global__ void k_eos_tab(double *__restrict__ rho, float *__restrict__ p, float *__restrict__ cs,
                          const uint8_t *__restrict__ ptype, long long pool_end, const EosTab E)
{
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= pool_end) return;
    const uint8_t t = ptype[g];
    if (t == PT_INVALID) return;
    const int a = t & 7;
    if (!E.on[a] || (E.real_only[a] && (t & PT_GHOST))) return;
    double r = rho[g];
    const double rho0 = E.rho0[a];
    if (E.hg[a] && r < rho0) {
        r = rho0;
        rho[g] = r;
    }
    const double ratio = r * (1.0 / rho0);
    const double Bc = rho0 * E.c0[a] * E.c0[a] / E.gamma[a];
{ double rg_, rh_; tait_powers(ratio, E.gamma[a], rg_, rh_);
    p[g] = (float)((E.hg[a] ? 0.0 : E.p0[a]) + Bc * (rg_ - 1.0));
    cs[g] = (float)(E.c0[a] * rh_); }
}

// k_dt_propose + k_dt_commit in one launch (one rank: nothing to reduce in between), and
// the reduction slots are re-armed for the next step's fused stage kernel
__global__ void k_dt_advance(long long *__restrict__ red, double *__restrict__ tc, double cfl, int fixed_h,
                             double prev_factor, double new_factor, int adaptive, int advance, double t_final, double t_eps)
{
    if (adaptive) {
        const double mc = o2d(red[9]), mf = o2d(red[11]);
        const double f_cfl = mc < -1e299 ? -1.0 : mc, f_force = mf < -1e299 ? -1.0 : mf;
        double hmin = fmin(1.0, o2d(red[12]));
        if (!fixed_h || tc[3] < 0.0) tc[3] = hmin;
        hmin = tc[3];
        const double inf = __longlong_as_double(0x7ff0000000000000LL);
        double dt_cfl = inf, dt_force = inf;
        if (f_cfl > 0.0) dt_cfl = hmin / f_cfl;
        if (f_force > 0.0) dt_force = sqrt(hmin / sqrt(f_force));
        const double dt_min = fmin(dt_cfl, dt_force);
        tc[2] = (dt_min <= 0.0 || isinf(dt_min)) ? 1e20 : cfl * dt_min;
    }
    red[9] = d2o(-1e300); red[11] = d2o(-1e300); red[12] = d2o(1e300);
    const double dt_old = tc[0];
    if (advance) tc[1] += dt_old;
    const double t = tc[1];
    if (fabs(t_final - t) < t_eps) return;
    const double undamped = dt_old / prev_factor;
    double dt = undamped;
    if (adaptive) {
        dt = tc[2];
        if (dt >= 1e20) dt = undamped;
    }
    dt *= new_factor;
    if (t + dt > t_final - t_eps) dt = t_final - t;
    tc[0] = dt;
}

// _box_wrap_periodic (nnps_base.pyx:699-743): real and ghost particles alike
__global__ void k_box_wrap(double *__restrict__ x, double *__restrict__ y, double *__restrict__ z,
                           const uint8_t *__restrict__ ptype, long long pool_end, GridDev D /* xmin = lo, cell = L */)
{
    long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= pool_end || ptype[g] == PT_INVALID) return;
    double *p[3] = {x, y, z};
#pragma unroll
    for (int d = 0; d < 3; d++) {
        if (!D.periodic[d]) continue;
        double v = p[d][g];
        const double lo = D.xmin[d], L = D.cell[d];
        if (v < lo) v += L;
        if (v > lo + L) v -= L;
        p[d][g] = v;
    }
}
__global__ void k_f64_to_f32(const double *__restrict__ in, float *__restrict__ out, long long n)
{
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (float)in[i];
}
__global__ void k_f32_to_f64(const float *__restrict__ in, double *__restrict__ out, long long n)
{
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (double)in[i];
}

// per array (min, max) of h and of m over the real particles, as ordered int64 (d2o):
// out[4 a + 0 / 1] = min h / -max h, out[4 a + 2 / 3] = min m / -max m (everything a minimum,
// so that one initial value serves every slot).  Decides whether the R32 list kernel applies.
__global__ void k_uni_minmax(const double *__restrict__ h, const double *__restrict__ m,
                             const uint8_t *__restrict__ ptype, long long pool_end, long long *__restrict__ out)
{
    const unsigned FULL = 0xffffffffu;
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const uint8_t t = g < pool_end ? ptype[g] : (uint8_t)PT_INVALID;
    const bool valid = t != PT_INVALID && !(t & PT_GHOST);
    double v[4] = {1e300, 1e300, 1e300, 1e300};
    if (valid) {
        v[0] = h[g]; v[1] = -v[0];
        v[2] = m[g]; v[3] = -v[2];
    }
    // pools are array after array: a warp almost always holds one array, reduce it first
    const int arr = valid ? (t & 7) : -1;
    const int arr0 = __shfl_sync(FULL, arr, 0);
    const bool one = __ballot_sync(FULL, arr == arr0 || arr < 0) == FULL;
    if (one) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1)
#pragma unroll
            for (int k = 0; k < 4; k++) v[k] = fmin(v[k], __shfl_xor_sync(FULL, v[k], o));
    }
    if (one ? ((threadIdx.x & 31) == 0 && arr0 >= 0) : valid) {
        long long *o = out + 4 * (one ? arr0 : arr);
#pragma unroll
        for (int k = 0; k < 4; k++) atomicMin(o + k, d2o(v[k]));
    }
}
