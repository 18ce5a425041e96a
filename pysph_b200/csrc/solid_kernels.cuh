// solid_kernels.cuh -- elastic-dynamics passes.
// Part of the single translation unit b200sph.cu (included there, in this order; not a
// stand-alone header).

// --------------------------------------------------------------------------
// Elastic dynamics (solid_mech/basic.py:604-651), elastic arrays only.  NOT YET RUN ON
// HARDWARE.  Sorted records: AB = {A, B}, C3 = (rho, p, cs, type) [ctx->C], and the
// stress records T = (s - p I) / rho^2 and R (artificial stress), 6 components each:
//   T01 = (T00, T01, T02, T11)   T2R = (T12, T22, R00, R01)   R2 = (R02, R11, R12, R22)
// --------------------------------------------------------------------------
struct SolidArgs {
    const float4 *AB;
    float4 *C3, *T01, *T2R, *R2;
    const uint32_t *perm;
    const double *rho;
    const double *s[6];
    float *p, *vg[9], *r[6], *as[6];
    float *arho, *au, *av, *aw, *ax, *ay, *az;
    long long n;
    float cellx, celly, cellz, k2, kfac;
    unsigned elastic_mask, source_mask;   // destinations (and sources); all sources (+ rigid solids)
    int grad3d, ghost_group1;
    float eps, alpha, beta, eps_xsph;
    double c0_ref[B200SPH_MAX_ARRAYS], rho_ref[B200SPH_MAX_ARRAYS], G[B200SPH_MAX_ARRAYS];
    float wdeltap[B200SPH_MAX_ARRAYS], nexp[B200SPH_MAX_ARRAYS];
    unsigned long long *pair_counter;
};

__global__ void k_pack_solid(const double *__restrict__ u, const double *__restrict__ v, const double *__restrict__ w,
                             const double *__restrict__ m, const double *__restrict__ rho, const float *__restrict__ p,
                             const float *__restrict__ cs, const uint8_t *__restrict__ ptype,
                             const uint32_t *__restrict__ perm, long long n, float4 *__restrict__ B,
                             float4 *__restrict__ AB, float4 *__restrict__ C3)
{
    long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    const uint32_t g = perm[s];
    float4 b;
    b.x = (float)u[g]; b.y = (float)v[g]; b.z = (float)w[g]; b.w = (float)m[g];
    B[s] = b;
    AB[2 * s + 1] = b;
    C3[s] = make_float4((float)rho[g], p[g], cs[g], __int_as_float((int)ptype[g]));
}

// cyclic Jacobi for a symmetric 3x3 matrix (fp64): eigenvalues d, eigenvectors = columns of v
__device__ __forceinline__ void eigen_sym3(double a[3][3], double v[3][3], double d[3])
{
#pragma unroll
    for (int i = 0; i < 3; i++)
#pragma unroll
        for (int j = 0; j < 3; j++) v[i][j] = (i == j) ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 30; sweep++) {
        const double off = a[0][1] * a[0][1] + a[0][2] * a[0][2] + a[1][2] * a[1][2];
        const double diag = a[0][0] * a[0][0] + a[1][1] * a[1][1] + a[2][2] * a[2][2];
        if (off <= 1e-30 * diag || off == 0.0) break;
#pragma unroll
        for (int pq = 0; pq < 3; pq++) {
            const int p = pq == 2 ? 1 : 0, q = pq == 0 ? 1 : 2;
            if (a[p][q] == 0.0) continue;
            const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
            const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
            const double c = 1.0 / sqrt(t * t + 1.0), sn = t * c;
#pragma unroll
            for (int k = 0; k < 3; k++) {
                const double akp = a[k][p], akq = a[k][q];
                a[k][p] = c * akp - sn * akq;
                a[k][q] = sn * akp + c * akq;
            }
#pragma unroll
            for (int k = 0; k < 3; k++) {
                const double apk = a[p][k], aqk = a[q][k];
                a[p][k] = c * apk - sn * aqk;
                a[q][k] = sn * apk + c * aqk;
            }
#pragma unroll
            for (int k = 0; k < 3; k++) {
                const double vkp = v[k][p], vkq = v[k][q];
                v[k][p] = c * vkp - sn * vkq;
                v[k][q] = sn * vkp + c * vkq;
            }
        }
    }
    d[0] = a[0][0];
    d[1] = a[1][1];
    d[2] = a[2][2];
}

// group 1: IsothermalEOS, VelocityGradient2D/3D (the pair loop), MonaghanArtificialStress and
// -- it needs only this particle's gradient -- HookesDeviatoricStressRate of group 2; writes
// the stress records group 2 gathers
template <int K, int DIM>
__global__ void __launch_bounds__(LIST_NT, 4) k_solid_pass1(const SolidArgs a, const uint32_t *__restrict__ cnt,
                                                           const uint32_t *__restrict__ lst, const int capg)
{
    const int tid = threadIdx.x;
    const unsigned FULL = 0xffffffffu;
    const long long s = (long long)blockIdx.x * LIST_NT + tid;
    bool active = s < a.n, ghost_src = false;
    float4 Ai = make_float4(0.f, 0.f, 0.f, 0.f), Bi = Ai;
    int ti = 0, count = 0;
    if (active) {
        ti = __float_as_int(a.C3[s].w);
        const bool elastic = (a.elastic_mask >> (ti & 7)) & 1u;
        // ghost_group1: ghosts are destinations of group 1 like everyone else (real=False)
        ghost_src = elastic ? ((ti & PT_GHOST) && !a.ghost_group1) : (((a.source_mask >> (ti & 7)) & 1u) != 0);
        if (ghost_src || !elastic) active = false;
    }
    if (ghost_src) {
        // a ghost (group 1 is real=True) or a particle of a rigid solid (a destination of
        // nothing) is a source of group 2 with the values it carries
        const uint32_t g = a.perm[s];
        const double rho = a.rho[g], p = (double)a.p[g], rho21 = 1.0 / (rho * rho);
        a.T01[s] = make_float4((float)((a.s[0][g] - p) * rho21), (float)(a.s[1][g] * rho21), (float)(a.s[2][g] * rho21),
                               (float)((a.s[3][g] - p) * rho21));
        a.T2R[s] = make_float4((float)(a.s[4][g] * rho21), (float)((a.s[5][g] - p) * rho21), a.r[0][g], a.r[1][g]);
        a.R2[s] = make_float4(a.r[2][g], a.r[3][g], a.r[4][g], a.r[5][g]);
    }
    if (active) {
        ld_256(a.AB + 2 * (size_t)s, Ai, Bi);
        count = (int)cnt[s];
    }
    int cmax = count;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cmax = max(cmax, __shfl_xor_sync(FULL, cmax, o));
    const uint32_t *my = lst + ((size_t)(s >> 5) * (size_t)capg) * 32u + (uint32_t)(s & 31);
    const float hi2 = a.k2 * Ai.w * Ai.w;
    float g00 = 0.f, g01 = 0.f, g02 = 0.f, g10 = 0.f, g11 = 0.f, g12 = 0.f, g20 = 0.f, g21 = 0.f, g22 = 0.f;
    unsigned npairs = 0;
    struct Rec { float4 A, B, C; };
    list_walk<Rec>(my, count, cmax,
        [&](const uint32_t e, Rec &r) {
            const uint32_t j = LIST_J(e);
            ld_256(a.AB + 2u * j, r.A, r.B);
            r.C = a.C3[j];
        },
        [&](const bool live, const uint32_t e, const Rec &r) {
            const float4 Aj = r.A, Bj = r.B, Cj = r.C;
            const float4 T = list_cell_offset(e, a.cellx, a.celly, a.cellz);
            const float xij = Ai.x - Aj.x + T.x, yij = Ai.y - Aj.y + T.y, zij = Ai.z - Aj.z + T.z;
            const float r2 = xij * xij + yij * yij + zij * zij;
            if (live && ((r2 < hi2) || (r2 < a.k2 * Aj.w * Aj.w)) && ((a.source_mask >> (__float_as_int(Cj.w) & 7)) & 1u)) {
                npairs++;
                const float rinv = r2 > 1e-24f ? frsqrt(r2) : 0.0f;
                const float h1 = frcp(0.5f * (Ai.w + Aj.w));
                float w, dw;
                sph_kernel<K>(r2 * rinv * h1, w, dw);
                const float gt = dw * a.kfac * hpow<DIM>(h1) * h1 * rinv;   // DWIJ = gt * XIJ
                const float tmp = -Bj.w * frcp(Cj.x) * gt;                 // basic_equations.py:88-98
                const float du = tmp * (Bi.x - Bj.x), dv = tmp * (Bi.y - Bj.y), dwv = tmp * (Bi.z - Bj.z);
                g00 += du * xij; g01 += du * yij;
                g10 += dv * xij; g11 += dv * yij;
                if (a.grad3d) {
                    g02 += du * zij; g12 += dv * zij;
                    g20 += dwv * xij; g21 += dwv * yij; g22 += dwv * zij;
                }
            }
        });
    if (active) {
        const uint32_t g = a.perm[s];
        const int arr = ti & 7;
        const double rho = a.rho[g];
        const double p = a.c0_ref[arr] * a.c0_ref[arr] * (rho - a.rho_ref[arr]);   // solid_mech/basic.py:100-101
        a.p[g] = (float)p;
        double sd[6];
#pragma unroll
        for (int k = 0; k < 6; k++) sd[k] = a.s[k][g];
        // velocity gradient: the 2-D equation leaves the other five components alone
        float vgl[9];
        if (a.grad3d) {
            vgl[0] = g00; vgl[1] = g01; vgl[2] = g02; vgl[3] = g10; vgl[4] = g11; vgl[5] = g12;
            vgl[6] = g20; vgl[7] = g21; vgl[8] = g22;
#pragma unroll
            for (int k = 0; k < 9; k++) a.vg[k][g] = vgl[k];
        } else {
#pragma unroll
            for (int k = 0; k < 9; k++) vgl[k] = a.vg[k][g];
            vgl[0] = g00; vgl[1] = g01; vgl[3] = g10; vgl[4] = g11;
            a.vg[0][g] = g00; a.vg[1][g] = g01; a.vg[3][g] = g10; a.vg[4][g] = g11;
        }
        // MonaghanArtificialStress solid_mech/basic.py:170-242
        double S[3][3], Rv[3][3], ev[3], rd[3];
        S[0][0] = sd[0] - p; S[1][1] = sd[3] - p; S[2][2] = sd[5] - p;
        S[0][1] = S[1][0] = sd[1];
        S[0][2] = S[2][0] = sd[2];
        S[1][2] = S[2][1] = sd[4];
        eigen_sym3(S, Rv, ev);
        const double rho21 = 1.0 / (rho * rho);
#pragma unroll
        for (int k = 0; k < 3; k++) rd[k] = ev[k] > 0.0 ? -(double)a.eps * ev[k] * rho21 : 0.0;
        float rr[6];
        {
            const int IA[6] = {0, 0, 0, 1, 1, 2}, IB[6] = {0, 1, 2, 1, 2, 2};
#pragma unroll
            for (int q = 0; q < 6; q++) {
                double sum = 0.0;
#pragma unroll
                for (int k = 0; k < 3; k++) sum += Rv[IA[q]][k] * rd[k] * Rv[IB[q]][k];
                rr[q] = (float)sum;
                a.r[q][g] = rr[q];
            }
        }
        // HookesDeviatoricStressRate solid_mech/basic.py:420-505
        {
            double vv[3][3], ss[3][3], ep[3][3], om[3][3];
#pragma unroll
            for (int k = 0; k < 9; k++) vv[k / 3][k % 3] = (double)vgl[k];
            ss[0][0] = sd[0]; ss[0][1] = ss[1][0] = sd[1]; ss[0][2] = ss[2][0] = sd[2];
            ss[1][1] = sd[3]; ss[1][2] = ss[2][1] = sd[4]; ss[2][2] = sd[5];
#pragma unroll
            for (int i = 0; i < 3; i++)
#pragma unroll
                for (int j = 0; j < 3; j++) {
                    ep[i][j] = 0.5 * (vv[i][j] + vv[j][i]);
                    om[i][j] = 0.5 * (vv[i][j] - vv[j][i]);
                }
            const double tmp = 2.0 * a.G[arr];
            const double trace = (1.0 / 3.0) * (ep[0][0] + ep[1][1] + ep[2][2]);
            const int IA[6] = {0, 0, 0, 1, 1, 2}, IB[6] = {0, 1, 2, 1, 2, 2};
#pragma unroll
            for (int q = 0; q < 6; q++) {
                const int i = IA[q], j = IB[q];
                double t1 = 0.0, t2 = 0.0;
#pragma unroll
                for (int k = 0; k < 3; k++) {
                    t1 += ss[i][k] * om[j][k];
                    t2 += ss[k][j] * om[i][k];
                }
                a.as[q][g] = (float)(tmp * (ep[i][j] - (i == j ? trace : 0.0)) + t1 + t2);
            }
        }
        // records for group 2
        const float T00 = (float)((sd[0] - p) * rho21), T11 = (float)((sd[3] - p) * rho21), T22 = (float)((sd[5] - p) * rho21);
        const float T01 = (float)(sd[1] * rho21), T02 = (float)(sd[2] * rho21), T12 = (float)(sd[4] * rho21);
        a.T01[s] = make_float4(T00, T01, T02, T11);
        a.T2R[s] = make_float4(T12, T22, rr[0], rr[1]);
        a.R2[s] = make_float4(rr[2], rr[3], rr[4], rr[5]);
        a.C3[s].y = (float)p;
    }
    if (a.pair_counter) {
        if (ti & PT_GHOST) npairs = 0;   // ghost destinations (ghost_group1) are the owner's pairs
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) npairs += __shfl_xor_sync(FULL, npairs, o);
        if ((tid & 31) == 0 && npairs) atomicAdd(a.pair_counter, (unsigned long long)npairs);
    }
}

// group 2: ContinuityEquation, MomentumEquationWithStress, MonaghanArtificialViscosity, XSPHCorrection
template <int K, int DIM>
__global__ void __launch_bounds__(LIST_NT, 4) k_solid_pass2(const SolidArgs a, const uint32_t *__restrict__ cnt,
                                                           const uint32_t *__restrict__ lst, const int capg)
{
    const int tid = threadIdx.x;
    const unsigned FULL = 0xffffffffu;
    const long long s = (long long)blockIdx.x * LIST_NT + tid;
    bool active = s < a.n;
    float4 Ai = make_float4(0.f, 0.f, 0.f, 0.f), Bi = Ai, Ci = make_float4(1.f, 0.f, 0.f, 0.f), Ti1 = Ai, Ti2 = Ai, Ti3 = Ai;
    int ti = 0, count = 0;
    if (active) {
        Ci = a.C3[s];
        ti = __float_as_int(Ci.w);
        if ((ti & PT_GHOST) || !((a.elastic_mask >> (ti & 7)) & 1u)) active = false;
    }
    if (active) {
        ld_256(a.AB + 2 * (size_t)s, Ai, Bi);
        Ti1 = a.T01[s]; Ti2 = a.T2R[s]; Ti3 = a.R2[s];
        count = (int)cnt[s];
    }
    int cmax = count;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cmax = max(cmax, __shfl_xor_sync(FULL, cmax, o));
    const uint32_t *my = lst + ((size_t)(s >> 5) * (size_t)capg) * 32u + (uint32_t)(s & 31);
    const float hi2 = a.k2 * Ai.w * Ai.w;
    const float wdp = a.wdeltap[ti & 7], nexp = a.nexp[ti & 7];
    const float wdp1 = wdp > 0.f ? frcp(wdp) : 0.f;
    float arho = 0.f, au = 0.f, av = 0.f, aw = 0.f, ax = 0.f, ay = 0.f, az = 0.f;
    unsigned npairs = 0;
    struct Rec { float4 A, B, C, T1, T2, T3; };
    list_walk<Rec>(my, count, cmax,
        [&](const uint32_t e, Rec &r) {
            const uint32_t j = LIST_J(e);
            ld_256(a.AB + 2u * j, r.A, r.B);
            r.C = a.C3[j]; r.T1 = a.T01[j]; r.T2 = a.T2R[j]; r.T3 = a.R2[j];
        },
        [&](const bool live, const uint32_t e, const Rec &r) {
            const float4 Aj = r.A, Bj = r.B, Cj = r.C, Tj1 = r.T1, Tj2 = r.T2, Tj3 = r.T3;
            const float4 T = list_cell_offset(e, a.cellx, a.celly, a.cellz);
            const float xij = Ai.x - Aj.x + T.x, yij = Ai.y - Aj.y + T.y, zij = Ai.z - Aj.z + T.z;
            const float r2 = xij * xij + yij * yij + zij * zij;
            const int tj = __float_as_int(Cj.w) & 7;
            if (live && ((r2 < hi2) || (r2 < a.k2 * Aj.w * Aj.w)) && ((a.source_mask >> tj) & 1u)) {
                npairs++;
                const float rinv = r2 > 1e-24f ? frsqrt(r2) : 0.0f;
                const float hij = 0.5f * (Ai.w + Aj.w);
                const float h1 = frcp(hij);
                float w, dw;
                sph_kernel<K>(r2 * rinv * h1, w, dw);
                const float fac = a.kfac * hpow<DIM>(h1);
                const float wij = w * fac;
                const float gt = dw * fac * h1 * rinv;
                const float dwx = gt * xij, dwy = gt * yij, dwz = gt * zij;
                const float mb = Bj.w;
                const float uij = Bi.x - Bj.x, vij = Bi.y - Bj.y, wwij = Bi.z - Bj.z;
                const float vdotx = uij * xij + vij * yij + wwij * zij;
                arho += mb * (uij * dwx + vij * dwy + wwij * dwz);   // basic_equations.py:190-192
                // MomentumEquationWithStress solid_mech/basic.py:267-387
                float fab = 0.f;
                if (wdp > 0.f) fab = powf(wij * wdp1, nexp);
                const float m00 = Ti1.x + Tj1.x + fab * (Ti2.z + Tj2.z);
                const float m01 = Ti1.y + Tj1.y + fab * (Ti2.w + Tj2.w);
                const float m02 = Ti1.z + Tj1.z + fab * (Ti3.x + Tj3.x);
                const float m11 = Ti1.w + Tj1.w + fab * (Ti3.y + Tj3.y);
                const float m12 = Ti2.x + Tj2.x + fab * (Ti3.z + Tj3.z);
                const float m22 = Ti2.y + Tj2.y + fab * (Ti3.w + Tj3.w);
                float fu = mb * (m00 * dwx + m01 * dwy + m02 * dwz);
                float fv = mb * (m01 * dwx + m11 * dwy + m12 * dwz);
                float fw = mb * (m02 * dwx + m12 * dwy + m22 * dwz);
                // MonaghanArtificialViscosity basic_equations.py:240-257
                const float rhoij1 = 2.0f * frcp(Ci.x + Cj.x);
                if (vdotx < 0.f) {
                    const float cij = 0.5f * (Ci.z + Cj.z);
                    const float muij = hij * vdotx * frcp(r2 + 0.01f * hij * hij);
                    const float piij = (-a.alpha * cij * muij + a.beta * muij * muij) * rhoij1;
                    fu -= mb * piij * dwx;
                    fv -= mb * piij * dwy;
                    fw -= mb * piij * dwz;
                }
                au += fu; av += fv; aw += fw;
                if (tj == (ti & 7)) {   // XSPHCorrection(sources=[dest]) basic_equations.py:290-295
                    const float f = -a.eps_xsph * mb * wij * rhoij1;
                    ax += f * uij; ay += f * vij; az += f * wwij;
                }
            }
        });
    if (active) {
        const uint32_t g = a.perm[s];
        a.arho[g] = arho;
        a.au[g] = au; a.av[g] = av; a.aw[g] = aw;
        a.ax[g] = ax + Bi.x; a.ay[g] = ay + Bi.y; a.az[g] = az + Bi.z;   // post_loop :297-300
    }
    if (a.pair_counter) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) npairs += __shfl_xor_sync(FULL, npairs, o);
        if ((tid & 31) == 0 && npairs) atomicAdd(a.pair_counter, (unsigned long long)npairs);
    }
}

struct StageSolidArgs {
    double *x, *y, *z, *u, *v, *w, *rho, *s[6];
    double *x0, *y0, *z0, *u0, *v0, *w0, *rho0, *s0[6];
    const float *au, *av, *aw, *ax, *ay, *az, *arho, *as[6];
    const uint8_t *ptype;
    long long pool_end;
    int arr, which;
    double f;
};
// SolidMechStep integrator_step.py:173-252 (real particles)
__device__ __forceinline__ void stage_solid_body(const StageSolidArgs &a)
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
#pragma unroll
        for (int k = 0; k < 6; k++) a.s0[k][g] = a.s[k][g];
        return;
    }
    const double f = a.f;
    a.u[g] = a.u0[g] + f * (double)a.au[g];
    a.v[g] = a.v0[g] + f * (double)a.av[g];
    a.w[g] = a.w0[g] + f * (double)a.aw[g];
    a.x[g] = a.x0[g] + f * (double)a.ax[g];
    a.y[g] = a.y0[g] + f * (double)a.ay[g];
    a.z[g] = a.z0[g] + f * (double)a.az[g];
    a.rho[g] = a.rho0[g] + f * (double)a.arho[g];
#pragma unroll
    for (int k = 0; k < 6; k++) a.s[k][g] = a.s0[k][g] + f * (double)a.as[k][g];
}
__global__ void k_stage_solid(StageSolidArgs a) { stage_solid_body(a); }
__global__ void k_stage_solid_devdt(StageSolidArgs a, const double *__restrict__ tc)
{
    const double dt = tc[0];
    a.f = a.which == 1 ? 0.5 * dt : dt;
    stage_solid_body(a);
}

// refresh the packed positions in the FROZEN sorted order / cell frames of the last
// build and measure how far particles moved (and h grew) since then.
// red_u32[0] = max |dx|^2 (float bits), red_u32[1] = max (h - h_build) (float bits, >= 0)
__global__ void k_pack_pos_light(const double *__restrict__ x, const double *__restrict__ y,
                                 const double *__restrict__ z, const double *__restrict__ h,
                                 const uint32_t *__restrict__ perm, const uint32_t *__restrict__ skey,
                                 long long n, GridDev G, const float4 *__restrict__ A0,
                                 float4 *__restrict__ A, float4 *__restrict__ AB,
                                 float4 *__restrict__ R, unsigned *__restrict__ red_u32)
{
    long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    float d2 = 0.f, dh = 0.f;
    if (s < n) {
        const uint32_t g = perm[s];
        uint32_t key = skey[s];
        uint32_t cx, cy, cz;
        grid_decode(G.zorder, (uint32_t)G.nc[0], (uint32_t)G.nc[1], key, cx, cy, cz);
        float4 a;
        a.x = (float)(x[g] - (G.xmin[0] + (double)cx * G.cell[0]));
        a.y = (float)(y[g] - (G.xmin[1] + (double)cy * G.cell[1]));
        a.z = (float)(z[g] - (G.xmin[2] + (double)cz * G.cell[2]));
        a.w = (float)h[g];
        A[s] = a;
        AB[2 * s] = a;
        float *r = reinterpret_cast<float *>(R + 2 * s);   // the 32-byte source record (PairArgs.R)
        r[0] = a.x; r[1] = a.y; r[2] = a.z;
        const float4 b = A0[s];
        const float dx = a.x - b.x, dy = a.y - b.y, dz = a.z - b.z;
        d2 = dx * dx + dy * dy + dz * dz;
        dh = fmaxf(a.w - b.w, 0.f);
    }
    for (int o = 16; o > 0; o >>= 1) {
        d2 = fmaxf(d2, __shfl_xor_sync(0xffffffffu, d2, o));
        dh = fmaxf(dh, __shfl_xor_sync(0xffffffffu, dh, o));
    }
    if ((threadIdx.x & 31) == 0) {
        if (d2 > 0.f) atomicMax(&red_u32[0], __float_as_uint(d2));
        if (dh > 0.f) atomicMax(&red_u32[1], __float_as_uint(dh));
    }
}


// neighbour query for one destination particle with the pair kernel's accept test
// (cell by cell; periodic axes wrap).  One warp.
__global__ void k_neighbors(const float4 *__restrict__ A /* {A,B} interleaved: A of particle s at [2 s] */, const float4 *__restrict__ C,
                            const uint32_t *__restrict__ cell_start, const uint32_t *__restrict__ skey,
                            const uint32_t *__restrict__ perm, long long s, int src_arr,
                            long long src_off, GridDev G, float k2,
                            uint32_t *__restrict__ out, long long cap, unsigned long long *count)
{
    const int lane = threadIdx.x;
    const int ncx = G.nc[0], ncy = G.nc[1], ncz = G.nc[2];
    const float4 Ai = A[2 * (size_t)s];
    uint32_t kq = skey[s];
    uint32_t ucx, ucy, ucz;
    grid_decode(G.zorder, (uint32_t)ncx, (uint32_t)ncy, kq, ucx, ucy, ucz);
    const int cx = (int)ucx, cy = (int)ucy, cz = (int)ucz;
    const float hi2 = k2 * Ai.w * Ai.w;
    unsigned long long n = 0;
    for (int r = 0; r < 27; r++) {
        const int dx = (r % 3) - 1, dy = ((r / 3) % 3) - 1, dz = (r / 9) - 1;
        int xx = cx + dx, yy = cy + dy, zz = cz + dz;
        if (G.periodic[0]) xx = (xx + ncx) % ncx;
        if (G.periodic[1]) yy = (yy + ncy) % ncy;
        if (G.periodic[2]) zz = (zz + ncz) % ncz;
        if (xx < 0 || xx >= ncx || yy < 0 || yy >= ncy || zz < 0 || zz >= ncz) continue;
        const uint32_t c = (uint32_t)xx + (uint32_t)ncx * grid_row(G.zorder, (uint32_t)ncy, (uint32_t)yy, (uint32_t)zz);
        const uint32_t rs = cell_start[c], re = cell_start[c + 1];
        for (uint32_t t0 = rs; t0 < re; t0 += 32) {
            const uint32_t t = t0 + lane;
            bool ok = false;
            if (t < re) {
                const float4 Aj = A[2 * (size_t)t];
                const float xij = Ai.x - (float)dx * (float)G.cell[0] - Aj.x;
                const float yij = Ai.y - (float)dy * (float)G.cell[1] - Aj.y;
                const float zij = Ai.z - (float)dz * (float)G.cell[2] - Aj.z;
                const float r2 = xij * xij + yij * yij + zij * zij;
                ok = ((r2 < hi2) || (r2 < k2 * Aj.w * Aj.w)) &&
                     ((__float_as_int(C[t].w) & 7) == src_arr);
            }
            const unsigned m = __ballot_sync(0xffffffffu, ok);
            if (ok) {
                const unsigned long long pos = n + __popc(m & ((1u << lane) - 1u));
                if ((long long)pos < cap) out[pos] = (uint32_t)((long long)perm[t] - src_off);
            }
            n += __popc(m);
        }
    }
    if (lane == 0) *count = n;
}
