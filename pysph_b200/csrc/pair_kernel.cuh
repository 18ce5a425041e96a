// pair_kernel.cuh -- the fused WCSPH pair kernel without lists (k_pair) and what it shares with k_pair_list.
// Part of the single translation unit b200sph.cu (included there, in this order; not a
// stand-alone header).

// --------------------------------------------------------------------------
// the fused pair kernel
// --------------------------------------------------------------------------
struct PairArgs {
    const float4 *A, *B, *C, *AB;
    // the 32-byte source records of the R32 variant, two float4 per sorted slot: R[2s] = (x, y, z
    // cell-relative as in A, +-rho), R[2s+1] = (u, v, w, p / rho^2) -- the fp32 values A / B / C
    // carry; rho > 0, so its sign bit is free and holds the source class (0 / 1) that stands for
    // h, m and cs.  Written wherever A / AB / C are written for real particles.
    const float4 *R;
    // the R32 variant of k_pair_list: per source class, an array of the class (its byte of
    // emask gives the class's equation bits), m and cs / rho^3 = c0 / rho0^3
    int r32_rep[2];
    float r32_m[2], r32_coef[2];
    const uint32_t *cell_start, *skey, *perm;
    float *arho, *au, *av, *aw, *ax, *ay, *az, *dt_cfl, *dt_force;
    double *rho;  // SummationDensity destination (fp64 state)
    long long n;
    int ncx, ncy, ncz;
    int zorder;                 // rows along the Z-curve of (cy, cz), see grid_row
    float cellx, celly, cellz;  // internal cell edges
    float k2;                   // radius_scale^2
    float kfac;      // kernel.fac for this dim
    float deltap;
    unsigned long long emask[B200SPH_MAX_ARRAYS];  // per dest type: 8 bits per source type
    float c0, alpha, beta, gx, gy, gz, eps_xsph;
    float nu4, eta;             // LaminarViscosity: 4 nu, eta
    int tensile, real_only;
    unsigned long long *pair_counter;  // may be null
    // Group(start_idx, stop_idx): destinations [dlo, dhi) of every array, as indices INTO the
    // array (equation.py:448-520); read by the RANGED instantiations of k_pair_list only
    long long doff[B200SPH_MAX_ARRAYS], dlo[B200SPH_MAX_ARRAYS], dhi[B200SPH_MAX_ARRAYS];
};

#define PAIR_WARPS 8
#define PAIR_CHUNK 16
#define QCAP 64

struct Acc {
    float arho, au, av, aw, ax, ay, az, cfl, rsum;
};

// EQS: what the Group can contain, known when the kernel is chosen -- the low 8 bits are the
// equation bits that may occur, PAIR_EQS_TENSILE that the tensile correction may be on.
// The default admits everything; a narrower set lets the compiler drop the other
// equations' code and registers (k_pair_list has a variant for the WCSPH scheme's Group).
#define PAIR_EQS_TENSILE 0x100
#define PAIR_EQS_ALL 0x1FF
#define PAIR_EQS_WCSPH (B200SPH_EQ_CONTINUITY | B200SPH_EQ_MOMENTUM | B200SPH_EQ_XSPH)
// one accepted pair: `bits` are the equations of (destination, source); qv = (x_ij, h_j),
// Bj = (u, v, w, m)_j, Cj = (rho, p / rho^2, cs)_j
template <int K, int DIM, int EQS = PAIR_EQS_ALL>
__device__ __forceinline__ void pair_eval(const PairArgs &a, const unsigned bits, const float4 qv, const float4 Bj,
                                          const float4 Cj, const float4 Ai, const float4 Bi,
                                          const float4 Ci, const float tmpi, Acc &acc, unsigned &npairs)
{
    if (!bits) return;
    npairs++;
    const float xij = qv.x, yij = qv.y, zij = qv.z, hj = qv.w;
    // precomputed symbols, equation.py:188-297
    const float r2 = xij * xij + yij * yij + zij * zij;
    const bool far = r2 > 1e-24f;          // RIJ > 1e-12 guard of kernels.py:128-132
    const float rinv = far ? frsqrt(r2) : 0.0f;
    const float rij = r2 * rinv;
    const float hij = 0.5f * (Ai.w + hj);
    const float h1 = frcp(hij);
    const float q = rij * h1;
    const float fac = a.kfac * hpow<DIM>(h1);
    float w, dw;
    sph_kernel<K>(q, w, dw);
    const float wij = w * fac;
    const float gt = dw * fac * h1 * rinv;  // DWIJ = gt * XIJ  (gradient(), kernels.py:126-136)
    const float mj = Bj.w;
    const float uij = Bi.x - Bj.x, vij = Bi.y - Bj.y, wwij = Bi.z - Bj.z;
    const float vdotx = uij * xij + vij * yij + wwij * zij;

    if (bits & B200SPH_EQ_SUMMATION_DENSITY) acc.rsum += mj * wij;  // basic_equations.py:28-29
    if (bits & B200SPH_EQ_CONTINUITY)                              // basic_equations.py:190-192
        acc.arho += mj * gt * vdotx;
    if (bits & (B200SPH_EQ_MOMENTUM | B200SPH_EQ_MONAGHAN_AV | B200SPH_EQ_XSPH | (EQS & B200SPH_EQ_LAMINAR))) {
        const float rhoij1 = frcp(0.5f * (Ci.x + Cj.x));
        // wc/basic.py:215-222, basic_equations.py:245-252 (vdotx < 0 only); branch-free: in a
        // warp some lane almost always takes it, and a select is cheaper than a
        // reconvergence scope
        const float cij = 0.5f * (Ci.z + Cj.z);
        const float muij = hij * vdotx * frcp(r2 + 0.01f * hij * hij);
        const float piij = vdotx < 0.0f ? (-a.alpha * cij * muij + a.beta * muij * muij) * rhoij1 : 0.0f;
        if (bits & B200SPH_EQ_MOMENTUM) {
            if (r2 > 1e-12f)  // wc/basic.py:224-228
                acc.cfl = fmaxf(acc.cfl, fabsf(hij * vdotx * rinv * rinv) + a.c0);
            const float tmpj = Cj.y;  // p_j / rho_j^2 (precomputed in k_pack_state)
            float tmp = tmpi + tmpj;
            if ((EQS & PAIR_EQS_TENSILE) && a.tensile) {  // wc/basic.py:233-248
                float wdp, dwdp;
                sph_kernel<K>(a.deltap, wdp, dwdp);
                float fij = w / wdp;  // WIJ/WDP: the fac*h^-dim normalisation cancels
                fij = fij * fij;
                fij = fij * fij;
                const float Ri = tmpi > 0.0f ? 0.01f * tmpi : 0.2f * fabsf(tmpi);
                const float Rj = tmpj > 0.0f ? 0.01f * tmpj : 0.2f * fabsf(tmpj);
                tmp += (Ri + Rj) * fij;
            }
            const float f = -mj * (tmp + piij) * gt;  // wc/basic.py:255-257
            acc.au += f * xij;
            acc.av += f * yij;
            acc.aw += f * zij;
        }
        if (bits & B200SPH_EQ_MONAGHAN_AV) {  // basic_equations.py:254-257
            const float f = -mj * piij * gt;
            acc.au += f * xij;
            acc.av += f * yij;
            acc.aw += f * zij;
        }
        if ((EQS & B200SPH_EQ_LAMINAR) && (bits & B200SPH_EQ_LAMINAR)) {  // wc/viscosity.py:12-27
            // Fij = DWIJ . XIJ = gt r^2
            const float f = mj * a.nu4 * (gt * r2) * frcp((Ci.x + Cj.x) * (r2 + a.eta * hij * hij));
            acc.au += f * uij;
            acc.av += f * vij;
            acc.aw += f * wwij;
        }
        if (bits & B200SPH_EQ_XSPH) {  // basic_equations.py:290-295
            const float f = -a.eps_xsph * mj * wij * rhoij1;
            acc.ax += f * uij;
            acc.ay += f * vij;
            acc.az += f * wwij;
        }
    }
}

template <int K, int DIM, int EQS = PAIR_EQS_ALL>
__device__ __forceinline__ void pair_body(const PairArgs &a, const float4 qv, const float4 Bj,
                                          const float4 Cj, const float4 Ai, const float4 Bi,
                                          const float4 Ci, const unsigned long long mask_i,
                                          const float tmpi, Acc &acc, unsigned &npairs)
{
    const int tj = __float_as_int(Cj.w) & 7;
    const unsigned bits = (unsigned)(mask_i >> (8 * tj)) & (unsigned)(EQS & 0xFF);
    pair_eval<K, DIM, EQS>(a, bits, qv, Bj, Cj, Ai, Bi, Ci, tmpi, acc, npairs);
}

template <int K, int DIM>
__global__ void __launch_bounds__(PAIR_WARPS * 32) k_pair(const PairArgs a)
{
    __shared__ float4 q_v[PAIR_WARPS][QCAP];
    __shared__ uint32_t q_i[PAIR_WARPS][QCAP];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned FULL = 0xffffffffu;
    const unsigned lt_mask = (1u << lane) - 1u;
    const long long first = ((long long)blockIdx.x * PAIR_WARPS + warp) * PAIR_CHUNK;

    uint32_t cur_key = 0xFFFFFFFFu;
    int cx = 0;
    // lane r < 9 holds the candidate range of neighbour row r = (dy+1) + 3*(dz+1)
    uint32_t r_rs = 0, r_b1 = 0, r_b2 = 0, r_re = 0;
    unsigned npairs = 0;

    for (int kk = 0; kk < PAIR_CHUNK; kk++) {
        const long long s = first + kk;
        if (s >= a.n) break;
        const float4 Ci = a.C[s];
        const int ti = __float_as_int(Ci.w);
        if (a.real_only && (ti & PT_GHOST)) continue;
        const unsigned long long mask_i = a.emask[ti & 7];
        if (!mask_i) continue;
        const float4 Ai = a.A[s];
        const float4 Bi = a.B[s];
        const uint32_t key = a.skey[s];
        if (key != cur_key) {
            cur_key = key;
            uint32_t ucx, ucy, ucz;
            grid_decode(a.zorder, (uint32_t)a.ncx, (uint32_t)a.ncy, key, ucx, ucy, ucz);
            cx = (int)ucx;
            const int cy = (int)ucy, cz = (int)ucz;
            r_rs = r_b1 = r_b2 = r_re = 0;
            if (lane < 9) {
                const int yy = cy + (lane % 3) - 1, zz = cz + (lane / 3) - 1;
                if (yy >= 0 && yy < a.ncy && zz >= 0 && zz < a.ncz) {
                    const uint32_t base = grid_row(a.zorder, (uint32_t)a.ncy, (uint32_t)yy, (uint32_t)zz) * (uint32_t)a.ncx;
                    const int x0 = max(cx - 1, 0), x1 = min(cx + 1, a.ncx - 1);
                    r_rs = a.cell_start[base + x0];
                    r_b1 = a.cell_start[base + cx];
                    r_b2 = a.cell_start[base + cx + 1];
                    r_re = a.cell_start[base + x1 + 1];
                }
            }
        }
        const float hi2 = a.k2 * Ai.w * Ai.w;
        const float tmpi = Ci.y;  // p_i / rho_i^2
        Acc acc = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        int qn = 0, qhead = 0;

        for (int r = 0; r < 9; r++) {
            const uint32_t rs = __shfl_sync(FULL, r_rs, r);
            const uint32_t re = __shfl_sync(FULL, r_re, r);
            if (rs >= re) continue;
            const uint32_t b1 = __shfl_sync(FULL, r_b1, r);
            const uint32_t b2 = __shfl_sync(FULL, r_b2, r);
            const float yoff = Ai.y - (float)((r % 3) - 1) * a.celly;
            const float zoff = Ai.z - (float)((r / 3) - 1) * a.cellz;
            for (uint32_t t0 = rs; t0 < re; t0 += 32) {
                const uint32_t t = t0 + lane;
                bool ok = false;
                float xij = 0.f, yij = 0.f, zij = 0.f, hj = 0.f;
                if (t < re) {
                    const float4 Aj = a.A[t];
                    const float xo = t >= b2 ? a.cellx : (t >= b1 ? 0.0f : -a.cellx);
                    xij = Ai.x - Aj.x - xo;
                    yij = yoff - Aj.y;
                    zij = zoff - Aj.z;
                    hj = Aj.w;
                    const float r2 = xij * xij + yij * yij + zij * zij;
                    // linked_list_nnps.pyx:188: (xij2 < hi2) or (xij2 < hj2)
                    ok = (r2 < hi2) || (r2 < a.k2 * hj * hj);
                }
                const unsigned m = __ballot_sync(FULL, ok);
                if (m) {
                    if (ok) {
                        const int pos = (qhead + qn + __popc(m & lt_mask)) & (QCAP - 1);
                        q_v[warp][pos] = make_float4(xij, yij, zij, hj);
                        q_i[warp][pos] = t;
                    }
                    qn += __popc(m);
                    __syncwarp();
                    if (qn >= 32) {
                        const int e = (qhead + lane) & (QCAP - 1);
                        const uint32_t tq = q_i[warp][e];
                        pair_body<K, DIM>(a, q_v[warp][e], a.B[tq], a.C[tq], Ai, Bi, Ci, mask_i,
                                          tmpi, acc, npairs);
                        qhead = (qhead + 32) & (QCAP - 1);
                        qn -= 32;
                        __syncwarp();
                    }
                }
            }
        }
        if (lane < qn) {
            const int e = (qhead + lane) & (QCAP - 1);
            const uint32_t tq = q_i[warp][e];
            pair_body<K, DIM>(a, q_v[warp][e], a.B[tq], a.C[tq], Ai, Bi, Ci, mask_i, tmpi, acc, npairs);
        }
        __syncwarp();

        // warp reduction of the per-particle sums
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            acc.arho += __shfl_xor_sync(FULL, acc.arho, o);
            acc.au += __shfl_xor_sync(FULL, acc.au, o);
            acc.av += __shfl_xor_sync(FULL, acc.av, o);
            acc.aw += __shfl_xor_sync(FULL, acc.aw, o);
            acc.ax += __shfl_xor_sync(FULL, acc.ax, o);
            acc.ay += __shfl_xor_sync(FULL, acc.ay, o);
            acc.az += __shfl_xor_sync(FULL, acc.az, o);
            acc.rsum += __shfl_xor_sync(FULL, acc.rsum, o);
            acc.cfl = fmaxf(acc.cfl, __shfl_xor_sync(FULL, acc.cfl, o));
        }
        if (lane == 0) {
            unsigned all_bits = 0;
#pragma unroll
            for (int j = 0; j < B200SPH_MAX_ARRAYS; j++) all_bits |= (unsigned)(mask_i >> (8 * j)) & 0xFFu;
            const uint32_t g = a.perm[s];
            if (all_bits & B200SPH_EQ_SUMMATION_DENSITY) a.rho[g] = (double)acc.rsum;
            if (all_bits & B200SPH_EQ_CONTINUITY) a.arho[g] = acc.arho;
            if (all_bits & B200SPH_EQ_MOMENTUM) {
                // post_loop wc/basic.py:259-269
                const float fu = acc.au + a.gx, fv = acc.av + a.gy, fw = acc.aw + a.gz;
                a.au[g] = fu; a.av[g] = fv; a.aw[g] = fw;
                a.dt_cfl[g] = acc.cfl;
                a.dt_force[g] = fu * fu + fv * fv + fw * fw;
            } else if (all_bits & (B200SPH_EQ_MONAGHAN_AV | B200SPH_EQ_LAMINAR)) {
                a.au[g] = acc.au; a.av[g] = acc.av; a.aw[g] = acc.aw;
            }
            if (all_bits & B200SPH_EQ_XSPH) {
                // post_loop basic_equations.py:297-300
                a.ax[g] = acc.ax + Bi.x; a.ay[g] = acc.ay + Bi.y; a.az[g] = acc.az + Bi.z;
            }
        }
    }
    if (a.pair_counter) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) npairs += __shfl_xor_sync(FULL, npairs, o);
        if (lane == 0 && npairs) atomicAdd(a.pair_counter, (unsigned long long)npairs);
    }
}
