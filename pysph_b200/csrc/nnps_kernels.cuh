// nnps_kernels.cuh -- cell keys, counting sort, cell-relative repack.
// Part of the single translation unit b200sph.cu (included there, in this order; not a
// stand-alone header).

// --------------------------------------------------------------------------
// NNPS build kernels
// --------------------------------------------------------------------------

// cell id = floor((p - xmin)/cell) per axis (find_cell_id_raw, nnps_base.pxd:39-80),
// flat = cx + ncx*cy + ncx*ncy*cz (flatten_raw, nnps_base.pxd:84-96) or, zorder, cx + ncx *
// morton(cy, cz) (z_order.h:24-46 interleaves all three; see grid_row); the arrival
// counter replaces the linked-list push (linked_list_nnps.pyx:285-286).
__global__ void k_cell_count(const double *__restrict__ x, const double *__restrict__ y,
                             const double *__restrict__ z, const uint8_t *__restrict__ ptype,
                             long long pool_end, GridDev G, uint32_t *__restrict__ key_of,
                             uint32_t *__restrict__ off_in, uint32_t *__restrict__ cell_cnt)
{
    long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= pool_end) return;
    if (ptype[g] == PT_INVALID) return;
    int cx = (int)floor((x[g] - G.xmin[0]) / G.cell[0]);
    int cy = (int)floor((y[g] - G.xmin[1]) / G.cell[1]);
    int cz = (int)floor((z[g] - G.xmin[2]) / G.cell[2]);
    cx = min(max(cx, 0), G.nc[0] - 1);
    cy = min(max(cy, 0), G.nc[1] - 1);
    cz = min(max(cz, 0), G.nc[2] - 1);
    uint32_t key = (uint32_t)cx + (uint32_t)G.nc[0] * grid_row(G.zorder, (uint32_t)G.nc[1], (uint32_t)cy, (uint32_t)cz);
    key_of[g] = key;
    off_in[g] = atomicAdd(&cell_cnt[key], 1u);
}

__global__ void k_scatter(const uint32_t *__restrict__ key_of, const uint32_t *__restrict__ off_in,
                          const uint8_t *__restrict__ ptype, long long pool_end,
                          const uint32_t *__restrict__ cell_start, uint32_t *__restrict__ perm_tmp)
{
    long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= pool_end) return;
    if (ptype[g] == PT_INVALID) return;
    perm_tmp[cell_start[key_of[g]] + off_in[g]] = (uint32_t)g;
}

// make the order inside every cell canonical (ascending pool index) so that the
// build -- and therefore every fp32 sum downstream -- is run-to-run deterministic.
__global__ void k_canon(const uint32_t *__restrict__ perm_tmp, const uint32_t *__restrict__ key_of,
                        const uint32_t *__restrict__ cell_start, long long n,
                        uint32_t *__restrict__ perm, uint32_t *__restrict__ skey,
                        uint32_t *__restrict__ rank)
{
    long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    const uint32_t g = perm_tmp[s];
    const uint32_t key = key_of[g];
    const uint32_t cs = cell_start[key], ce = cell_start[key + 1];
    uint32_t r = 0;
    for (uint32_t t = cs; t < ce; t++) r += (perm_tmp[t] < g) ? 1u : 0u;
    const uint32_t d = cs + r;
    perm[d] = g;
    skey[d] = key;
    rank[g] = d;
}

// A[s] = (x, y, z relative to the particle's own cell origin, h)
__global__ void k_pack_pos(const double *__restrict__ x, const double *__restrict__ y,
                           const double *__restrict__ z, const double *__restrict__ h,
                           const uint32_t *__restrict__ perm, const uint32_t *__restrict__ skey,
                           long long n, GridDev G, float4 *__restrict__ A, float4 *__restrict__ AB,
                           const uint8_t *__restrict__ ptype, uint8_t *__restrict__ stype,
                           float4 *__restrict__ R = nullptr)
{
    long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    const uint32_t g = perm[s];
    if (stype) stype[s] = ptype[g];
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
    if (R) {   // the position half of the 32-byte source record (PairArgs.R)
        float *r = reinterpret_cast<float *>(R + 2 * s);
        r[0] = a.x; r[1] = a.y; r[2] = a.z;
    }
}

// B[s] = (u, v, w, m);  C[s] = (rho, p/rho^2, cs, type); pending TaitEOS /
// TaitEOSHGCorrection calls (wc/basic.py:60-65,118-126) are applied on the way.  The state
// half of the 32-byte source record R (PairArgs.R) goes with them: (rho with the source class
// in its sign bit, r32_cls bit a = array a is class 1) and (u, v, w, p/rho^2).
__global__ void k_pack_state(const double *__restrict__ u, const double *__restrict__ v,
                             const double *__restrict__ w, const double *__restrict__ m,
                             double *__restrict__ rho, float *__restrict__ p,
                             float *__restrict__ cs, const uint8_t *__restrict__ ptype,
                             const uint32_t *__restrict__ perm, long long n,
                             float4 *__restrict__ B, float4 *__restrict__ C,
                             float4 *__restrict__ AB, const EosTab E, const int eos_any,
                             float4 *__restrict__ R = nullptr, const unsigned r32_cls = 0)
{
    long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    const uint32_t g = perm[s];
    const int t = (int)ptype[g];
    float4 b, c;
    b.x = (float)u[g]; b.y = (float)v[g]; b.z = (float)w[g]; b.w = (float)m[g];
    double r = rho[g];
    float pg, csg;
    const int a = t & 7;
    if (eos_any && E.on[a] && !(E.real_only[a] && (t & PT_GHOST))) {
        const double rho0 = E.rho0[a];
        if (E.hg[a] && r < rho0) {
            r = rho0;
            rho[g] = r;
        }
        const double ratio = r * (1.0 / rho0);
        const double Bc = rho0 * E.c0[a] * E.c0[a] / E.gamma[a];
{ double rg_, rh_; tait_powers(ratio, E.gamma[a], rg_, rh_);
        pg = (float)((E.hg[a] ? 0.0 : E.p0[a]) + Bc * (rg_ - 1.0));
        csg = (float)(E.c0[a] * rh_); }
        p[g] = pg;
        cs[g] = csg;
    } else {
        pg = p[g];
        csg = cs[g];
    }
    c.x = (float)r;
    c.y = (float)((double)pg / (r * r));
    c.z = csg;
    c.w = __int_as_float(t);
    B[s] = b;
    C[s] = c;
    AB[2 * s + 1] = b;
    if (R) {
        reinterpret_cast<float *>(R + 2 * s)[3] = __uint_as_float((unsigned)__float_as_int(c.x) | (((r32_cls >> a) & 1u) << 31));
        R[2 * s + 1] = make_float4(b.x, b.y, b.z, c.y);
    }
}
