// pair_list.cuh -- persistent neighbour lists: k_list_build and the dominant kernel k_pair_list.
// Part of the single translation unit b200sph.cu (included there, in this order; not a
// stand-alone header).

// --------------------------------------------------------------------------
// persistent neighbour lists (the default fast path)
//
// k_list_build runs the reference's accept test widened by a skin S
//   r^2 < (k h_i + S)^2  or  r^2 < (k h_j + S)^2
// once per (re)build and stores, for every destination, the sorted indices of
// the candidates that pass, 32 destinations interleaved ("transposed") so that
// the consumer reads them coalesced.  The lists stay valid while
//   2 max|x - x_build| + k max(h - h_build) <= S            (checked every update),
// so an evaluation normally only runs k_pair_list: one THREAD per destination
// walks its list, re-applies the EXACT accept test of linked_list_nnps.pyx:188
// on the current positions and evaluates the equations.  Results are identical
// to rebuilding the neighbours every evaluation; only the cost is amortised.
// entry = j << 6 | code: j = sorted index (26 bits), code = (dxc+1) + 4 (dy+1) + 16 (dz+1).
// The index sits in the HIGH bits so that a consumer gets it with one shift and both record
// addresses with one IMAD.WIDE each (no mask), the code with one AND.
// --------------------------------------------------------------------------
#define LIST_JBITS 26
#define LIST_CBITS 6
#define LIST_ENTRY(j, code) (((uint32_t)(j) << LIST_CBITS) | (uint32_t)(code))
#define LIST_J(e) ((uint32_t)(e) >> LIST_CBITS)
#define LIST_CODE(e) ((uint32_t)(e) & 63u)
#define LIST_NT 128
// Skin controller.  Per evaluation a build costs c0 (1+s)^3 (list entries) + R / L(s)
// (rebuild cost R over a lifetime L that grows linearly with the skin s); the minimum is
// where L s = R / (3 c0 (1+s)^2) ~ 2 for the measured R / c0 ~ 5.5, i.e. the target
// lifetime is L* = SKIN_KAPPA / s evaluations.
#define SKIN_KAPPA 2.0

struct ListBuildArgs {
    const float4 *A;
    const uint32_t *cell_start, *skey;
    long long n;
    int ncx, ncy, ncz;
    int zorder;                     // rows along the Z-curve of (cy, cz), see grid_row
    int px, py, pz;                 // periodic axes (cell indices wrap, images shift by nc * cell)
    float cellx, celly, cellz;      // internal cell edges (>= k hmax + S)
    float kr, S;     // radius scale, absolute skin
    uint32_t *cnt;   // [n] neighbours per destination
    uint32_t *lst;   // null: count only
    int capg;        // entries reserved per destination
    unsigned *max_count;
    // the (destination type, source type) pairs for which some equation of the Group exists
    // (8 bits per source type, as PairArgs.emask; all ones: no filter): an entry the pair
    // kernel would gather only to find no equation for it is not stored.  stype[s] = particle
    // type byte (array id | ghost bit) in sorted order.
    unsigned long long emask[B200SPH_MAX_ARRAYS];
    const uint8_t *stype;
};

// One THREAD per destination, one warp per 32 consecutive destinations of the sorted order
// (normally 1-2 cells of one cell row).  For each of the 9 neighbour rows (dy, dz) the warp
// stages the candidates of the cells [cx_min - 1, cx_max + 1] -- one contiguous range of
// the sorted arrays -- tile by tile into shared memory with coalesced loads; every lane
// then walks the tile (broadcast reads), keeps the candidates of ITS three cells, applies
// the skin-widened accept test (on x coordinates relative to the segment's first cell, the
// widened radius squared once per candidate at staging time) and appends to its own list.
// The list only has to CONTAIN every pair the exact test can accept while the build is valid
// (there is a 2 % margin on the skin for the fp32 drift measurement); which candidates of the
// skin shell it holds beyond that is immaterial.  Entries come out in the order
// "row (dy, dz), then ascending sorted index", which is also the order the pair kernels
// sum in.  (The first builder of this file put a warp on ONE destination with the lanes
// across candidates: 1.4 G warp instructions at 1.2 M particles, 91 % issue-bound,
// profiles/r02a_ncu_summary.md; this one executes about a third of that.)
// PERIODIC: y / z row indices wrap; on a periodic x axis the cells that wrap (cx = -1 seen
// from cx = 0, cx = ncx seen from ncx - 1) are staged as extra segments after the 9 rows,
// first all "left" wraps then all "right" wraps.  Because coordinates are relative to the
// particle's own cell and a periodic axis is tiled exactly (L = nc * cell), the image shift
// of a wrapped neighbour cell is the same "- d * cell" offset as for an ordinary neighbour
// cell -- the consumer kernels do not know about periodicity at all, and no ghost
// particles are materialised (reference: _create_ghosts_periodic, nnps_base.pyx:744-940).
#define LB_WARPS 4
#define LB_TILE 128
template <bool PERIODIC>
__global__ void __launch_bounds__(LB_WARPS * 32) k_list_build(const ListBuildArgs a)
{
    __shared__ float4 s_A[LB_WARPS][LB_TILE];
    __shared__ int s_cx[LB_WARPS][LB_TILE];     // cell x index | source type << 24
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned FULL = 0xffffffffu;
    const long long s = ((long long)blockIdx.x * LB_WARPS + warp) * 32 + lane;
    const bool valid = s < a.n;
    float4 Ai = make_float4(0.f, 0.f, 0.f, 0.f);
    uint32_t cxi = 0, cyi = 0, czi = 0, row_i = 0xFFFFFFFFu;
    unsigned long long mask_i = 0;
    if (valid) {
        Ai = a.A[s];
        grid_decode(a.zorder, (uint32_t)a.ncx, (uint32_t)a.ncy, a.skey[s], cxi, cyi, czi);
        row_i = cyi + (uint32_t)a.ncy * czi;
        mask_i = a.emask[a.stype[s] & 7];
    }
    const float hi = a.kr * Ai.w + a.S;
    const float hi2 = hi * hi;
    uint32_t *out = (a.lst && valid) ? a.lst + ((size_t)(s >> 5) * (size_t)a.capg) * 32u + (uint32_t)(s & 31) : nullptr;
    unsigned count = 0;
    // the lanes of a warp usually share one cell row; at a row end they are served row by row
    unsigned todo = __ballot_sync(FULL, valid);
    while (todo) {
        const int leader = __ffs(todo) - 1;
        const uint32_t row = __shfl_sync(FULL, row_i, leader);
        const bool mine = valid && row_i == row;
        const unsigned group = __ballot_sync(FULL, mine);
        todo &= ~group;
        const int cy = (int)__shfl_sync(FULL, cyi, leader), cz = (int)__shfl_sync(FULL, czi, leader);
        int cxa = mine ? (int)cxi : 0x7fffffff, cxb = mine ? (int)cxi : -1;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            cxa = min(cxa, __shfl_xor_sync(FULL, cxa, o));
            cxb = max(cxb, __shfl_xor_sync(FULL, cxb, o));
        }
        // segments: 0..8 the rows (dy, dz); PERIODIC in x: 9..17 the cell ncx - 1 seen as cx = -1,
        // 18..26 the cell 0 seen as cx = ncx
        for (int seg = 0; seg < (PERIODIC ? 27 : 9); seg++) {
            const int q = seg % 9, kind = seg / 9;
            if (PERIODIC && kind == 1 && !(a.px && cxa == 0)) continue;
            if (PERIODIC && kind == 2 && !(a.px && cxb == a.ncx - 1)) continue;
            int yy = cy + (q % 3) - 1, zz = cz + (q / 3) - 1;
            if (PERIODIC) {
                if (a.py) yy = (yy + a.ncy) % a.ncy;
                if (a.pz) zz = (zz + a.ncz) % a.ncz;
            }
            if (yy < 0 || yy >= a.ncy || zz < 0 || zz >= a.ncz) continue;
            const uint32_t base = grid_row(a.zorder, (uint32_t)a.ncy, (uint32_t)yy, (uint32_t)zz) * (uint32_t)a.ncx;
            uint32_t rs, re;
            int cx_fixed = 0;                       // kind 1 / 2: the apparent cell index of the wrapped cell
            if (kind == 0) {
                rs = a.cell_start[base + max(cxa - 1, 0)];
                re = a.cell_start[base + min(cxb + 1, a.ncx - 1) + 1];
            } else if (kind == 1) {
                rs = a.cell_start[base + a.ncx - 1];
                re = a.cell_start[base + a.ncx];
                cx_fixed = -1;
            } else {
                rs = a.cell_start[base];
                re = a.cell_start[base + 1];
                cx_fixed = a.ncx;
            }
            if (rs >= re) continue;
            // x relative to the cell cxa - 1 for the lane and for every candidate of the segment:
            // no per-candidate cell arithmetic in the loop below, and a candidate two or more
            // cells away in x cannot pass the distance test (the cell edge is the widened cut-off)
            const int x0c = cxa - 1;
            const float xoff = Ai.x + (float)((int)cxi - x0c) * a.cellx;
            const float yoff = Ai.y - (float)((q % 3) - 1) * a.celly;
            const float zoff = Ai.z - (float)((q / 3) - 1) * a.cellz;
            const uint32_t rcode = (uint32_t)(4 * (q % 3) + 16 * (q / 3));
            for (uint32_t t0 = rs; t0 < re; t0 += LB_TILE) {
                const int tn = (int)min((uint32_t)LB_TILE, re - t0);
                __syncwarp();
                for (int k = lane; k < tn; k += 32) {
                    float4 Aj = a.A[t0 + k];
                    const int cxj = kind == 0 ? (int)(a.skey[t0 + k] - base) : cx_fixed;
                    const float hj = a.kr * Aj.w + a.S;
                    Aj.x += (float)(cxj - x0c) * a.cellx;
                    Aj.w = hj * hj;
                    s_A[warp][k] = Aj;
                    s_cx[warp][k] = (cxj + 1) | ((int)(a.stype[t0 + k] & 7) << 24);   // cxj >= -1
                }
                __syncwarp();
                if (mine && mask_i) {
#pragma unroll 4
                    for (int k = 0; k < tn; k++) {
                        const float4 Aj = s_A[warp][k];
                        const float xij = xoff - Aj.x, yij = yoff - Aj.y, zij = zoff - Aj.z;
                        const float r2 = xij * xij + yij * yij + zij * zij;
                        if ((r2 < hi2) || (r2 < Aj.w)) {
                            const int cj = s_cx[warp][k];
                            const int dxc1 = (cj & 0xFFFFFF) - 1 - (int)cxi + 1;     // dxc + 1
                            if ((unsigned)dxc1 <= 2u && ((mask_i >> (8 * (cj >> 24))) & 0xFFull)) {
                                if (out && count < (unsigned)a.capg) out[(size_t)count * 32u] = LIST_ENTRY(t0 + (uint32_t)k, rcode + (uint32_t)dxc1);
                                count++;
                            }
                        }
                    }
                }
            }
        }
    }
    if (valid) a.cnt[s] = count;
    unsigned wmax = count;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) wmax = max(wmax, __shfl_xor_sync(FULL, wmax, o));
    if (lane == 0 && wmax) atomicMax(a.max_count, wmax);
}

// one 256-bit read-only load (LDG.E.ENL2.256 on sm_100a): a whole 32-byte sector
__device__ __forceinline__ void ld_256(const float4 *p, float4 &b, float4 &c)
{
    asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w), "=f"(c.x), "=f"(c.y), "=f"(c.z), "=f"(c.w)
                 : "l"(p));
}

// The list consumer (the default fast path): one THREAD per destination walks its
// list.  Per entry it gathers {A, B} = (x, y, z, h, u, v, w, m) with ONE 256-bit load
// (exactly one 32-byte sector) and C = (rho, p/rho^2, cs, type) with one 128-bit load,
// both issued one entry ahead of their use; list entries stream in (evict-first) two
// entries ahead.  The gathers and instruction issue bound this kernel at the same time
// (profiles/), hence the sector-sized records and the hand-scheduled loop: two entries
// per trip with ping-pong record registers (no register-rotation moves), 32-bit record
// indices (one IMAD.WIDE per address).
__device__ __forceinline__ void ld_rec(const PairArgs &a, const uint32_t e, float4 &A, float4 &B, float4 &C)
{
    const uint32_t j = LIST_J(e);
    ld_256(a.AB + 2u * j, A, B);
    C = __ldg(a.C + j);
}

// The software-pipelined walk over one destination's list that every list consumer shares:
// two entries per trip with ping-pong record registers; entries stream in (evict-first) two
// entries ahead, the record of an entry is loaded one entry ahead of its use.  `load(e, rec)`
// gathers the records entry e names -- unconditionally: an entry past the lane's own count
// reads as 0 = "record 0, same cell" -- and `body(live, e, rec)` does the work, live = false
// for the lanes whose list is shorter than the warp's longest.
template <class Rec, class Load, class Body>
__device__ __forceinline__ void list_walk(const uint32_t *nxt, const int count, int cmax, Load load, Body body)
{
    uint32_t e0 = count > 0 ? __ldcs(nxt) : 0u;
    uint32_t e1 = count > 1 ? __ldcs(nxt + 32) : 0u;
    nxt += 64;
    Rec r0, r1;
    load(e0, r0);
    for (int rem = count; cmax > 0; cmax -= 2, rem -= 2, nxt += 64) {
        const uint32_t e2 = rem > 2 ? __ldcs(nxt) : 0u;
        load(e1, r1);
        body(rem > 0, e0, r0);
        const uint32_t e3 = rem > 3 ? __ldcs(nxt + 32) : 0u;
        load(e2, r0);
        body(rem > 1, e1, r1);
        e0 = e2;
        e1 = e3;
    }
}

// the cell offset a list entry carries, as the vector to ADD to (x_i - x_j) of cell-relative
// coordinates: -(d - 1) * cell per axis, d the 2-bit code field.  (code field | 0x4B000000) as a
// float is 2^23 + field exactly, so the decode is one LOP3 + one FADD per axis; a shared-memory
// table of the 64 vectors cost 16 % of the LSU data-pipe wavefronts in k_pair_list.
__device__ __forceinline__ float4 list_cell_offset(const uint32_t e, const float cellx, const float celly, const float cellz)
{
    const float dxc = __uint_as_float((e & 3u) | 0x4B000000u) - 8388609.0f;
    const float dyc = __uint_as_float(((e >> 2) & 3u) | 0x4B000000u) - 8388609.0f;
    const float dzc = __uint_as_float(((e >> 4) & 3u) | 0x4B000000u) - 8388609.0f;
    return make_float4(-dxc * cellx, -dyc * celly, -dzc * cellz, 0.f);
}

// one list entry: cell-offset lookup, distance, the exact accept test, the equations.  `live`
// is false for the lanes whose list is shorter than the warp's longest (their entry reads
// as 0 and their record as record 0, so everything up to the test is harmless to execute).
template <int K, int DIM, int EQS>
__device__ __forceinline__ void pair_entry(const PairArgs &a, const bool live, const uint32_t e,
                                           const float4 Aj, const float4 Bj, const float4 Cj, const float4 Ai,
                                           const float4 Bi, const float4 Ci, const float hi2,
                                           const unsigned long long mask_i, Acc &acc, unsigned &npairs)
{
    // cell offset of the neighbour's cell relative to the destination's, decoded arithmetically:
    // (code field | 0x4B000000) as a float is 2^23 + field, exactly, so field - 1 costs one
    // LOP3 and one FADD per axis.  (A shared-memory table of the 64 offset vectors was the
    // alternative: its divergent 128-bit reads were 16 % of the LSU data-pipe wavefronts,
    // the pipe that bounds this kernel -- profiles/r02a_ncu_summary.md.)
    const float dxc = __uint_as_float((e & 3u) | 0x4B000000u) - 8388609.0f;
    const float dyc = __uint_as_float(((e >> 2) & 3u) | 0x4B000000u) - 8388609.0f;
    const float dzc = __uint_as_float(((e >> 4) & 3u) | 0x4B000000u) - 8388609.0f;
    const float xij = fmaf(-dxc, a.cellx, Ai.x - Aj.x), yij = fmaf(-dyc, a.celly, Ai.y - Aj.y),
                zij = fmaf(-dzc, a.cellz, Ai.z - Aj.z);
    const float r2 = xij * xij + yij * yij + zij * zij;
    // the exact accept test, linked_list_nnps.pyx:188
    if (live && ((r2 < hi2) || (r2 < a.k2 * Aj.w * Aj.w)))
        pair_body<K, DIM, EQS>(a, make_float4(xij, yij, zij, Aj.w), Bj, Cj, Ai, Bi, Ci, mask_i, Ci.y, acc, npairs);
}

// The same entry from the 32-byte record R (the R32 variant: one h for every particle, m and
// the Tait EOS uniform within each of at most two source classes, no ghosts).  h_j = h_i makes
// the two-sided accept test one-sided; the sign bit of rho_j selects the class: its equation
// bits, m_j, and cs_j = c0 (rho_j / rho0)^3 recomputed in fp32 (the only arithmetic that differs
// from the 48-byte path: a few ulp of cs_j inside Pi_ij).
template <int K, int DIM, int EQS>
__device__ __forceinline__ void pair_entry_r32(const PairArgs &a, const bool live, const uint32_t e,
                                               const float4 Pj, const float4 Qj, const float4 Ai,
                                               const float4 Bi, const float4 Ci, const float hi2,
                                               const unsigned bits0, const unsigned bits1,
                                               Acc &acc, unsigned &npairs)
{
    const float dxc = __uint_as_float((e & 3u) | 0x4B000000u) - 8388609.0f;
    const float dyc = __uint_as_float(((e >> 2) & 3u) | 0x4B000000u) - 8388609.0f;
    const float dzc = __uint_as_float(((e >> 4) & 3u) | 0x4B000000u) - 8388609.0f;
    const float xij = fmaf(-dxc, a.cellx, Ai.x - Pj.x), yij = fmaf(-dyc, a.celly, Ai.y - Pj.y),
                zij = fmaf(-dzc, a.cellz, Ai.z - Pj.z);
    const float r2 = xij * xij + yij * yij + zij * zij;
    if (live && r2 < hi2) {
        const bool c1 = __float_as_int(Pj.w) < 0;
        const float rhoj = fabsf(Pj.w);
        const float csj = (c1 ? a.r32_coef[1] : a.r32_coef[0]) * (rhoj * rhoj * rhoj);
        pair_eval<K, DIM, EQS>(a, c1 ? bits1 : bits0, make_float4(xij, yij, zij, Ai.w),
                               make_float4(Qj.x, Qj.y, Qj.z, c1 ? a.r32_m[1] : a.r32_m[0]),
                               make_float4(rhoj, Qj.w, csj, 0.f), Ai, Bi, Ci, Ci.y, acc, npairs);
    }
}

// R32: the sources come from the 32-byte records R (pair_entry_r32); the destination still
// reads its own A / B / C, once and coalesced
template <int K, int DIM, int MINB, int EQS, bool RANGED = false, bool R32 = false>
__global__ void __launch_bounds__(LIST_NT, MINB) k_pair_list(const PairArgs a, const uint32_t *__restrict__ cnt,
                                                            const uint32_t *__restrict__ lst, const int capg,
                                                            const uint32_t *__restrict__ chunk_ids)
{
    const int tid = threadIdx.x;
    const unsigned FULL = 0xffffffffu;
    // chunk_ids: this launch covers a subset of the CTA-sized chunks (the interior /
    // boundary split of the slab decomposition, k_chunk_classify)
    const long long s = (long long)(chunk_ids ? chunk_ids[blockIdx.x] : blockIdx.x) * LIST_NT + tid;
    bool active = s < a.n;
    float4 Ai = make_float4(0.f, 0.f, 0.f, 0.f), Bi = Ai, Ci = Ai;
    unsigned long long mask_i = 0;
    int count = 0;
    if (active) {
        Ci = a.C[s];
        const int ti = __float_as_int(Ci.w);
        mask_i = a.emask[ti & 7];
        if ((a.real_only && (ti & PT_GHOST)) || !mask_i) active = false;
        if (RANGED && active) {   // Group(start_idx, stop_idx): only these destinations of the array
            const long long li = (long long)a.perm[s] - a.doff[ti & 7];
            if (li < a.dlo[ti & 7] || li >= a.dhi[ti & 7]) active = false;
        }
    }
    if (active) {
        ld_256(a.AB + 2 * (size_t)s, Ai, Bi);
        count = (int)cnt[s];
    }
    int cmax = count;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cmax = max(cmax, __shfl_xor_sync(FULL, cmax, o));
    const uint32_t *nxt = lst + ((size_t)(s >> 5) * (size_t)capg) * 32u + (uint32_t)(s & 31);
    const float hi2 = a.k2 * Ai.w * Ai.w;
    Acc acc = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    unsigned npairs = 0;
    if constexpr (R32) {
        const unsigned bits0 = (unsigned)(mask_i >> (8 * a.r32_rep[0])) & (unsigned)(EQS & 0xFF);
        const unsigned bits1 = (unsigned)(mask_i >> (8 * a.r32_rep[1])) & (unsigned)(EQS & 0xFF);
        struct Rec { float4 P, Q; };
        list_walk<Rec>(nxt, count, cmax,
            [&](const uint32_t e, Rec &r) { ld_256(a.R + 2u * LIST_J(e), r.P, r.Q); },
            [&](const bool live, const uint32_t e, const Rec &r) {
                pair_entry_r32<K, DIM, EQS>(a, live, e, r.P, r.Q, Ai, Bi, Ci, hi2, bits0, bits1, acc, npairs);
            });
    } else {
        struct Rec { float4 A, B, C; };
        list_walk<Rec>(nxt, count, cmax,
            [&](const uint32_t e, Rec &r) { ld_rec(a, e, r.A, r.B, r.C); },
            [&](const bool live, const uint32_t e, const Rec &r) {
                pair_entry<K, DIM, EQS>(a, live, e, r.A, r.B, r.C, Ai, Bi, Ci, hi2, mask_i, acc, npairs);
            });
    }
    if (active) {
        unsigned all_bits = 0;
#pragma unroll
        for (int j = 0; j < B200SPH_MAX_ARRAYS; j++) all_bits |= (unsigned)(mask_i >> (8 * j)) & (unsigned)(EQS & 0xFF);
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
    if (a.pair_counter) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) npairs += __shfl_xor_sync(FULL, npairs, o);
        if ((tid & 31) == 0 && npairs) atomicAdd(a.pair_counter, (unsigned long long)npairs);
    }
}
