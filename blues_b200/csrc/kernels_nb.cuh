// Neighbour-list construction (K1) and the tiled direct-space pair kernel (K2).
#pragma once
#include <cooperative_groups.h>
#include "engine.cuh"

// ---------------------------------------------------------------------------------------------------------
// k_begin_eval: clear accumulators before a force evaluation, advance the noise counters (the rebuild request is
// latched by k_sort_atoms, which runs first so that reciprocal space can start before the zeroing).
//   cm_mode: 0 keep, 1 zero cm_acc[parity], 2 zero cm_acc[parity] and flip parity (single-kernel steps)
// ---------------------------------------------------------------------------------------------------------
__global__ void k_begin_eval(Dev d, int advance_noise, int advance_md, int cm_mode, int* cm_parity) {
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nthreads = (long long)gridDim.x * blockDim.x;
    const long long nf = (long long)d.R * 3 * d.N;
    for (long long i = tid; i < nf; i += nthreads) d.f_env[i] = 0;
    if (d.alch_on)
        for (long long i = tid; i < nf * ALCH_SLOTS; i += nthreads) d.f_alch[i] = 0;
    if (blockIdx.x == 0) {
        for (int i = threadIdx.x; i < d.R * N_ETERMS; i += blockDim.x) d.eacc[i] = 0;
        for (int i = threadIdx.x; i < d.R * ALCH_SLOTS * 3; i += blockDim.x) d.alch_acc[i] = 0;
        for (int i = threadIdx.x; i < d.R; i += blockDim.x) {
            Globals& g = d.g[i];
            g.noise_counter += advance_noise;
            g.md_counter += advance_md;
        }
        if (cm_mode) {
            const int p = *cm_parity;
            for (int i = threadIdx.x; i < d.R * 3; i += blockDim.x) d.cm_acc[(size_t)p * d.R * 3 + i] = 0;
            __syncthreads();
            if (cm_mode == 2 && threadIdx.x == 0) *cm_parity = p ^ 1;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// k_sort_atoms: one CTA per walker.  Deterministic counting sort of the atoms by Morton-ranked cell (cell edge >=
// half the list cutoff), atoms inside a cell ordered by topology index so that every later accumulation order —
// and therefore every float sum — is reproducible.  Builds the sorted mirrors and the inverse permutation.
// Early exit unless a rebuild was latched by k_begin_eval.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float wrap01(float f) { f -= floorf(f); return f >= 1.0f ? 0.0f : f; }

__device__ __forceinline__ void atom_cell_coords(const Dev& d, float4 p, int& cx, int& cy, int& cz) {
    // non-finite coordinates (a walker that blew up) must not index out of bounds: clamp into the grid
    cx = max(0, min((int)(wrap01(p.x * d.boxf[3]) * d.ncell[0]), d.ncell[0] - 1));
    cy = max(0, min((int)(wrap01(p.y * d.boxf[4]) * d.ncell[1]), d.ncell[1] - 1));
    cz = max(0, min((int)(wrap01(p.z * d.boxf[5]) * d.ncell[2]), d.ncell[2] - 1));
}

#ifndef SORT_CTAS
#define SORT_CTAS 16        /* CTAs of the sort cluster: 16 needs cudaFuncAttributeNonPortableClusterSizeAllowed (set at bl_create) */
#endif
#define BUILD_GROUP 8          /* atoms per k_build_list work group */
// latched = 1: the preceding k_integrate launch (IntegrateArgs::pre_eval) has latched do_rebuild and cleared the energy
// accumulators; this kernel then only handles the momentum parity (cm_mode as in k_begin_eval) and exits without a
// cluster barrier unless a rebuild is due
__global__ void __cluster_dims__(SORT_CTAS, 1, 1) __launch_bounds__(1024) k_sort_atoms(Dev d, int latched, int cm_mode, int* cm_parity) {
    // one thread-block cluster (8 CTAs, hardware cluster barrier) per walker
    namespace cg = cooperative_groups;
    cudaGridDependencySynchronize();       // programmatic dependent launch: no-op when launched without the attribute
    cg::cluster_group cluster = cg::this_cluster();
    const int r = blockIdx.y;
    Globals& g = d.g[r];
    const int cta = (int)cluster.block_rank();
    if (latched) {
        if (cm_mode && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x < 32) {
            const int p = *cm_parity;
            for (int i = threadIdx.x; i < d.R * 3; i += 32) d.cm_acc[(size_t)p * d.R * 3 + i] = 0;
            __syncwarp();
            if (cm_mode == 2 && threadIdx.x == 0) *cm_parity = p ^ 1;
        }
        if (!g.do_rebuild) return;             // uniform over the cluster, no barrier needed
    } else {
        if (cta == 0 && threadIdx.x == 0) {
            // latch: the Verlet list is rebuilt (cell sort + search) when some atom moved > skin / 2 since the last build,
            // or on request (host wrote coordinates, box changed); the alchemical pair list follows the same schedule
            g.do_rebuild = g.rebuild_request == 2 || g.prune_request;
            g.do_prune = g.do_rebuild;
            g.rebuild_request = 0;
            g.prune_request = 0;
        }
        cluster.sync();
        if (!g.do_rebuild) return;                 // uniform over the cluster
    }
    const int tid = cta * blockDim.x + threadIdx.x, nt = SORT_CTAS * blockDim.x;
    const int lane = threadIdx.x & 31, warp = tid >> 5, nwarps = nt >> 5;
    const int N = d.N, Npad = d.Npad, ncells = d.ncells;
    int* start = d.cell_start + (size_t)r * (ncells + 1);
    int* cursor = d.cell_cursor + (size_t)r * (ncells + 1);
    int* acell = d.atom_cell + (size_t)r * N;
    const float4* posq = d.posq + (size_t)r * N;
    int* orig_s = d.orig_s + (size_t)r * Npad;
    __shared__ int s_part[1024];

    for (int c = tid; c <= ncells; c += nt) cursor[c] = 0;
    cluster.sync();
    for (int a = tid; a < N; a += nt) {
        int cell = 0;
        if (d.periodic) {
            int cx, cy, cz;
            atom_cell_coords(d, posq[a], cx, cy, cz);
            cell = (cx * d.ncell[1] + cy) * d.ncell[2] + cz;       // row-major: a z-column of cells is contiguous
        }
        acell[a] = cell;
        atomicAdd(&cursor[cell], 1);
    }
    cluster.sync();
    if (cta == 0) {
        // exclusive scan of the per-cell counts by the first CTA
        const int t = threadIdx.x, n1 = blockDim.x;
        const int per = (ncells + n1 - 1) / n1;
        const int c0 = min(t * per, ncells), c1 = min(c0 + per, ncells);
        int sum = 0;
        for (int c = c0; c < c1; ++c) sum += cursor[c];
        s_part[t] = sum;
        __syncthreads();
        for (int off = 1; off < n1; off <<= 1) {
            int v = (t >= off) ? s_part[t - off] : 0;
            __syncthreads();
            s_part[t] += v;
            __syncthreads();
        }
        int run = s_part[t] - sum;
        for (int c = c0; c < c1; ++c) { int v = cursor[c]; start[c] = run; cursor[c] = run; run += v; }
        if (t == n1 - 1) start[ncells] = N;
    }
    cluster.sync();
    // scatter (arbitrary order inside a cell) ...
    for (int a = tid; a < N; a += nt) orig_s[atomicAdd(&cursor[acell[a]], 1)] = a;
    cluster.sync();
    // ... then order every cell's segment by topology index: one warp per cell, rank by counting smaller keys
    for (int c = warp; c < ncells; c += nwarps) {
        const int s0 = start[c], n = start[c + 1] - s0;
        if (n <= 1) continue;
        if (n <= 64) {
            const int v0 = lane < n ? orig_s[s0 + lane] : 0x7fffffff;
            const int v1 = lane + 32 < n ? orig_s[s0 + 32 + lane] : 0x7fffffff;
            int r0 = 0, r1 = 0;
            for (int m = 0; m < 32; ++m) {
                const int a0 = __shfl_sync(0xffffffffu, v0, m), a1 = __shfl_sync(0xffffffffu, v1, m);
                r0 += (a0 < v0) + (a1 < v0);
                r1 += (a0 < v1) + (a1 < v1);
            }
            __syncwarp();
            if (lane < n) orig_s[s0 + r0] = v0;
            if (lane + 32 < n) orig_s[s0 + r1] = v1;
        } else if (lane == 0) {
            for (int i = s0 + 1; i < s0 + n; ++i) {
                const int v = orig_s[i];
                int j = i - 1;
                while (j >= s0 && orig_s[j] > v) { orig_s[j + 1] = orig_s[j]; --j; }
                orig_s[j + 1] = v;
            }
        }
    }
    cluster.sync();
    int* rank = d.rank + (size_t)r * N;
    float4* posq_s = d.posq_s + (size_t)r * Npad;
    float2* sigeps_s = d.sigeps_s + (size_t)r * Npad;
    float4* pos_ref = d.pos_ref + (size_t)r * N;          // reference positions of the displacement test
    for (int s = tid; s < N; s += nt) {
        const int a = orig_s[s];
        rank[a] = s;
        const float4 p = posq[a];
        const float2 se = d.sigeps[a];
        posq_s[s] = p;
        sigeps_s[s] = se;
        d.mobile_s[(size_t)r * Npad + s] = d.invmass[a] > 0.0 ? 1 : 0;
        pos_ref[a] = p;
    }
    const float qnan = __int_as_float(0x7fc00000);
    for (int s = N + tid; s < Npad; s += nt) {
        posq_s[s] = make_float4(qnan, qnan, qnan, 0.f);
        sigeps_s[s] = make_float2(0.f, 0.f);
        d.mobile_s[(size_t)r * Npad + s] = 0;
        orig_s[s] = -1;
    }
    if (tid == 0) {
        g.item_overflow = 0;
        g.n_rebuilds += 1;
        g.build_cursor = 0;
    }
    if (cta == SORT_CTAS - 1) {
        // groups of <= BUILD_GROUP consecutive sorted atoms that never straddle a cell column (k_build_list works on
        // one group per warp; a group confined to a column has a compact search region)
        const int t = threadIdx.x, n1 = blockDim.x;
        const int ncols = d.periodic ? d.ncell[0] * d.ncell[1] : 1, ncz = d.periodic ? d.ncell[2] : 1;
        const int per = (ncols + n1 - 1) / n1;
        const int c0 = min(t * per, ncols), c1 = min(c0 + per, ncols);
        int sum = 0;
        for (int c = c0; c < c1; ++c) sum += (start[(c + 1) * ncz] - start[c * ncz] + BUILD_GROUP - 1) / BUILD_GROUP;
        __syncthreads();                       // s_part was last read before the previous cluster barrier
        s_part[t] = sum;
        __syncthreads();
        for (int off = 1; off < n1; off <<= 1) {
            int v = (t >= off) ? s_part[t - off] : 0;
            __syncthreads();
            s_part[t] += v;
            __syncthreads();
        }
        int run = s_part[t] - sum;
        int* groups = d.group_first + (size_t)r * d.group_capacity;
        for (int c = c0; c < c1; ++c) {
            const int s0 = start[c * ncz], n = start[(c + 1) * ncz] - s0;
            for (int k = 0; k < n; k += BUILD_GROUP) groups[run++] = (s0 + k) * 16 + min(BUILD_GROUP, n - k);
        }
        if (t == n1 - 1) g.n_groups = s_part[t];
    }
}

// ---------------------------------------------------------------------------------------------------------
// Exclusion test on topology indices: a 64-bit window mask covers partners within +-32, a sorted code list the rest.
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool pair_excluded(const Dev& d, int oi, ull wi, bool fari, int oj, bool farj) {
    if (oi < 0 || oj < 0) return false;
    int dd = oj - oi + 32;
    if ((unsigned)dd < 64u) return (wi >> dd) & 1ull;
    if (fari && farj) {
        long long code = oi < oj ? (long long)oi * d.N + oj : (long long)oj * d.N + oi;
        int lo = 0, hi = d.n_far - 1;
        while (lo <= hi) {
            int mid = (lo + hi) >> 1;
            long long v = d.far_codes[mid];
            if (v == code) return true;
            if (v < code) lo = mid + 1; else hi = mid - 1;
        }
    }
    return false;
}

// ---------------------------------------------------------------------------------------------------------
// k_build_list: Verlet list (cutoff + skin) by cell search.  Full list (i sees j and j sees i): the pair kernel needs
// no j-side force scatter and no exclusion test.
//
// Persistent single-warp CTAs fetch groups of <= 8 consecutive cell-sorted atoms (never straddling a cell column) from
// a work counter.  Lane = (atom a = lane & 7, candidate subset q = lane >> 3).  The warp walks the cell columns around
// the group's bounding box; candidates are staged 32 at a time in shared memory, already shifted to the periodic image
// that can be in range (the next chunk's loads are in flight meanwhile), and in iteration t lane (a, q) tests candidate
// 8 q + t against atom a: one LDS and ~10 ALU instructions per 32 distance tests.  Exclusions are only looked at in
// chunks that hold a candidate inside the exclusion window of a group atom (warp-uniform test), i.e. almost never.
// Survivors are appended to per-lane sub-lists in shared memory; when the group is done the warp concatenates the four
// sub-lists of every atom into its row with coalesced stores.  Scan order is fixed, hence so is the order of every
// row (reproducible float sums downstream), whichever warp happens to process the group.
// ---------------------------------------------------------------------------------------------------------
#define NL_LANES 8
#define NL_BLOCK 128
#define BUILD_SLACK 8       /* a chunk appends at most 8 entries per lane between two capacity checks */

__device__ __forceinline__ void sts_idx(unsigned int addr, unsigned short v) {
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"(v) : "memory");
}
__device__ __forceinline__ void sts_idx(unsigned int addr, int v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

#define BUILD_MAX_RUNS 64       /* a group sees at most 5 x 5 cell columns, each one run plus one periodic wrap */

// Phase 1 of a group: tabulate the runs of cell-sorted atoms that can hold neighbours — one (x, y) cell column per lane,
// its z range cut to the reach of the group's bounding box, split where it wraps — so that all cell_start loads are in
// flight together.  runs[k] = (shift x, y, z, first sorted index as bits), off[k] = candidates before run k.
__device__ __forceinline__ int build_group_runs(const Dev& d, const int* __restrict__ start, int lane, bool rx, bool ry,
                                                bool rz, int x0, int x1, int y0, int y1, int za, int zb, float lox, float hix,
                                                float loy, float hiy, float loz, float hiz, float4* runs, int* off) {
    const float bx = d.boxf[0], by = d.boxf[1], bz = d.boxf[2];
    const int ncx = d.ncell[0], ncy = d.ncell[1], ncz = d.ncell[2];
    const float ex = bx / ncx, ey = by / ncy, ez = bz / ncz;
    const float cut2 = d.list_cutoff2;
    const int nyc = y1 - y0 + 1, ncols = (x1 - x0 + 1) * nyc;       // <= 25 (checked by the caller)
    int nseg = 0, s0v[2] = {0, 0}, lenv[2] = {0, 0};
    float szv[2] = {0.f, 0.f}, sx = 0.f, sy = 0.f;
    if (lane < ncols) {
        const int rxc = x0 + lane / nyc, ryc = y0 + lane % nyc;
        int ax = rxc, ay = ryc;
        float dxc = 0.f, dyc = 0.f;
        if (!rx) {
            if (ax < 0) { ax += ncx; sx = -bx; } else if (ax >= ncx) { ax -= ncx; sx = bx; }
            dxc = fmaxf(0.f, fmaxf(rxc * ex - hix, lox - (rxc + 1) * ex));   // gap between the group and the slab
        }
        if (!ry) {
            if (ay < 0) { ay += ncy; sy = -by; } else if (ay >= ncy) { ay -= ncy; sy = by; }
            dyc = fmaxf(0.f, fmaxf(ryc * ey - hiy, loy - (ryc + 1) * ey));
        }
        const float rem2 = cut2 - dxc * dxc - dyc * dyc;
        if (rem2 > 0.f) {                                                     // else: column out of reach
            int z0 = 0, z1 = ncz - 1;
            if (!rz) {
                // both ends clamped to [za - zreach, zb + zreach]: a walker that blew up has coordinates of any magnitude, the
                // float -> int conversion then saturates and `z0 + ncz` below would wrap around
                const float zr = sqrtf(rem2);
                z0 = min(zb + d.zreach, max(za - d.zreach, (int)floorf((loz - zr) / ez)));
                z1 = max(za - d.zreach, min(zb + d.zreach, (int)floorf((hiz + zr) / ez)));
            }
            const int row = (ax * ncy + ay) * ncz;
            // at most two of the three segments exist (the z range is no longer than the column)
#pragma unroll
            for (int seg = 0; seg < 3; ++seg) {
                int a0, a1;
                float sz = 0.f;
                if (seg == 0) { a0 = max(z0, 0); a1 = min(z1, ncz - 1); }
                else if (seg == 1) { a0 = z0 + ncz; a1 = z0 < 0 ? ncz - 1 : -1; sz = -bz; }
                else { a0 = 0; a1 = z1 >= ncz ? z1 - ncz : -1; sz = bz; }
                if (a0 <= a1 && nseg < 2) {
                    const int b0 = start[row + a0], b1 = start[row + a1 + 1];
                    if (b1 > b0) { s0v[nseg] = b0; lenv[nseg] = b1 - b0; szv[nseg] = sz; ++nseg; }
                }
            }
        }
    }
    // compact the runs in column order; exclusive prefix of their lengths
    int pos = nseg, cum = lenv[0] + lenv[1];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int p2 = __shfl_up_sync(0xffffffffu, pos, o), c2 = __shfl_up_sync(0xffffffffu, cum, o);
        if (lane >= o) { pos += p2; cum += c2; }
    }
    const int nruns = __shfl_sync(0xffffffffu, pos, 31), total = __shfl_sync(0xffffffffu, cum, 31);
    pos -= nseg;
    cum -= lenv[0] + lenv[1];
    for (int j = 0; j < nseg; ++j) {
        runs[pos + j] = make_float4(sx, sy, szv[j], __int_as_float(s0v[j]));
        off[pos + j] = cum;
        cum += lenv[j];
    }
    if (lane == 0) off[nruns] = total;
    __syncwarp();
    return nruns;
}

// Phase 2: stream the candidates of all runs 32 at a time.
// Move the 32 shared-memory sub-lists to the rows of the group's atoms (coalesced stores).  Lane (a, q) holds the
// entries of atom a found among candidates 8q..8q+7 of every chunk since the last flush; a row is the sequence of
// flushes, each holding the atom's four sub-lists in subset order.  Scan order is fixed, hence so is every row.
// `done` = entries already in the row of this lane's atom (equal across the four lanes of an atom).
// Not inlined: flushes are rare (every ~30 chunks) and the chunk loop must stay lean; returns the new `done`.
template <typename IDX>
__device__ __noinline__ int build_flush(const IDX* subs, int stride, IDX* rows, int nl_M, int lane, int cnt, int done) {
    __syncwarp();
    int off = 0;
#pragma unroll
    for (int k = 1; k < 4; ++k) {
        const int c = __shfl_up_sync(0xffffffffu, cnt, 8 * k);
        if (lane >= 8 * k) off += c;
    }
    const int total = __shfl_sync(0xffffffffu, off + cnt, 24 + (lane & (BUILD_GROUP - 1)));   // lane (a, 3) knows it
    const int base = done + off;
    for (int L = 0; L < 32; ++L) {
        const int nL = __shfl_sync(0xffffffffu, cnt, L), oL = __shfl_sync(0xffffffffu, base, L);
        const IDX* src = subs + (size_t)L * stride;
        IDX* dst = rows + (size_t)(L & (BUILD_GROUP - 1)) * nl_M + oL;
        for (int k = lane; k < nL; k += 32)
            if (oL + k < nl_M) dst[k] = src[k];
    }
    __syncwarp();
    return done + total;
}

template <bool RINT, typename IDX>
__device__ __forceinline__ void build_stream(const Dev& d, const float4* __restrict__ posq_s, const int* __restrict__ orig_s,
                                             const float4* runs, const int* off, int nruns, bool rx, bool ry, bool rz,
                                             float4* cand, IDX* mysub, int cq, int lane, float4 pi, int oi, ull wi,
                                             bool fari, bool anyfar, const int (&og)[BUILD_GROUP],
                                             const unsigned int (&osp)[BUILD_GROUP], int& cnt, int& done,
                                             const IDX* subs, int stride, IDX* rows) {
    const float cut2 = d.list_cutoff2;
    const float bx = d.boxf[0], by = d.boxf[1], bz = d.boxf[2], ibx = d.boxf[3], iby = d.boxf[4], ibz = d.boxf[5];
    const float qnan = __int_as_float(0x7fc00000);
    const int q = lane >> 3;
    const unsigned int sub_addr = (unsigned int)__cvta_generic_to_shared(mysub);
    const int total = off[nruns];
    int kp = 0;                                           // run of this lane's next candidate (monotonic)
    // software pipeline: the candidates of the next chunk are requested before the current chunk is processed (deeper
    // pipelines were measured slower: the extra registers and moves cost more than the residual latency)
    float4 cnext = make_float4(qnan, qnan, qnan, 0.f);
    int ojnext = 0;
    auto fetch = [&](int c) {
        cnext = make_float4(qnan, qnan, qnan, 0.f);
        if (c < total) {
            while (c >= off[kp + 1]) ++kp;
            const float4 rn = runs[kp];
            const int s = __float_as_int(rn.w) + (c - off[kp]);
            const float4 p = posq_s[s];
            ojnext = orig_s[s];
            cnext = make_float4(p.x + rn.x, p.y + rn.y, p.z + rn.z, __int_as_float(s));   // shifted image; w = sorted index
        }
    };
    fetch(lane);
    for (int c0 = 0; c0 < total; c0 += 32) {
        bool near = false;
        {
            const float4 c = cnext;
            const int oj = ojnext;
            const bool have = c0 + lane < total;
            fetch(c0 + 32 + lane);
            if (have) {
#pragma unroll
                for (int k = 0; k < BUILD_GROUP; ++k)               // inside the exclusion window of a group atom
                    near = near || (unsigned int)(oj - og[k]) <= osp[k];
            }
            __syncwarp();
            cand[lane + (lane >> 3)] = c;                           // 8-candidate pieces, padded: conflict-free LDS
            __syncwarp();
        }
        const bool check = anyfar || __any_sync(0xffffffffu, near);   // warp-uniform
        unsigned int wp = sub_addr + (unsigned int)cnt * (unsigned int)sizeof(IDX);     // shared-space byte address
        if (!check) {
            // fast path: no candidate of this chunk can be excluded from (or be) an atom of the group.  All eight
            // candidates are loaded and measured before the first store, so the eight chains overlap; every store is
            // unconditional and only the write pointer advance is predicated.
            float r2v[8];
            int sv[8];
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                const float4 c = cand[q * 9 + t];                  // candidate 8 q + t of the chunk
                float dx = c.x - pi.x, dy = c.y - pi.y, dz = c.z - pi.z;
                if (RINT) {
                    if (rx) dx -= bx * rintf(dx * ibx);
                    if (ry) dy -= by * rintf(dy * iby);
                    if (rz) dz -= bz * rintf(dz * ibz);
                }
                r2v[t] = dx * dx + dy * dy + dz * dz;
                sv[t] = __float_as_int(c.w);
            }
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                sts_idx(wp, (IDX)sv[t]);
                wp += r2v[t] < cut2 ? (unsigned int)sizeof(IDX) : 0u;   // NaN (padding) compares false
            }
        } else {
#pragma unroll 1
            for (int t = 0; t < 8; ++t) {
                const float4 c = cand[q * 9 + t];
                float dx = c.x - pi.x, dy = c.y - pi.y, dz = c.z - pi.z;
                if (RINT) {
                    if (rx) dx -= bx * rintf(dx * ibx);
                    if (ry) dy -= by * rintf(dy * iby);
                    if (rz) dz -= bz * rintf(dz * ibz);
                }
                if (dx * dx + dy * dy + dz * dz < cut2) {
                    const int sj = __float_as_int(c.w);
                    const int oj = orig_s[sj];
                    const unsigned int dd = (unsigned int)(oj - oi + 32);
                    bool ok = true;
                    if (dd < 64u) ok = !((wi >> dd) & 1ull);           // includes the atom itself (bit 32)
                    else if (fari) ok = !pair_excluded(d, oi, wi, true, oj, d.has_far[oj]);   // rare
                    if (ok) { sts_idx(wp, (IDX)sj); wp += (unsigned int)sizeof(IDX); }
                }
            }
        }
        cnt = (int)((wp - sub_addr) / (unsigned int)sizeof(IDX));
        // a chunk appends at most 8 entries per lane: flush before any sub-list could run past its cq + BUILD_SLACK slots
        if (__any_sync(0xffffffffu, cnt > cq)) { done = build_flush<IDX>(subs, stride, rows, d.nl_M, lane, cnt, done); cnt = 0; }
    }
}

__host__ __device__ inline int build_sub_stride(int cq, int idx_bytes) {
    // entries per sub-list, rounded so that the stride in 32-bit words is odd (lanes appending at equal offsets then
    // hit different banks)
    const int words = ((cq + BUILD_SLACK) * idx_bytes + 3) / 4 | 1;
    return words * 4 / idx_bytes;
}
#define BUILD_HEAD_F4 (36 + BUILD_MAX_RUNS + (BUILD_MAX_RUNS + 4) / 4)    /* candidates, run table, run offsets */
__host__ __device__ inline size_t build_smem_bytes(int cq, int idx_bytes) {
    return BUILD_HEAD_F4 * sizeof(float4) + (size_t)32 * build_sub_stride(cq, idx_bytes) * idx_bytes;
}

template <typename IDX>
__global__ void __launch_bounds__(32) k_build_list(Dev d, int cq) {
    extern __shared__ float4 s_build[];
    float4* cand = s_build;
    const int stride = build_sub_stride(cq, (int)sizeof(IDX));
    float4* runs = s_build + 36;
    int* off = reinterpret_cast<int*>(s_build + 36 + BUILD_MAX_RUNS);
    IDX* subs = reinterpret_cast<IDX*>(s_build + BUILD_HEAD_F4);
    const int lane = threadIdx.x;
    IDX* mysub = subs + (size_t)lane * stride;
    const int N = d.N, Npad = d.Npad;
    // the CTAs are shared by all walkers of the context: each starts on walker blockIdx.x % R and moves on to the next
    // walker whose list is being rebuilt when a queue runs dry
    for (int wk = 0; wk < d.R; ++wk) {
    const int r = (blockIdx.x + wk) % d.R;
    Globals& g = d.g[r];
    if (!g.do_rebuild) continue;
    const float4* __restrict__ posq_s = d.posq_s + (size_t)r * Npad;
    const int* __restrict__ orig_s = d.orig_s + (size_t)r * Npad;
    const int* __restrict__ start = d.cell_start + (size_t)r * (d.ncells + 1);
    const int* __restrict__ groups = d.group_first + (size_t)r * d.group_capacity;
    const int n_groups = g.n_groups;
    const int a = lane & (BUILD_GROUP - 1);
    for (;;) {
        int gi = 0;
        if (lane == 0) gi = atomicAdd(&g.build_cursor, 1);
        gi = __shfl_sync(0xffffffffu, gi, 0);
        if (gi >= n_groups) break;
        const int packed = groups[gi];
        const int i0 = packed >> 4, na = packed & 15;
        const bool valid = a < na;
        const int i = valid ? i0 + a : i0;
        const float qnan = __int_as_float(0x7fc00000);
        const float4 pa = posq_s[i];
        const float4 pi = valid ? pa : make_float4(qnan, qnan, qnan, 0.f);   // idle lanes: never in range
        const int oi = orig_s[i];
        const ull wi = valid ? (d.excl_win[oi] | (1ull << 32)) : 0ull;
        const bool fari = valid ? d.has_far[oi] : false;
        const bool anyfar = __any_sync(0xffffffffu, fari);
        // exclusion window of every atom of the group as [og, og + osp] in topology indices (waters: their own molecule)
        int og[BUILD_GROUP];
        unsigned int osp[BUILD_GROUP];
        {
            const int below = valid ? 32 - (__ffsll((long long)wi) - 1) : 0, above = valid ? 31 - __clzll((long long)wi) : 0;
#pragma unroll
            for (int k = 0; k < BUILD_GROUP; ++k) {
                og[k] = __shfl_sync(0xffffffffu, oi - below, k);
                osp[k] = (unsigned int)__shfl_sync(0xffffffffu, below + above, k);
            }
        }
        int cnt = 0, done = 0;
        IDX* rows = reinterpret_cast<IDX*>(d.nl_list) + ((size_t)r * Npad + i0) * d.nl_M;
        if (!d.periodic) {
            if (lane == 0) { runs[0] = make_float4(0.f, 0.f, 0.f, __int_as_float(0)); off[0] = 0; off[1] = N; }
            __syncwarp();
            build_stream<false, IDX>(d, posq_s, orig_s, runs, off, 1, false, false, false, cand, mysub, cq, lane, pi, oi,
                                     wi, fari, anyfar, og, osp, cnt, done, subs, stride, rows);
        } else {
            const int ncx = d.ncell[0], ncy = d.ncell[1], ncz = d.ncell[2];
            // bounding box of the group, in cells and in space (idle lanes hold the first atom); a group never
            // straddles a cell column, so xa == xb and ya == yb and the search covers at most 5 x 5 columns
            int cx, cy, cz;
            atom_cell_coords(d, pa, cx, cy, cz);
            const int xa = __reduce_min_sync(0xffffffffu, cx), xb = __reduce_max_sync(0xffffffffu, cx);
            const int ya = __reduce_min_sync(0xffffffffu, cy), yb = __reduce_max_sync(0xffffffffu, cy);
            const int za = __reduce_min_sync(0xffffffffu, cz), zb = __reduce_max_sync(0xffffffffu, cz);
            const float lox = warp_min(pa.x), hix = warp_max(pa.x), loy = warp_min(pa.y), hiy = warp_max(pa.y);
            const float loz = warp_min(pa.z), hiz = warp_max(pa.z);
            // a dimension whose scan range would cover a cell twice is scanned once, with the rint() minimum image
            const bool rx = xb - xa + 5 > ncx, ry = yb - ya + 5 > ncy, rz = zb - za + 2 * d.zreach + 1 > ncz;
            const int x0 = rx ? 0 : xa - 2, x1 = rx ? ncx - 1 : xb + 2;
            const int y0 = ry ? 0 : ya - 2, y1 = ry ? ncy - 1 : yb + 2;
            const int nruns = build_group_runs(d, start, lane, rx, ry, rz, x0, x1, y0, y1, za, zb, lox, hix, loy, hiy, loz,
                                               hiz, runs, off);
            if (rx || ry || rz)
                build_stream<true, IDX>(d, posq_s, orig_s, runs, off, nruns, rx, ry, rz, cand, mysub, cq, lane, pi, oi, wi,
                                        fari, anyfar, og, osp, cnt, done, subs, stride, rows);
            else
                build_stream<false, IDX>(d, posq_s, orig_s, runs, off, nruns, false, false, false, cand, mysub, cq, lane,
                                         pi, oi, wi, fari, anyfar, og, osp, cnt, done, subs, stride, rows);
        }
        // whatever is left in the sub-lists
        const int total = build_flush<IDX>(subs, stride, rows, d.nl_M, lane, cnt, done);                                              // lanes 0..7: atoms 0..7 of the group
        if (__any_sync(0xffffffffu, total > d.nl_M)) { if (lane == 0) g.item_overflow = 1; }
        if (lane < na) d.nl_count[(size_t)r * Npad + i0 + lane] = min(total, d.nl_M);
        __syncwarp();
    }
    }
}

// ---------------------------------------------------------------------------------------------------------
// Direct-space pair kernels: Lennard-Jones + Coulomb (Ewald erfc / reaction field / plain) over the Verlet list.
// ---------------------------------------------------------------------------------------------------------
#define NB_NOCUT 0
#define NB_RF 2
#define NB_PME 4

__device__ __forceinline__ float erfc_times(float ar, float expar) {
    // Abramowitz & Stegun 7.1.26: erfc(x) = poly(t) exp(-x^2), |error| <= 1.5e-7
    const float t = __fdividef(1.0f, 1.0f + 0.3275911f * ar);
    return (0.254829592f + (-0.284496736f + (1.421413741f + (-1.453152027f + 1.061405429f * t) * t) * t) * t) * t * expar;
}

// rintf for |x| < 2^22 on the FMA pipe (two adds with the 1.5 * 2^23 constant, round-half-even like rintf, bitwise the
// same result): the XU pipe, which also serves rsqrt / rcp / ex2, is the busiest execution unit of the pair loop
__device__ __forceinline__ float rint_fma(float x) { return __fadd_rn(__fadd_rn(x, 12582912.0f), -12582912.0f); }

// ---------------------------------------------------------------------------------------------------------
// k_pair2: the pair sum of energy evaluations, and of force-only evaluations that k_pair4 does not cover.  NL_LANES
// lanes share one i-atom (register resident); a lane owns the entries part, part + NL_LANES, ... of the atom's row and
// works in trips of U = 2 entries, software pipelined: while trip t is computed the gathers of trip t + 1 and the
// index loads of trip t + 2 are in flight.  Without the pipeline, 67 % of the stall samples were long-scoreboard waits
// at the two consumers of a dependent load chain — the list index, then the gather it addresses
// (profiles/r01_final2_ncu_summary.md, source page).  j data are gathered from the cell-sorted mirrors; the partial
// forces are combined by warp shuffles in a fixed order and leave the warp as 64-bit fixed-point atomics.
// Reads may run up to two trips past the end of a row: rows are contiguous (the next row holds valid indices) and the
// array carries that much slack after the last row; such entries are masked by their position in the row.
// EWALD 1: real-space Ewald force from the polynomial of Dev::ewk (no MUFU.EX2 / MUFU.RCP: the XU pipe is the busiest
// unit of the pair loop); energies, on the steps that need them, still come from erfc.
// ---------------------------------------------------------------------------------------------------------
#define PAIR_SLACK_ENTRIES 512
// volatile so that the loads of the NEXT trips keep their place at the top of the loop body (the compiler otherwise
// sinks them to the bottom, next to their consumers in the following iteration, and the latency is exposed again)
__device__ __forceinline__ float4 ldg_nc_f4(const float4* p) {
    float4 v;
    asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ float2 ldg_nc_f2(const float2* p) {
    float2 v;
    asm volatile("ld.global.nc.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ int ldg_nc_idx(const unsigned short* p) {
    unsigned short v;
    asm volatile("ld.global.nc.u16 %0, [%1];" : "=h"(v) : "l"(p));
    return (int)v;
}
__device__ __forceinline__ int ldg_nc_idx(const int* p) {
    int v;
    asm volatile("ld.global.nc.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
// one trip: U entries of this lane, data already in registers
template <int METHOD, bool ENERGY, int U, int EWALD>
__device__ __forceinline__ void pair_trip(const Dev& d, const float4 (&pc)[U], const float2 (&ec)[U], int first, int nm,
                                          const float4 pi, const float2 se_i, float qi, float cut2, float& fx, float& fy,
                                          float& fz, float& etot) {
    const float bx = d.boxf[0], by = d.boxf[1], bz = d.boxf[2];
    const float ibx = d.boxf[3], iby = d.boxf[4], ibz = d.boxf[5];
#pragma unroll
    for (int u = 0; u < U; ++u) {
        const float4 pj = pc[u];
        const float2 se_j = ec[u];
        float dx = pi.x - pj.x, dy = pi.y - pj.y, dz = pi.z - pj.z;
        if (METHOD != NB_NOCUT) {
            dx -= bx * rint_fma(dx * ibx);
            dy -= by * rint_fma(dy * iby);
            dz -= bz * rint_fma(dz * ibz);
        }
        const float r2 = dx * dx + dy * dy + dz * dz;
        const bool inr = (first + u < nm) && (r2 < cut2);
        const float invr = rsqrtf(r2);
        const float invr2 = invr * invr;
        const float sig = se_i.x + se_j.x;
        const float s2 = sig * sig * invr2;
        const float s6 = s2 * s2 * s2;
        const float eps4 = se_i.y * se_j.y;
        float de = eps4 * (12.0f * s6 * s6 - 6.0f * s6) * invr2;
        const float qq = qi * pj.w;
        float e = 0.f;
        if (METHOD == NB_PME) {
            if (EWALD == 1) {
                const float tt = fmaf(r2, d.ewk_scale, -1.0f);
                float k = d.ewk[EWK_DEG];
#pragma unroll
                for (int c = EWK_DEG - 1; c >= 0; --c) k = fmaf(k, tt, d.ewk[c]);
                de += qq * fmaf(-d.alpha3, k, invr * invr2);
                if (ENERGY) {
                    const float ar = d.alpha * r2 * invr;
                    e = eps4 * (s6 * s6 - s6) + qq * invr * erfc_times(ar, __expf(-ar * ar));
                }
            } else {
                const float ar = d.alpha * r2 * invr;
                const float ex = __expf(-ar * ar);
                const float ec2 = erfc_times(ar, ex);
                de += qq * invr * (ec2 + (float)TWO_OVER_SQRT_PI * ar * ex) * invr2;
                if (ENERGY) e = eps4 * (s6 * s6 - s6) + qq * invr * ec2;
            }
        } else if (METHOD == NB_RF) {
            de += qq * (invr - 2.0f * d.krf * r2) * invr2;
            if (ENERGY) e = eps4 * (s6 * s6 - s6) + qq * (invr + d.krf * r2 - d.crf);
        } else {
            de += qq * invr * invr2;
            if (ENERGY) e = eps4 * (s6 * s6 - s6) + qq * invr;
        }
        // select, not a mask multiply: entries past the end of the row or in the skin shell may be anything
        de = inr ? de : 0.f;
        fx += dx * de; fy += dy * de; fz += dz * de;
        if (ENERGY) etot += inr ? e : 0.f;
    }
}

template <int METHOD, bool ENERGY, typename IDX, int EWALD>
__global__ void __launch_bounds__(NL_BLOCK) k_pair2(Dev d, int skip_frozen) {
    constexpr int LANES = NL_LANES, U = 2;
    const int r = blockIdx.y;
    const int lane = threadIdx.x & 31;
    const int part = lane & (LANES - 1);
    const int i = (blockIdx.x * NL_BLOCK + threadIdx.x) / LANES;
    const int N = d.N, Npad = d.Npad;
    if (i >= Npad) return;
    // the force on an atom without mass moves nothing: inside a step program its row is not evaluated (full lists: the
    // forces it exerts on its mobile neighbours come from THEIR rows); host force queries and energy launches pass 0
    if (skip_frozen && !d.mobile_s[(size_t)r * Npad + i]) return;
    const float4* __restrict__ posq_s = d.posq_s + (size_t)r * Npad;
    const float2* __restrict__ sigeps_s = d.sigeps_s + (size_t)r * Npad;
    const IDX* __restrict__ lp = reinterpret_cast<const IDX*>(d.nl_list) + ((size_t)r * Npad + i) * d.nl_M + part;
    const int cnt = d.nl_count[(size_t)r * Npad + i];
    const int nm = cnt > part ? (cnt - part + LANES - 1) / LANES : 0;        // entries owned by this lane
    const int ntrip = (nm + U - 1) / U;
    const float cut2 = METHOD == NB_NOCUT ? 3.0e38f : d.cutoff2;
    const float4 pi = posq_s[i];
    const float2 se_i = sigeps_s[i];
    const float qi = pi.w * (float)ONE_4PI_EPS0;
    float fx = 0.f, fy = 0.f, fz = 0.f, etot = 0.f;
    // two buffers of gathered data (trips t, t + 1 in flight or in use) and two of indices (trips t + 2, t + 3)
    int iA[U], iB[U];
    float4 pA[U], pB[U];
    float2 eA[U], eB[U];
#pragma unroll
    for (int u = 0; u < U; ++u) { iA[u] = ldg_nc_idx(lp + LANES * u); iB[u] = ldg_nc_idx(lp + LANES * (U + u)); }
#pragma unroll
    for (int u = 0; u < U; ++u) { pA[u] = ldg_nc_f4(posq_s + iA[u]); eA[u] = ldg_nc_f2(sigeps_s + iA[u]); }
#pragma unroll
    for (int u = 0; u < U; ++u) { pB[u] = ldg_nc_f4(posq_s + iB[u]); eB[u] = ldg_nc_f2(sigeps_s + iB[u]); }
#pragma unroll
    for (int u = 0; u < U; ++u) { iA[u] = ldg_nc_idx(lp + LANES * (2 * U + u)); iB[u] = ldg_nc_idx(lp + LANES * (3 * U + u)); }
    for (int t = 0; t < ntrip; t += 2) {
        pair_trip<METHOD, ENERGY, U, EWALD>(d, pA, eA, t * U, nm, pi, se_i, qi, cut2, fx, fy, fz, etot);
#pragma unroll
        for (int u = 0; u < U; ++u) { pA[u] = ldg_nc_f4(posq_s + iA[u]); eA[u] = ldg_nc_f2(sigeps_s + iA[u]); }
#pragma unroll
        for (int u = 0; u < U; ++u) iA[u] = ldg_nc_idx(lp + LANES * ((t + 4) * U + u));
        pair_trip<METHOD, ENERGY, U, EWALD>(d, pB, eB, (t + 1) * U, nm, pi, se_i, qi, cut2, fx, fy, fz, etot);
#pragma unroll
        for (int u = 0; u < U; ++u) { pB[u] = ldg_nc_f4(posq_s + iB[u]); eB[u] = ldg_nc_f2(sigeps_s + iB[u]); }
#pragma unroll
        for (int u = 0; u < U; ++u) iB[u] = ldg_nc_idx(lp + LANES * ((t + 5) * U + u));
    }
#pragma unroll
    for (int o = LANES / 2; o > 0; o >>= 1) {
        fx += __shfl_xor_sync(0xffffffffu, fx, o);
        fy += __shfl_xor_sync(0xffffffffu, fy, o);
        fz += __shfl_xor_sync(0xffffffffu, fz, o);
    }
    if (part == 0 && i < N) {
        const int oi = d.orig_s[(size_t)r * Npad + i];
        long long* fenv = d.f_env + (size_t)r * 3 * N;
        fx_addf(&fenv[oi], fx, (float)FORCE_SCALE);
        fx_addf(&fenv[N + oi], fy, (float)FORCE_SCALE);
        fx_addf(&fenv[2 * N + oi], fz, (float)FORCE_SCALE);
    }
    if (ENERGY) {
        // every pair appears in both atoms' lists
        const float e = warp_sum(etot);
        if (lane == 0 && e != 0.f) fx_add(&d.eacc[r * N_ETERMS + E_PAIR], 0.5 * (double)e, ENERGY_SCALE);
    }
}

// ---------------------------------------------------------------------------------------------------------
// k_pair4: k_pair2's pipeline with the arithmetic of TWO list entries per instruction — Blackwell's packed FP32 pair
// operations (PTX add/mul/fma .f32x2 → SASS FADD2 / FMUL2 / FFMA2 on 64-bit register pairs).  ncu on k_pair2
// (profiles/r02a_*): 71 issue slots per entry, 52 of them FP32, issue-bound at 72 % of the slots; the packed form needs
// ~26 FP32 slots per entry, so the loop becomes bound by the FP32 pipe itself.  The two entries of a trip sit in the
// low / high halves; the scalar results that feed a pair (coordinate differences, rsqrt, per-atom parameters) are
// written by scalar instructions into adjacent registers, which ptxas pairs without moves.  PME, forces only, polynomial
// Ewald kernel of degree DEG (Dev::ewk2, fitted at bl_create: 10 up to (alpha rc)^2 = 4.8, 12 beyond — float rounding,
// not the fit, limits both).  Energy steps and the other methods use k_pair2.
// ---------------------------------------------------------------------------------------------------------
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 f2_pack(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void f2_unpack(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 f2_fma(f32x2 a, f32x2 b, f32x2 c) { f32x2 r; asm("fma.rn.ftz.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ f32x2 f2_mul(f32x2 a, f32x2 b) { f32x2 r; asm("mul.rn.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f32x2 f2_add(f32x2 a, f32x2 b) { f32x2 r; asm("add.rn.ftz.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f32x2 f2_dup(float v) { return f2_pack(v, v); }

struct PairAcc2 { f32x2 fx, fy, fz; };

// two entries (p0, e0), (p1, e1) of one i-atom; in0 / in1: the entry lies inside the row
template <int DEG>
__device__ __forceinline__ void pair_trip_x2(const Dev& d, const float4 p0, const float2 e0, const float4 p1, const float2 e1,
                                             bool in0, bool in1, const float4 pi, const float2 se_i, float qi, float cut2,
                                             PairAcc2& acc) {
    const f32x2 magic = f2_dup(12582912.0f), nmagic = f2_dup(-12582912.0f);
    f32x2 dx = f2_pack(pi.x - p0.x, pi.x - p1.x);
    f32x2 dy = f2_pack(pi.y - p0.y, pi.y - p1.y);
    f32x2 dz = f2_pack(pi.z - p0.z, pi.z - p1.z);
    // minimum image: n = rint(d / L) by the 1.5 * 2^23 trick (the product and the first add fused), d -= L n
    dx = f2_fma(f2_dup(-d.boxf[0]), f2_add(f2_fma(dx, f2_dup(d.boxf[3]), magic), nmagic), dx);
    dy = f2_fma(f2_dup(-d.boxf[1]), f2_add(f2_fma(dy, f2_dup(d.boxf[4]), magic), nmagic), dy);
    dz = f2_fma(f2_dup(-d.boxf[2]), f2_add(f2_fma(dz, f2_dup(d.boxf[5]), magic), nmagic), dz);
    const f32x2 r2 = f2_fma(dz, dz, f2_fma(dy, dy, f2_mul(dx, dx)));
    float r2a, r2b;
    f2_unpack(r2, r2a, r2b);
    in0 = in0 && (r2a < cut2);
    in1 = in1 && (r2b < cut2);
    const f32x2 invr = f2_pack(rsqrtf(r2a), rsqrtf(r2b));
    const f32x2 invr2 = f2_mul(invr, invr);
    const f32x2 sig = f2_pack(se_i.x + e0.x, se_i.x + e1.x);
    const f32x2 s2 = f2_mul(f2_mul(sig, sig), invr2);
    const f32x2 s6 = f2_mul(f2_mul(s2, s2), s2);
    const f32x2 eps4 = f2_pack(se_i.y * e0.y, se_i.y * e1.y);
    // eps4 (12 s6^2 - 6 s6) / r^2
    f32x2 de = f2_mul(f2_mul(eps4, f2_mul(s6, f2_fma(s6, f2_dup(12.0f), f2_dup(-6.0f)))), invr2);
    const f32x2 qq = f2_pack(qi * p0.w, qi * p1.w);
    const f32x2 tt = f2_fma(r2, f2_dup(d.ewk_scale), f2_dup(-1.0f));
    f32x2 k = f2_dup(d.ewk2[DEG]);
#pragma unroll
    for (int c = DEG - 1; c >= 0; --c) k = f2_fma(k, tt, f2_dup(d.ewk2[c]));
    de = f2_fma(qq, f2_fma(f2_dup(-d.alpha3), k, f2_mul(invr, invr2)), de);
    float dea, deb;
    f2_unpack(de, dea, deb);
    // select, not a mask multiply: entries past the end of the row or in the skin shell may be anything
    de = f2_pack(in0 ? dea : 0.f, in1 ? deb : 0.f);
    acc.fx = f2_fma(dx, de, acc.fx);
    acc.fy = f2_fma(dy, de, acc.fy);
    acc.fz = f2_fma(dz, de, acc.fz);
}

#ifdef PAIR4_MIN_CTAS            /* experiment hook: cap the registers for more resident warps (measured: see DESIGN.md §11) */
#define PAIR4_BOUNDS __launch_bounds__(NL_BLOCK, PAIR4_MIN_CTAS)
#else
#define PAIR4_BOUNDS __launch_bounds__(NL_BLOCK)
#endif
template <typename IDX, int LANES, int U, int DEG>
__global__ void PAIR4_BOUNDS k_pair4(Dev d, int skip_frozen, int phase) {
    static_assert(U % 2 == 0, "entries are processed in packed pairs");
    const int r = blockIdx.y;
    // phase 1: only the walkers whose list is NOT being rebuilt in this evaluation (launched beside the builder, on its own
    // stream); phase 2: only the walkers whose list has just been rebuilt; 0: all
    if (phase != 0 && (d.g[r].do_rebuild != 0) != (phase == 2)) return;
    const int lane = threadIdx.x & 31;
    const int part = lane & (LANES - 1);
    const int N = d.N, Npad = d.Npad;
    // a launch with fewer CTAs than row blocks (BLUES_B200_PAIR_PER_SM: a bounded number of resident CTAs per SM, so that
    // the short kernels of the reciprocal-space chain find room beside it) walks the blocks with a grid stride
    for (int blk = blockIdx.x; blk * (NL_BLOCK / LANES) < Npad; blk += gridDim.x) {
    const int i = (blk * NL_BLOCK + threadIdx.x) / LANES;
    if (i >= Npad) continue;
    if (skip_frozen && !d.mobile_s[(size_t)r * Npad + i]) continue;      // (see k_pair2)
    const float4* __restrict__ posq_s = d.posq_s + (size_t)r * Npad;
    const float2* __restrict__ sigeps_s = d.sigeps_s + (size_t)r * Npad;
    const IDX* __restrict__ lp = reinterpret_cast<const IDX*>(d.nl_list) + ((size_t)r * Npad + i) * d.nl_M + part;
    const int cnt = d.nl_count[(size_t)r * Npad + i];
    const int nm = cnt > part ? (cnt - part + LANES - 1) / LANES : 0;        // entries owned by this lane
    const int ntrip = (nm + U - 1) / U;
    const float cut2 = d.cutoff2;
    const float4 pi = posq_s[i];
    const float2 se_i = sigeps_s[i];
    const float qi = pi.w * (float)ONE_4PI_EPS0;
    PairAcc2 acc;
    acc.fx = acc.fy = acc.fz = f2_dup(0.f);
    // the same two-deep software pipeline as k_pair2: gathers of trip t + 1 and index loads of trips t + 2, t + 3 in flight
    int iA[U], iB[U];
    float4 pA[U], pB[U];
    float2 eA[U], eB[U];
#pragma unroll
    for (int u = 0; u < U; ++u) { iA[u] = ldg_nc_idx(lp + LANES * u); iB[u] = ldg_nc_idx(lp + LANES * (U + u)); }
#pragma unroll
    for (int u = 0; u < U; ++u) { pA[u] = ldg_nc_f4(posq_s + iA[u]); eA[u] = ldg_nc_f2(sigeps_s + iA[u]); }
#pragma unroll
    for (int u = 0; u < U; ++u) { pB[u] = ldg_nc_f4(posq_s + iB[u]); eB[u] = ldg_nc_f2(sigeps_s + iB[u]); }
#pragma unroll
    for (int u = 0; u < U; ++u) { iA[u] = ldg_nc_idx(lp + LANES * (2 * U + u)); iB[u] = ldg_nc_idx(lp + LANES * (3 * U + u)); }
    for (int t = 0; t < ntrip; t += 2) {
#pragma unroll
        for (int u = 0; u < U; u += 2)
            pair_trip_x2<DEG>(d, pA[u], eA[u], pA[u + 1], eA[u + 1], t * U + u < nm, t * U + u + 1 < nm, pi, se_i, qi, cut2, acc);
#pragma unroll
        for (int u = 0; u < U; ++u) { pA[u] = ldg_nc_f4(posq_s + iA[u]); eA[u] = ldg_nc_f2(sigeps_s + iA[u]); }
#pragma unroll
        for (int u = 0; u < U; ++u) iA[u] = ldg_nc_idx(lp + LANES * ((t + 4) * U + u));
#pragma unroll
        for (int u = 0; u < U; u += 2)
            pair_trip_x2<DEG>(d, pB[u], eB[u], pB[u + 1], eB[u + 1], (t + 1) * U + u < nm, (t + 1) * U + u + 1 < nm, pi, se_i, qi, cut2, acc);
#pragma unroll
        for (int u = 0; u < U; ++u) { pB[u] = ldg_nc_f4(posq_s + iB[u]); eB[u] = ldg_nc_f2(sigeps_s + iB[u]); }
#pragma unroll
        for (int u = 0; u < U; ++u) iB[u] = ldg_nc_idx(lp + LANES * ((t + 5) * U + u));
    }
    float fx, fy, fz, hx, hy, hz;
    f2_unpack(acc.fx, fx, hx); f2_unpack(acc.fy, fy, hy); f2_unpack(acc.fz, fz, hz);
    fx += hx; fy += hy; fz += hz;
#pragma unroll
    for (int o = LANES / 2; o > 0; o >>= 1) {
        fx += __shfl_xor_sync(0xffffffffu, fx, o);
        fy += __shfl_xor_sync(0xffffffffu, fy, o);
        fz += __shfl_xor_sync(0xffffffffu, fz, o);
    }
    if (part == 0 && i < N) {
        const int oi = d.orig_s[(size_t)r * Npad + i];
        long long* fenv = d.f_env + (size_t)r * 3 * N;
        fx_addf(&fenv[oi], fx, (float)FORCE_SCALE);
        fx_addf(&fenv[N + oi], fy, (float)FORCE_SCALE);
        fx_addf(&fenv[2 * N + oi], fz, (float)FORCE_SCALE);
    }
    }
}

// ---------------------------------------------------------------------------------------------------------
// k_neighbor_pairs: enumerate (for tests) the non-excluded pairs within the cutoff found through the Verlet list.
// ---------------------------------------------------------------------------------------------------------
template <typename IDX>
__global__ void k_neighbor_pairs(Dev d, int r, long long* codes, unsigned long long capacity, unsigned long long* n_out) {
    const int Npad = d.Npad;
    const float4* posq_s = d.posq_s + (size_t)r * Npad;
    const int* orig_s = d.orig_s + (size_t)r * Npad;
    const float bx = d.boxf[0], by = d.boxf[1], bz = d.boxf[2];
    const float ibx = d.boxf[3], iby = d.boxf[4], ibz = d.boxf[5];
    const float cut2 = d.periodic ? d.cutoff2 : 3.0e38f;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < d.N; i += gridDim.x * blockDim.x) {
        const float4 pi = posq_s[i];
        const int oi = orig_s[i];
        const IDX* list = reinterpret_cast<const IDX*>(d.nl_list) + ((size_t)r * Npad + i) * d.nl_M;
        const int cnt = d.nl_count[(size_t)r * Npad + i];
        for (int k = 0; k < cnt; ++k) {
            const int s = (int)list[k];
            const int oj = orig_s[s];
            if (oj < oi) continue;                       // full list: report each pair once
            const float4 pj = posq_s[s];
            float dx = pi.x - pj.x, dy = pi.y - pj.y, dz = pi.z - pj.z;
            if (d.periodic) {
                dx -= bx * rintf(dx * ibx);
                dy -= by * rintf(dy * iby);
                dz -= bz * rintf(dz * ibz);
            }
            if (dx * dx + dy * dy + dz * dz < cut2) {
                unsigned long long slot = atomicAdd(n_out, 1ull);
                if (slot < capacity) codes[slot] = (long long)oi * d.N + oj;
            }
        }
    }
}
