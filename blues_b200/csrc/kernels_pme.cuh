// Smooth particle-mesh Ewald reciprocal space (K4 spread, K5 convolution, K6 gather) around cuFFT.
// Order-5 cardinal B-splines; weight of grid point base+k is M5(frac + 4 - k) (same convention as the oracle).
#pragma once
#include <cooperative_groups.h>
#include "engine.cuh"

// M5 weights and derivatives at fractional offset w in [0,1): out[k] = M5(w + 4 - k), dout[k] = M5'(w + 4 - k)
__device__ __forceinline__ void bspline5(float w, float* out, float* dout) {
    // build orders 2..5 by the standard recursion on the array a[k] = M_n(w + k), k = 0..n-1
    float a[PME_ORDER];
    a[0] = w; a[1] = 1.0f - w; a[2] = 0.f; a[3] = 0.f; a[4] = 0.f;      // order 2: M2(w), M2(w+1)
    float da[PME_ORDER];
#pragma unroll
    for (int n = 3; n <= PME_ORDER; ++n) {
        if (n == PME_ORDER) {
            // derivative of order n from order n-1: M_n'(u) = M_{n-1}(u) - M_{n-1}(u-1)
            da[0] = a[0];
#pragma unroll
            for (int k = 1; k < PME_ORDER - 1; ++k) da[k] = a[k] - a[k - 1];
            da[PME_ORDER - 1] = -a[PME_ORDER - 2];
        }
        const float div = 1.0f / (float)(n - 1);
        // M_n(u) = [u M_{n-1}(u) + (n-u) M_{n-1}(u-1)] / (n-1), with u = w + k
#pragma unroll
        for (int k = n - 1; k >= 0; --k) {
            float u = w + (float)k;
            float lo = (k < n - 1) ? a[k] : 0.f;          // M_{n-1}(u)   (zero for u >= n-1)
            float hi = (k > 0) ? a[k - 1] : 0.f;          // M_{n-1}(u-1)
            a[k] = div * (u * lo + ((float)n - u) * hi);
        }
    }
#pragma unroll
    for (int k = 0; k < PME_ORDER; ++k) {
        out[k] = a[PME_ORDER - 1 - k];
        dout[k] = da[PME_ORDER - 1 - k];
    }
}

__device__ __forceinline__ void pme_atom_setup(const Dev& d, float4 p, int* base, float* frac) {
    float fx = p.x * d.boxf[3], fy = p.y * d.boxf[4], fz = p.z * d.boxf[5];
    fx -= floorf(fx); fy -= floorf(fy); fz -= floorf(fz);
    float ux = fx * d.gx, uy = fy * d.gy, uz = fz * d.gz;
    int ix = (int)ux, iy = (int)uy, iz = (int)uz;
    frac[0] = ux - ix; frac[1] = uy - iy; frac[2] = uz - iz;
    base[0] = ix >= d.gx ? ix - d.gx : ix;
    base[1] = iy >= d.gy ? iy - d.gy : iy;
    base[2] = iz >= d.gz ? iz - d.gz : iz;
}

// k_pme_spread: one CTA per x-plane of the charge grid (and walker).  The plane (gy x gz points) lives in shared
// memory as 32-bit fixed point; the CTA walks the atoms whose order-5 stencil can touch the plane — a contiguous run
// of the cell-sorted mirror, because cells are ordered with x slowest — and accumulates with shared-memory integer
// atomics (order independent → deterministic).  The finished plane is written once, as float: no global atomics,
// no separate conversion pass.
#define SPREAD_SCALE 8388608.0f            /* 2^23 */
#define SPREAD_MAX_RUNS 64
// gridDim.y = CTAs per x-plane, each owning a band of y-rows.  More, smaller bands shorten the kernel when one walker
// leaves the device mostly idle (latency bound); fewer bands recompute fewer B-splines when many walkers fill it.  At
// <= 2 walkers the host picks the band count that makes the launch ONE wave of one CTA per SM (24 planes x 6 bands = 144
// CTAs on 148 SMs: 21 us; 8 bands = 192 CTAs ran as two unequal waves: 27 us).
//
// Frozen atoms (use_cache, Dev::grid_frozen): the sums are integers, so "frozen share + mobile share" is bit for bit the
// plane a launch over all atoms produces.  State 0 of the walker: this launch accumulates the two shares separately
// (second shared plane), stores the frozen one and k_pme_gather* flips the state once the whole grid is done; state 1:
// the plane starts from the stored share and frozen atoms are skipped after a one-byte load.
template <int SPREAD_THREADS>
__global__ void __launch_bounds__(SPREAD_THREADS) k_pme_spread(Dev d, int use_cache) {
    extern __shared__ int s_plane[];            // [rows * gz] (+ the same again for the frozen share in state 0)
    __shared__ int s_run0[SPREAD_MAX_RUNS], s_runoff[SPREAD_MAX_RUNS + 1];
    const int r = blockIdx.z, plane = blockIdx.x, part = blockIdx.y;
    const int ysplit = (int)gridDim.y;                          // CTAs per x-plane, each owning a band of y-rows
    const int ya = part * d.gy / ysplit, yb = (part + 1) * d.gy / ysplit;   // rows [ya, yb)
    const int npts = (yb - ya) * d.gz;
    const int cstate = use_cache ? d.frozen_grid_state[r] : -1;            // -1: no cache, 0: fill it, 1: use it
    int* s_frozen = s_plane + npts;
    int* cache = use_cache ? d.grid_frozen + (size_t)r * d.gsize + ((size_t)plane * d.gy + ya) * d.gz : nullptr;
    const unsigned char* __restrict__ mobile_s = d.mobile_s + (size_t)r * d.Npad;
    if (cstate == 1) for (int k = threadIdx.x; k < npts; k += blockDim.x) s_plane[k] = cache[k];
    else for (int k = threadIdx.x; k < npts; k += blockDim.x) { s_plane[k] = 0; if (cstate == 0) s_frozen[k] = 0; }
    const float4* __restrict__ posq_s = d.posq_s + (size_t)r * d.Npad;
    const int* __restrict__ start = d.cell_start + (size_t)r * (d.ncells + 1);
    const int ncx = d.ncell[0], ncy = d.ncell[1], ncz = d.ncell[2];
    // atoms with base_x in [plane-4, plane] and base_y in [ya-4, yb-1]: the cell columns that cover those fractional
    // ranges, plus one cell of margin each side because the sorted order is only refreshed with the neighbour list
    int cxa = (int)floorf((float)(plane - 4) / d.gx * ncx) - 1;
    int cxb = (int)floorf((float)(plane + 1) / d.gx * ncx) + 1;
    if (cxb - cxa + 1 >= ncx) { cxa = 0; cxb = ncx - 1; }
    int cya = (int)floorf((float)(ya - 4) / d.gy * ncy) - 1;
    int cyb = (int)floorf((float)yb / d.gy * ncy) + 1;
    if (cyb - cya + 1 >= ncy) { cya = 0; cyb = ncy - 1; }
    // for one cell-plane cx the columns cya..cyb are contiguous in the sorted order (two runs when the range wraps);
    // the runs are tabulated first so that the atom loop below is one flat, latency-tolerant index space
    const int nruns = min(2 * (cxb - cxa + 1), SPREAD_MAX_RUNS);
    if (threadIdx.x < nruns) {
        const int run = threadIdx.x;
        const int cx = (((cxa + (run >> 1)) % ncx) + ncx) % ncx;
        int c0 = 0, c1 = -1;                              // y-cell range [c0, c1] of this run, not wrapped
        if ((run & 1) == 0) { c0 = max(cya, 0); c1 = min(cyb, ncy - 1); }
        else if (cya < 0) { c0 = cya + ncy; c1 = ncy - 1; }
        else if (cyb >= ncy) { c0 = 0; c1 = cyb - ncy; }
        int s0 = 0, n = 0;
        if (c0 <= c1) { s0 = start[(cx * ncy + c0) * ncz]; n = start[(cx * ncy + c1 + 1) * ncz] - s0; }
        s_run0[run] = s0;
        s_runoff[run + 1] = n;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        s_runoff[0] = 0;
        for (int k = 0; k < nruns; ++k) s_runoff[k + 1] += s_runoff[k];
    }
    __syncthreads();
    const int total = s_runoff[nruns];
    {
        int run = 0;
        for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
            while (idx >= s_runoff[run + 1]) ++run;
            const int s = s_run0[run] + (idx - s_runoff[run]);
            int* dst = s_plane;
            if (cstate >= 0 && !mobile_s[s]) {
                if (cstate == 1) continue;
                dst = s_frozen;
            }
            const float4 p = posq_s[s];
            if (p.w == 0.f) continue;
            int base[3];
            float frac[3];
            pme_atom_setup(d, p, base, frac);
            int i = plane - base[0];
            if (i < 0) i += d.gx;
            if (i >= PME_ORDER) continue;
            // y-rows of the stencil that fall into this CTA's band
            int jrow[PME_ORDER];
            bool any = false;
#pragma unroll
            for (int j = 0; j < PME_ORDER; ++j) {
                int gy = base[1] + j; gy -= gy >= d.gy ? d.gy : 0;
                jrow[j] = (gy >= ya && gy < yb) ? gy - ya : -1;
                any = any || jrow[j] >= 0;
            }
            if (!any) continue;
            float wx[PME_ORDER], wy[PME_ORDER], wz[PME_ORDER], dw[PME_ORDER];
            bspline5(frac[0], wx, dw);
            bspline5(frac[1], wy, dw);
            bspline5(frac[2], wz, dw);
            float qx = 0.f;
#pragma unroll
            for (int k = 0; k < PME_ORDER; ++k) qx = (k == i) ? p.w * wx[k] : qx;
            qx *= SPREAD_SCALE;
#pragma unroll
            for (int j = 0; j < PME_ORDER; ++j) {
                if (jrow[j] < 0) continue;
                const float qxy = qx * wy[j];
#pragma unroll
                for (int k = 0; k < PME_ORDER; ++k) {
                    int gz = base[2] + k; gz -= gz >= d.gz ? d.gz : 0;
                    atomicAdd(&dst[jrow[j] * d.gz + gz], __float2int_rn(qxy * wz[k]));
                }
            }
        }
    }
    __syncthreads();
    float* out = d.grid_r + (size_t)r * d.gsize + ((size_t)plane * d.gy + ya) * d.gz;
    if (cstate == 0) {
        for (int k = threadIdx.x; k < npts; k += blockDim.x) {
            cache[k] = s_frozen[k];
            out[k] = (float)(s_plane[k] + s_frozen[k]) * (1.0f / SPREAD_SCALE);
        }
    } else {
        for (int k = threadIdx.x; k < npts; k += blockDim.x) out[k] = (float)s_plane[k] * (1.0f / SPREAD_SCALE);
    }
}

// multiply the transformed charge grid by the influence function; optional energy
template <bool ENERGY>
__global__ void __launch_bounds__(256) k_pme_convolve(Dev d) {
    const int r = blockIdx.y;
    const int nzc = d.gz / 2 + 1;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    double e = 0.0;
    if (idx < d.csize) {
        const int kz = idx % nzc;
        const int ky = (idx / nzc) % d.gy;
        const int kx = idx / (nzc * d.gy);
        float2 c = d.grid_c[(size_t)r * d.csize + idx];
        float eterm = 0.f;
        if (idx != 0) {
            const int mx = kx <= d.gx / 2 ? kx : kx - d.gx;
            const int my = ky <= d.gy / 2 ? ky : ky - d.gy;
            const float fx = mx * d.boxf[3], fy = my * d.boxf[4], fz = kz * d.boxf[5];
            const float m2 = fx * fx + fy * fy + fz * fz;
            const float V = d.boxf[0] * d.boxf[1] * d.boxf[2];
            const float denom = m2 * d.bmod_x[kx] * d.bmod_y[ky] * d.bmod_z[kz] * 3.14159265358979f * V;
            const float pi2_over_a2 = 9.8696044010893586f / (d.alpha * d.alpha);
            eterm = (float)ONE_4PI_EPS0 * expf(-pi2_over_a2 * m2) / denom;
        }
        if (ENERGY) {
            // half-spectrum weights: planes kz = 0 and (even gz) kz = gz/2 count once, all others twice
            const double w = (kz == 0 || (2 * kz == d.gz)) ? 1.0 : 2.0;
            e = 0.5 * w * (double)eterm * ((double)c.x * c.x + (double)c.y * c.y);
        }
        c.x *= eterm;
        c.y *= eterm;
        d.grid_c[(size_t)r * d.csize + idx] = c;
    }
    if (ENERGY) {
        e = warp_sum(e);
        if ((threadIdx.x & 31) == 0 && e != 0.0) fx_add(&d.eacc[r * N_ETERMS + E_PME], e, ENERGY_SCALE);
    }
}

// skip_frozen: forces on atoms of mass 0 are not needed (an evaluation inside the integrator program; blues/simulation.py:
// 364-480 freezes by zeroing masses).  The first thread also marks the frozen share of the charge grid as stored — the
// whole spread launch that wrote it has finished by the time any gather thread runs.
__global__ void __launch_bounds__(128) k_pme_gather(Dev d, int skip_frozen) {
    const int r = blockIdx.y;
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a == 0 && d.grid_frozen) d.frozen_grid_state[r] = 1;
    if (a >= d.N) return;
    if (skip_frozen && d.mass[a] == 0.0) return;
    const float4 p = d.posq[(size_t)r * d.N + a];
    if (p.w == 0.f) return;
    int base[3];
    float frac[3];
    pme_atom_setup(d, p, base, frac);
    float wx[PME_ORDER], wy[PME_ORDER], wz[PME_ORDER], dx[PME_ORDER], dy[PME_ORDER], dz[PME_ORDER];
    bspline5(frac[0], wx, dx);
    bspline5(frac[1], wy, dy);
    bspline5(frac[2], wz, dz);
    const float* grid = d.grid_r + (size_t)r * d.gsize;
    float fx = 0.f, fy = 0.f, fz = 0.f;
#pragma unroll
    for (int i = 0; i < PME_ORDER; ++i) {
        int gx = base[0] + i; gx -= gx >= d.gx ? d.gx : 0;
#pragma unroll
        for (int j = 0; j < PME_ORDER; ++j) {
            int gy = base[1] + j; gy -= gy >= d.gy ? d.gy : 0;
            const float* row = grid + ((size_t)gx * d.gy + gy) * d.gz;
            float s0 = 0.f, s1 = 0.f;
#pragma unroll
            for (int k = 0; k < PME_ORDER; ++k) {
                int gz = base[2] + k; gz -= gz >= d.gz ? d.gz : 0;
                const float v = row[gz];
                s0 += v * wz[k];
                s1 += v * dz[k];
            }
            fx += dx[i] * wy[j] * s0;
            fy += wx[i] * dy[j] * s0;
            fz += wx[i] * wy[j] * s1;
        }
    }
    // d.grid_r now holds the (unnormalised) inverse transform of G*S: potential phi = that value
    const float q = p.w;
    long long* fenv = d.f_env + (size_t)r * 3 * d.N;
    fx_addf(&fenv[a], -q * fx * d.gx * d.boxf[3], (float)FORCE_SCALE);
    fx_addf(&fenv[d.N + a], -q * fy * d.gy * d.boxf[4], (float)FORCE_SCALE);
    fx_addf(&fenv[2 * d.N + a], -q * fz * d.gz * d.boxf[5], (float)FORCE_SCALE);
}

// Latency-oriented gather for contexts with one or two walkers: five lanes per atom, one stencil x-plane each (25 grid
// loads per lane instead of 125), combined with shuffles.  Six atoms per warp (lanes 30, 31 idle).
__global__ void __launch_bounds__(128) k_pme_gather5(Dev d, int skip_frozen) {
    const int r = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int slot = lane / PME_ORDER, i = lane - slot * PME_ORDER;       // atom slot 0..5 (6 = idle), x-plane 0..4
    const int a = warp * 6 + slot;
    if (blockIdx.x == 0 && threadIdx.x == 0 && d.grid_frozen) d.frozen_grid_state[r] = 1;      // (see k_pme_gather)
    const bool active = slot < 6 && a < d.N && !(skip_frozen && d.mass[min(a, d.N - 1)] == 0.0);
    float fx = 0.f, fy = 0.f, fz = 0.f, q = 0.f;
    if (active) {
        const float4 p = d.posq[(size_t)r * d.N + a];
        q = p.w;
        if (q != 0.f) {
            int base[3];
            float frac[3];
            pme_atom_setup(d, p, base, frac);
            float wx[PME_ORDER], wy[PME_ORDER], wz[PME_ORDER], dx[PME_ORDER], dy[PME_ORDER], dz[PME_ORDER];
            bspline5(frac[0], wx, dx);
            bspline5(frac[1], wy, dy);
            bspline5(frac[2], wz, dz);
            float wxi = 0.f, dxi = 0.f;
#pragma unroll
            for (int k = 0; k < PME_ORDER; ++k) { wxi = (k == i) ? wx[k] : wxi; dxi = (k == i) ? dx[k] : dxi; }
            const float* grid = d.grid_r + (size_t)r * d.gsize;
            int gx = base[0] + i; gx -= gx >= d.gx ? d.gx : 0;
            float sx = 0.f, sy = 0.f, sz = 0.f;
#pragma unroll
            for (int j = 0; j < PME_ORDER; ++j) {
                int gy = base[1] + j; gy -= gy >= d.gy ? d.gy : 0;
                const float* row = grid + ((size_t)gx * d.gy + gy) * d.gz;
                float s0 = 0.f, s1 = 0.f;
#pragma unroll
                for (int k = 0; k < PME_ORDER; ++k) {
                    int gz = base[2] + k; gz -= gz >= d.gz ? d.gz : 0;
                    const float v = row[gz];
                    s0 += v * wz[k];
                    s1 += v * dz[k];
                }
                sx += wy[j] * s0;
                sy += dy[j] * s0;
                sz += wy[j] * s1;
            }
            fx = dxi * sx; fy = wxi * sy; fz = wxi * sz;
        }
    }
    // sum the five planes of each atom: lanes 5 slot + 1..4 into lane 5 slot (fixed order -> deterministic)
    float tx = fx, ty = fy, tz = fz;
#pragma unroll
    for (int k = 1; k < PME_ORDER; ++k) {
        const int src = min(lane + k, 31);
        const float ox = __shfl_sync(0xffffffffu, fx, src), oy = __shfl_sync(0xffffffffu, fy, src), oz = __shfl_sync(0xffffffffu, fz, src);
        tx += ox; ty += oy; tz += oz;
    }
    if (active && i == 0 && q != 0.f) {
        long long* fenv = d.f_env + (size_t)r * 3 * d.N;
        fx_addf(&fenv[a], -q * tx * d.gx * d.boxf[3], (float)FORCE_SCALE);
        fx_addf(&fenv[d.N + a], -q * ty * d.gy * d.boxf[4], (float)FORCE_SCALE);
        fx_addf(&fenv[2 * d.N + a], -q * tz * d.gz * d.boxf[5], (float)FORCE_SCALE);
    }
}
