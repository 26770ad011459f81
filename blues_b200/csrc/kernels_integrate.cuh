// Fused integrator (K8): one thread per constraint cluster runs a whole sequence of Langevin substeps
// (V / R / O with matrix-SHAKE + exact RATTLE), the H-step work bookkeeping (K9), plus small state kernels (K10/K11).
#pragma once
#include "engine.cuh"

// single-precision mirror of a position, wrapped into the primary cell (the neighbour search relies on it)
__device__ __forceinline__ float4 wrapped_mirror(const Dev& d, double x, double y, double z, float q) {
    if (d.periodic) {
        x -= d.boxd[0] * floor(x * d.boxd[3]);
        y -= d.boxd[1] * floor(y * d.boxd[4]);
        z -= d.boxd[2] * floor(z * d.boxd[5]);
        // a coordinate beyond ~1e15 box lengths (a walker that blew up; it is flagged like a NaN, see BLOWUP_LIMIT) no
        // longer wraps into the cell: park it at the origin so that every index derived from the mirror stays in range
        if (!(x >= 0.0 && x <= d.boxd[0])) x = 0.0;
        if (!(y >= 0.0 && y <= d.boxd[1])) y = 0.0;
        if (!(z >= 0.0 && z <= d.boxd[2])) z = 0.0;
    }
    return make_float4((float)x, (float)y, (float)z, q);
}

// A coordinate of this magnitude (nm) is a walker that blew up: OpenMM's "Particle coordinate is nan" follows within a
// step or two; here it raises the same per-walker flag at once (NaN compares false, so NaN is covered too).
#define BLOWUP_LIMIT 1.0e6

struct ClusterState {
    double x[MAX_CLUSTER_ATOMS][3];
    double v[MAX_CLUSTER_ATOMS][3];
    double im[MAX_CLUSTER_ATOMS];
};

// Solve the n x n system A y = b in place (Gaussian elimination with partial pivoting), n <= MAX_CLUSTER_CONS.
__device__ __forceinline__ void solve_small(double A[MAX_CLUSTER_CONS][MAX_CLUSTER_CONS], double* b, int n) {
    for (int c = 0; c < n; ++c) {
        int piv = c;
        double best = fabs(A[c][c]);
        for (int rr = c + 1; rr < n; ++rr)
            if (fabs(A[rr][c]) > best) { best = fabs(A[rr][c]); piv = rr; }
        if (piv != c) {
            for (int k = 0; k < n; ++k) { double t = A[c][k]; A[c][k] = A[piv][k]; A[piv][k] = t; }
            double t = b[c]; b[c] = b[piv]; b[piv] = t;
        }
        const double inv = 1.0 / A[c][c];
        for (int rr = c + 1; rr < n; ++rr) {
            const double f = A[rr][c] * inv;
            if (f != 0.0) {
                for (int k = c; k < n; ++k) A[rr][k] -= f * A[c][k];
                b[rr] -= f * b[c];
            }
        }
    }
    for (int c = n - 1; c >= 0; --c) {
        double s = b[c];
        for (int k = c + 1; k < n; ++k) s -= A[c][k] * b[k];
        b[c] = s / A[c][c];
    }
}

// coupling coefficient between constraints a and b of a cluster: how a unit multiplier on b moves the
// separation vector of a (through shared atoms and inverse masses)
__device__ __forceinline__ double coupling(const Cluster& c, const double* im, int a, int b) {
    const int ia = c.ca[a], ja = c.cb[a], ib = c.ca[b], jb = c.cb[b];
    return ((ia == ib) - (ia == jb)) * im[ia] - ((ja == ib) - (ja == jb)) * im[ja];
}

// RATTLE (exact, linear): remove velocity components along the constraints
__device__ __forceinline__ void constrain_velocities(const Cluster& c, ClusterState& s) {
    const int n = c.ncons;
    if (n == 0) return;
    double sv[MAX_CLUSTER_CONS][3];
    double A[MAX_CLUSTER_CONS][MAX_CLUSTER_CONS], rhs[MAX_CLUSTER_CONS];
    for (int a = 0; a < n; ++a) {
        const int i = c.ca[a], j = c.cb[a];
        double dvv = 0.0;
        for (int k = 0; k < 3; ++k) {
            sv[a][k] = s.x[i][k] - s.x[j][k];
            dvv += sv[a][k] * (s.v[i][k] - s.v[j][k]);
        }
        rhs[a] = -dvv;
    }
    for (int a = 0; a < n; ++a)
        for (int b = 0; b < n; ++b)
            A[a][b] = coupling(c, s.im, a, b) * (sv[a][0] * sv[b][0] + sv[a][1] * sv[b][1] + sv[a][2] * sv[b][2]);
    solve_small(A, rhs, n);
    for (int a = 0; a < n; ++a) {
        const int i = c.ca[a], j = c.cb[a];
        for (int k = 0; k < 3; ++k) {
            const double cc = rhs[a] * sv[a][k];
            s.v[i][k] += cc * s.im[i];
            s.v[j][k] -= cc * s.im[j];
        }
    }
}

// matrix SHAKE: move x along the reference directions (xref) until every |x_i - x_j|^2 = d^2
__device__ __forceinline__ void constrain_positions(const Cluster& c, ClusterState& s,
                                                    const double xref[MAX_CLUSTER_ATOMS][3], double tol) {
    const int n = c.ncons;
    if (n == 0) return;
    double rr[MAX_CLUSTER_CONS][3];
    for (int a = 0; a < n; ++a)
        for (int k = 0; k < 3; ++k) rr[a][k] = xref[c.ca[a]][k] - xref[c.cb[a]][k];
    for (int it = 0; it < 30; ++it) {
        double sv[MAX_CLUSTER_CONS][3], diff[MAX_CLUSTER_CONS];
        double worst = 0.0;
        for (int a = 0; a < n; ++a) {
            const int i = c.ca[a], j = c.cb[a];
            double s2 = 0.0;
            for (int k = 0; k < 3; ++k) { sv[a][k] = s.x[i][k] - s.x[j][k]; s2 += sv[a][k] * sv[a][k]; }
            diff[a] = c.d2[a] - s2;
            worst = fmax(worst, fabs(diff[a]) / c.d2[a]);
        }
        if (worst < tol) break;
        double A[MAX_CLUSTER_CONS][MAX_CLUSTER_CONS];
        for (int a = 0; a < n; ++a)
            for (int b = 0; b < n; ++b)
                A[a][b] = 2.0 * coupling(c, s.im, a, b) * (sv[a][0] * rr[b][0] + sv[a][1] * rr[b][1] + sv[a][2] * rr[b][2]);
        solve_small(A, diff, n);
        for (int a = 0; a < n; ++a) {
            const int i = c.ca[a], j = c.cb[a];
            for (int k = 0; k < 3; ++k) {
                const double cc = diff[a] * rr[a][k];
                s.x[i][k] += cc * s.im[i];
                s.x[j][k] -= cc * s.im[j];
            }
        }
    }
}

__device__ __forceinline__ double alch_energy(const Dev& d, int r, int slot) {
    const long long* a = d.alch_acc + (r * ALCH_SLOTS + slot) * 3;
    return (double)(a[0] + a[1] + a[2]) * (1.0 / ENERGY_SCALE);
}
__device__ __forceinline__ double env_energy(const Dev& d, int r) {
    long long s = 0;
    for (int k = 0; k <= E_PME; ++k) s += d.eacc[r * N_ETERMS + k];
    const double V = d.periodic ? d.boxd[0] * d.boxd[1] * d.boxd[2] : 1.0;
    double e = (double)s * (1.0 / ENERGY_SCALE);
    if (d.pme) e += d.self_energy_coeff - ONE_4PI_EPS0 * 3.14159265358979323846 * d.sumq * d.sumq / (2.0 * d.alphad * d.alphad * V);
    if (d.periodic) e += d.dispersion_coeff / V;
    return e;
}

struct IntegrateArgs {
    int nops;
    Op ops[MAX_OPS];
    int accum_cm;       // 0 none, 1 into cm_acc[parity], 2 into cm_acc[1-parity]
    int energy_valid;   // the preceding force evaluation produced energies (for OP_STEP_END bookkeeping)
    int noise_offset;   // O / MD ops executed by INTEGRATE launches since the last k_begin_eval
    int md_offset;
    // the launch is followed by a force evaluation (step programs only): every thread clears the force accumulators of its
    // own atoms once it has used them, and the last CTA of a walker to finish does what k_sort_atoms' latch and
    // k_begin_eval's first CTA otherwise do (rebuild latch, energy accumulators, noise counters, momentum parity) — one
    // kernel less on the critical path and a latch-free early exit for the sort kernel
    int pre_eval, pre_cm_mode, pre_adv_noise, pre_adv_md;
};

// ---------------------------------------------------------------------------------------------------------
// Register-resident cluster integrator.  SHAPE_STAR: constraints (0,1)..(0,NC) around atom 0 (X-H groups, free
// atoms with NC = 0); SHAPE_TRI: the rigid-water triangle (0,1),(0,2),(1,2).  All loops have compile-time bounds
// so x/v/… live in registers (no local-memory traffic), unlike the generic fallback further down.
// ---------------------------------------------------------------------------------------------------------
#define SHAPE_STAR 0
#define SHAPE_TRI 1
#define SHAPE_GENERIC 2

template <int SHAPE> __device__ __forceinline__ constexpr int con_a(int a) { return SHAPE == SHAPE_TRI ? (a == 2 ? 1 : 0) : 0; }
template <int SHAPE> __device__ __forceinline__ constexpr int con_b(int a) { return SHAPE == SHAPE_TRI ? (a == 0 ? 1 : 2) : a + 1; }

template <int NC>
__device__ __forceinline__ void solve_fixed(double (&A)[NC > 0 ? NC : 1][NC > 0 ? NC : 1], double (&b)[NC > 0 ? NC : 1]) {
    // closed-form solution (adjugate / determinant) of the 1x1, 2x2 and 3x3 constraint systems: ONE division and a
    // shallow dependency chain.  The integrator runs one cluster per thread with few warps per SM, so its run time is
    // the latency of this chain; Gaussian elimination (six dependent double divisions) was most of it.
    if (NC == 1) {
        b[0] = b[0] / A[0][0];
    } else if (NC == 2) {
        const double inv = 1.0 / (A[0][0] * A[1][1] - A[0][1] * A[1][0]);
        const double x0 = (b[0] * A[1][1] - A[0][1] * b[1]) * inv;
        const double x1 = (A[0][0] * b[1] - A[1][0] * b[0]) * inv;
        b[0] = x0; b[1] = x1;
    } else if (NC == 3) {
        const double c00 = A[1][1] * A[2][2] - A[1][2] * A[2][1];
        const double c01 = A[1][2] * A[2][0] - A[1][0] * A[2][2];
        const double c02 = A[1][0] * A[2][1] - A[1][1] * A[2][0];
        const double inv = 1.0 / (A[0][0] * c00 + A[0][1] * c01 + A[0][2] * c02);
        const double x0 = b[0] * c00 + b[1] * (A[0][2] * A[2][1] - A[0][1] * A[2][2]) + b[2] * (A[0][1] * A[1][2] - A[0][2] * A[1][1]);
        const double x1 = b[0] * c01 + b[1] * (A[0][0] * A[2][2] - A[0][2] * A[2][0]) + b[2] * (A[0][2] * A[1][0] - A[0][0] * A[1][2]);
        const double x2 = b[0] * c02 + b[1] * (A[0][1] * A[2][0] - A[0][0] * A[2][1]) + b[2] * (A[0][0] * A[1][1] - A[0][1] * A[1][0]);
        b[0] = x0 * inv; b[1] = x1 * inv; b[2] = x2 * inv;
    }
}

__device__ __forceinline__ void prefetch_l1(const void* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

template <int NA, int NC, int SHAPE>
struct FixedCluster {
    static constexpr int NCC = NC > 0 ? NC : 1;
    double x[NA][3], v[NA][3], im[NA], mass[NA];
    double d2[NCC];

    __device__ __forceinline__ double coup(int a, int b) const {
        const int ia = con_a<SHAPE>(a), ja = con_b<SHAPE>(a), ib = con_a<SHAPE>(b), jb = con_b<SHAPE>(b);
        return ((ia == ib) - (ia == jb)) * im[ia] - ((ja == ib) - (ja == jb)) * im[ja];
    }

    __device__ __forceinline__ void rattle() {
        if constexpr (NC > 0) {
        double sv[NCC][3], A[NCC][NCC], rhs[NCC];
#pragma unroll
        for (int a = 0; a < NC; ++a) {
            const int i = con_a<SHAPE>(a), j = con_b<SHAPE>(a);
            double dvv = 0.0;
#pragma unroll
            for (int k = 0; k < 3; ++k) { sv[a][k] = x[i][k] - x[j][k]; dvv += sv[a][k] * (v[i][k] - v[j][k]); }
            rhs[a] = -dvv;
        }
#pragma unroll
        for (int a = 0; a < NC; ++a)
#pragma unroll
            for (int b = 0; b < NC; ++b)
                A[a][b] = coup(a, b) * (sv[a][0] * sv[b][0] + sv[a][1] * sv[b][1] + sv[a][2] * sv[b][2]);
        solve_fixed<NC>(A, rhs);
#pragma unroll
        for (int a = 0; a < NC; ++a) {
            const int i = con_a<SHAPE>(a), j = con_b<SHAPE>(a);
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const double cc = rhs[a] * sv[a][k];
                v[i][k] += cc * im[i];
                v[j][k] -= cc * im[j];
            }
        }
        }
    }

    __device__ __forceinline__ void shake(const double (&xref)[NA][3], double tol) {
        if constexpr (NC > 0) {
        double rr[NCC][3];
#pragma unroll
        for (int a = 0; a < NC; ++a)
#pragma unroll
            for (int k = 0; k < 3; ++k) rr[a][k] = xref[con_a<SHAPE>(a)][k] - xref[con_b<SHAPE>(a)][k];
        // Newton's method converges quadratically: once every relative residual is below 0.1 sqrt(tol) the next update
        // lands far inside the tolerance, so the final residual evaluation (a third of a typical solve) is skipped.
        // The number of updates, hence the result, is the same as with the check.
        const double quad = 0.1 * sqrt(tol);
        for (int it = 0; it < 30; ++it) {
            double sv[NCC][3], diff[NCC], worst = -1.0e300, nearly = -1.0e300;
#pragma unroll
            for (int a = 0; a < NC; ++a) {
                const int i = con_a<SHAPE>(a), j = con_b<SHAPE>(a);
                double s2 = 0.0;
#pragma unroll
                for (int k = 0; k < 3; ++k) { sv[a][k] = x[i][k] - x[j][k]; s2 += sv[a][k] * sv[a][k]; }
                diff[a] = d2[a] - s2;
                worst = fmax(worst, fabs(diff[a]) - tol * d2[a]);        // |diff| / d2 < tol without the division
                nearly = fmax(nearly, fabs(diff[a]) - quad * d2[a]);
            }
            if (worst < 0.0) break;
            double A[NCC][NCC];
#pragma unroll
            for (int a = 0; a < NC; ++a)
#pragma unroll
                for (int b = 0; b < NC; ++b)
                    A[a][b] = 2.0 * coup(a, b) * (sv[a][0] * rr[b][0] + sv[a][1] * rr[b][1] + sv[a][2] * rr[b][2]);
            solve_fixed<NC>(A, diff);
#pragma unroll
            for (int a = 0; a < NC; ++a) {
                const int i = con_a<SHAPE>(a), j = con_b<SHAPE>(a);
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    const double cc = diff[a] * rr[a][k];
                    x[i][k] += cc * im[i];
                    x[j][k] -= cc * im[j];
                }
            }
            if (nearly < 0.0) break;
        }
        }
    }
};

// Runs the op list on one cluster; returns momentum / heat contributions and rebuild / NaN flags through refs.
template <int NA, int NC, int SHAPE>
__device__ __forceinline__ void run_cluster(const Dev& d, const IntegratorConsts& ic, const IntegrateArgs& args,
                                            const Cluster& c, int r, int parity, unsigned int noise0, unsigned int md0,
                                            double (&mom)[3], double& dheat, bool& moved, bool& bad) {
    const int N = d.N;
    double4* pos = d.pos + (size_t)r * N;
    double4* vel = d.vel + (size_t)r * N;
    const long long* fenv = d.f_env + (size_t)r * 3 * N;
    FixedCluster<NA, NC, SHAPE> s;
    int atom[NA];
#pragma unroll
    for (int k = 0; k < NA; ++k) {
        const int a = c.atom[k];
        atom[k] = a;
        const double4 p = pos[a], v = vel[a];
        s.x[k][0] = p.x; s.x[k][1] = p.y; s.x[k][2] = p.z;
        s.v[k][0] = v.x; s.v[k][1] = v.y; s.v[k][2] = v.z;
        s.im[k] = d.invmass[a];
        s.mass[k] = d.mass[a];
    }
    {
        // a cluster of frozen atoms (mass 0: freeze_radius / freeze_atoms) is never moved by any op: all that is left of
        // the launch for it is the clearing of its force accumulators before an evaluation
        bool any_mobile = false;
#pragma unroll
        for (int k = 0; k < NA; ++k) any_mobile = any_mobile || s.im[k] > 0.0;
        if (!any_mobile) {
            if (args.pre_eval) {
#pragma unroll
                for (int k = 0; k < NA; ++k)
#pragma unroll
                    for (int q = 0; q < 3; ++q) {
                        d.f_env[(size_t)r * 3 * N + q * N + atom[k]] = 0;
                        if (d.alch_on)
                            for (int sl = 0; sl < ALCH_SLOTS; ++sl) d.f_alch[((size_t)sl * d.R + r) * 3 * N + q * N + atom[k]] = 0;
                    }
            }
            return;
        }
    }
#pragma unroll
    for (int a = 0; a < NC; ++a) s.d2[a] = c.d2[a];
    // the forces of the first V step and the kicks of the first O step are needed a few hundred dependent instructions
    // from now: start pulling their lines into L1 (no registers held)
    for (int o = 0; o < args.nops; ++o) {
        const Op op = args.ops[o];
        if (op.kind == OP_V || op.kind == OP_MD) {
#pragma unroll
            for (int k = 0; k < NA; ++k)
#pragma unroll
                for (int q = 0; q < 3; ++q) {
                    prefetch_l1(&fenv[q * N + atom[k]]);
                    if (d.alch_on) prefetch_l1(&d.f_alch[((size_t)op.slot * d.R + r) * 3 * N + q * N + atom[k]]);
                }
            break;
        }
    }
    for (int o = 0; o < args.nops; ++o)
        if (args.ops[o].kind == OP_O || args.ops[o].kind == OP_MD) {
#pragma unroll
            for (int k = 0; k < NA; ++k) prefetch_l1(d.noise + ((size_t)r * MAX_NOISE_SETS * N + atom[k]) * 3);
            break;
        }
    int n_o = 0, n_md = 0;
    bool x_changed = false;
    double xref[NA][3], x1[NA][3];
    // every op = [update] -> optional SHAKE -> [velocity fix-up] -> optional RATTLE, so that the constraint solvers
    // are instantiated once per cluster shape (keeps the kernel small enough for the instruction cache)
    for (int o = 0; o < args.nops; ++o) {
        const Op op = args.ops[o];
        bool do_shake = false, do_rattle = false;
        int post = 0;
        double ke0 = 0.0;
        if (op.kind == OP_CM) {
            if (ic.remove_cm) {
                const long long* cm = d.cm_acc + ((size_t)parity * d.R + r) * 3;
                const double inv = 1.0 / (FORCE_SCALE * ic.total_mass);
                const double vx = (double)cm[0] * inv, vy = (double)cm[1] * inv, vz = (double)cm[2] * inv;
#pragma unroll
                for (int k = 0; k < NA; ++k)
                    if (s.im[k] > 0.0) { s.v[k][0] -= vx; s.v[k][1] -= vy; s.v[k][2] -= vz; }
            }
        } else if (op.kind == OP_V) {
            const long long* fa = d.alch_on ? d.f_alch + ((size_t)op.slot * d.R + r) * 3 * N : nullptr;
#pragma unroll
            for (int k = 0; k < NA; ++k) {
                const double sc = ic.hV * s.im[k] * (1.0 / FORCE_SCALE);
#pragma unroll
                for (int q = 0; q < 3; ++q) {
                    long long f = fenv[q * N + atom[k]];
                    if (fa) f += fa[q * N + atom[k]];
                    s.v[k][q] += sc * (double)f;
                }
            }
            do_rattle = true;
        } else if (op.kind == OP_R) {
#pragma unroll
            for (int k = 0; k < NA; ++k)
#pragma unroll
                for (int q = 0; q < 3; ++q) {
                    xref[k][q] = s.x[k][q];
                    if (s.im[k] > 0.0) s.x[k][q] += ic.hR * s.v[k][q];
                    x1[k][q] = s.x[k][q];
                }
            do_shake = do_rattle = true;
            post = 1;
            x_changed = true;
        } else if (op.kind == OP_O) {
#pragma unroll
            for (int k = 0; k < NA; ++k) {
                ke0 += 0.5 * s.mass[k] * (s.v[k][0] * s.v[k][0] + s.v[k][1] * s.v[k][1] + s.v[k][2] * s.v[k][2]);
                if (s.im[k] > 0.0) {
                    const double* nz = d.noise + (((size_t)r * MAX_NOISE_SETS + n_o) * N + atom[k]) * 3;
                    // k_noise stores the kicks already scaled by b sqrt(kT / m)
                    s.v[k][0] = ic.a * s.v[k][0] + nz[0];
                    s.v[k][1] = ic.a * s.v[k][1] + nz[1];
                    s.v[k][2] = ic.a * s.v[k][2] + nz[2];
                }
            }
            ++n_o;
            do_rattle = true;
            post = 3;
        } else if (op.kind == OP_MD) {
#pragma unroll
            for (int k = 0; k < NA; ++k) {
                double n[3] = {0.0, 0.0, 0.0};
                if (s.im[k] > 0.0) {
                    const double* nz = d.noise + (((size_t)r * MAX_NOISE_SETS + n_md) * N + atom[k]) * 3;
                    n[0] = nz[0]; n[1] = nz[1]; n[2] = nz[2];
                }
#pragma unroll
                for (int q = 0; q < 3; ++q) {
                    xref[k][q] = s.x[k][q];
                    if (s.im[k] > 0.0) {
                        long long fi = fenv[q * N + atom[k]];
                        if (d.alch_on) fi += d.f_alch[((size_t)op.slot * d.R + r) * 3 * N + q * N + atom[k]];
                        const double f = (double)fi * (1.0 / FORCE_SCALE);
                        s.v[k][q] = ic.md_vscale * s.v[k][q] + ic.md_fscale * s.im[k] * f + n[q];   // pre-scaled kick
                        s.x[k][q] += ic.dt * s.v[k][q];
                    }
                }
            }
            ++n_md;
            do_shake = true;
            post = 2;
            x_changed = true;
        } else if (op.kind == OP_CONSTRAIN) {
            x_changed = true;
#pragma unroll
            for (int k = 0; k < NA; ++k)
#pragma unroll
                for (int q = 0; q < 3; ++q) xref[k][q] = s.x[k][q];
            do_shake = do_rattle = true;
        }
        if (do_shake) s.shake(xref, ic.tol);
        if (post == 1) {
            const double ih = 1.0 / ic.hR;
#pragma unroll
            for (int k = 0; k < NA; ++k)
#pragma unroll
                for (int q = 0; q < 3; ++q) s.v[k][q] += (s.x[k][q] - x1[k][q]) * ih;
        } else if (post == 2) {
            const double idt = 1.0 / ic.dt;
#pragma unroll
            for (int k = 0; k < NA; ++k)
#pragma unroll
                for (int q = 0; q < 3; ++q)
                    if (s.im[k] > 0.0) s.v[k][q] = (s.x[k][q] - xref[k][q]) * idt;
        }
        if (do_rattle) s.rattle();
        if (post == 3) {
            double ke1 = 0.0;
#pragma unroll
            for (int k = 0; k < NA; ++k)
                ke1 += 0.5 * s.mass[k] * (s.v[k][0] * s.v[k][0] + s.v[k][1] * s.v[k][1] + s.v[k][2] * s.v[k][2]);
            dheat += ke1 - ke0;
        }
    }
    const float lim = d.skin_half2;
    if (args.pre_eval) {
#pragma unroll
        for (int k = 0; k < NA; ++k)
#pragma unroll
            for (int q = 0; q < 3; ++q) {
                d.f_env[(size_t)r * 3 * N + q * N + atom[k]] = 0;
                if (d.alch_on)
                    for (int sl = 0; sl < ALCH_SLOTS; ++sl) d.f_alch[((size_t)sl * d.R + r) * 3 * N + q * N + atom[k]] = 0;
            }
    }
    if (!x_changed) {
        // velocity-only launch (e.g. the trailing "V H" of a pass): positions, mirrors and the displacement test are
        // untouched
#pragma unroll
        for (int k = 0; k < NA; ++k) {
            vel[atom[k]] = make_double4(s.v[k][0], s.v[k][1], s.v[k][2], 0.0);
#pragma unroll
            for (int q = 0; q < 3; ++q) mom[q] += s.mass[k] * s.v[k][q];
        }
        return;
    }
#pragma unroll
    for (int k = 0; k < NA; ++k) {
        const int a = atom[k];
        pos[a] = make_double4(s.x[k][0], s.x[k][1], s.x[k][2], 0.0);
        vel[a] = make_double4(s.v[k][0], s.v[k][1], s.v[k][2], 0.0);
        const float4 pf = wrapped_mirror(d, s.x[k][0], s.x[k][1], s.x[k][2], d.charge[a]);
        d.posq[(size_t)r * N + a] = pf;
        { const size_t sl = (size_t)r * d.Npad + d.rank[(size_t)r * N + a]; d.posq_s[sl] = pf; }
        const float4 pr = d.pos_ref[(size_t)r * N + a];
        float ddx = pf.x - pr.x, ddy = pf.y - pr.y, ddz = pf.z - pr.z;
        if (d.periodic) {
            ddx -= d.boxf[0] * rintf(ddx * d.boxf[3]);
            ddy -= d.boxf[1] * rintf(ddy * d.boxf[4]);
            ddz -= d.boxf[2] * rintf(ddz * d.boxf[5]);
        }
        moved = moved || (ddx * ddx + ddy * ddy + ddz * ddz > lim);
        bad = bad || !(fabs(s.x[k][0]) < BLOWUP_LIMIT && fabs(s.x[k][1]) < BLOWUP_LIMIT && fabs(s.x[k][2]) < BLOWUP_LIMIT);
#pragma unroll
        for (int q = 0; q < 3; ++q) mom[q] += s.mass[k] * s.v[k][q];
    }
}

// generic fallback (dynamic indexing, local memory): clusters that are neither stars nor water triangles
__device__ __forceinline__ void run_cluster_generic(const Dev& d, const IntegratorConsts& ic, const IntegrateArgs& args,
                                                 const Cluster& c, int r, int parity, unsigned int noise0,
                                                 unsigned int md0, double (&mom)[3], double& dheat, bool& moved, bool& bad) {
    const int N = d.N;
    double4* pos = d.pos + (size_t)r * N;
    double4* vel = d.vel + (size_t)r * N;
    const long long* fenv = d.f_env + (size_t)r * 3 * N;
    ClusterState s;
    double mass[MAX_CLUSTER_ATOMS];
    for (int k = 0; k < c.natoms; ++k) {
        const int a = c.atom[k];
        const double4 p = pos[a], v = vel[a];
        s.x[k][0] = p.x; s.x[k][1] = p.y; s.x[k][2] = p.z;
        s.v[k][0] = v.x; s.v[k][1] = v.y; s.v[k][2] = v.z;
        s.im[k] = d.invmass[a];
        mass[k] = d.mass[a];
    }
    int n_o = 0, n_md = 0;
    for (int o = 0; o < args.nops; ++o) {
        const Op op = args.ops[o];
        switch (op.kind) {
        case OP_CM: {
            if (ic.remove_cm) {
                const long long* cm = d.cm_acc + ((size_t)parity * d.R + r) * 3;
                const double inv = 1.0 / (FORCE_SCALE * ic.total_mass);
                const double vx = (double)cm[0] * inv, vy = (double)cm[1] * inv, vz = (double)cm[2] * inv;
                for (int k = 0; k < c.natoms; ++k)
                    if (s.im[k] > 0.0) { s.v[k][0] -= vx; s.v[k][1] -= vy; s.v[k][2] -= vz; }
            }
        } break;
        case OP_V: {
            const long long* fa = d.alch_on ? d.f_alch + ((size_t)op.slot * d.R + r) * 3 * N : nullptr;
            for (int k = 0; k < c.natoms; ++k) {
                const int a = c.atom[k];
                const double sc = ic.hV * s.im[k] * (1.0 / FORCE_SCALE);
                for (int q = 0; q < 3; ++q) {
                    long long f = fenv[q * N + a];
                    if (fa) f += fa[q * N + a];
                    s.v[k][q] += sc * (double)f;
                }
            }
            constrain_velocities(c, s);
        } break;
        case OP_R: {
            double xref[MAX_CLUSTER_ATOMS][3], x1[MAX_CLUSTER_ATOMS][3];
            for (int k = 0; k < c.natoms; ++k)
                for (int q = 0; q < 3; ++q) {
                    xref[k][q] = s.x[k][q];
                    if (s.im[k] > 0.0) s.x[k][q] += ic.hR * s.v[k][q];
                    x1[k][q] = s.x[k][q];
                }
            constrain_positions(c, s, xref, ic.tol);
            const double ih = 1.0 / ic.hR;
            for (int k = 0; k < c.natoms; ++k)
                for (int q = 0; q < 3; ++q) s.v[k][q] += (s.x[k][q] - x1[k][q]) * ih;
            constrain_velocities(c, s);
        } break;
        case OP_O: {
            double ke0 = 0.0, ke1 = 0.0;
            for (int k = 0; k < c.natoms; ++k) {
                ke0 += 0.5 * mass[k] * (s.v[k][0] * s.v[k][0] + s.v[k][1] * s.v[k][1] + s.v[k][2] * s.v[k][2]);
                if (s.im[k] > 0.0) {
                    double n0, n1, n2;
                    philox_normal3(ic.seed, STREAM_LANGEVIN, (uint32_t)r, noise0 + n_o, (uint32_t)c.atom[k], n0, n1, n2);
                    const double sg = ic.b * sqrt(ic.kT * s.im[k]);
                    s.v[k][0] = ic.a * s.v[k][0] + sg * n0;
                    s.v[k][1] = ic.a * s.v[k][1] + sg * n1;
                    s.v[k][2] = ic.a * s.v[k][2] + sg * n2;
                }
            }
            ++n_o;
            constrain_velocities(c, s);
            for (int k = 0; k < c.natoms; ++k)
                ke1 += 0.5 * mass[k] * (s.v[k][0] * s.v[k][0] + s.v[k][1] * s.v[k][1] + s.v[k][2] * s.v[k][2]);
            dheat += ke1 - ke0;
        } break;
        case OP_MD: {
            double xref[MAX_CLUSTER_ATOMS][3];
            for (int k = 0; k < c.natoms; ++k) {
                const int a = c.atom[k];
                double n[3] = {0.0, 0.0, 0.0};
                if (s.im[k] > 0.0)
                    philox_normal3(ic.seed, STREAM_MD, (uint32_t)r, md0 + n_md, (uint32_t)a, n[0], n[1], n[2]);
                const double sq = ic.md_nscale * sqrt(s.im[k]);
                for (int q = 0; q < 3; ++q) {
                    xref[k][q] = s.x[k][q];
                    if (s.im[k] > 0.0) {
                        long long fi = fenv[q * N + a];
                        if (d.alch_on) fi += d.f_alch[((size_t)op.slot * d.R + r) * 3 * N + q * N + a];
                        const double f = (double)fi * (1.0 / FORCE_SCALE);
                        s.v[k][q] = ic.md_vscale * s.v[k][q] + ic.md_fscale * s.im[k] * f + sq * n[q];
                        s.x[k][q] += ic.dt * s.v[k][q];
                    }
                }
            }
            ++n_md;
            constrain_positions(c, s, xref, ic.tol);
            const double idt = 1.0 / ic.dt;
            for (int k = 0; k < c.natoms; ++k)
                for (int q = 0; q < 3; ++q)
                    if (s.im[k] > 0.0) s.v[k][q] = (s.x[k][q] - xref[k][q]) * idt;
        } break;
        case OP_CONSTRAIN: {
            double xref[MAX_CLUSTER_ATOMS][3];
            for (int k = 0; k < c.natoms; ++k)
                for (int q = 0; q < 3; ++q) xref[k][q] = s.x[k][q];
            constrain_positions(c, s, xref, ic.tol);
            constrain_velocities(c, s);
        } break;
        default: break;
        }
    }
    const float lim = d.skin_half2;
    if (args.pre_eval)
        for (int k = 0; k < c.natoms; ++k)
            for (int q = 0; q < 3; ++q) {
                d.f_env[(size_t)r * 3 * N + q * N + c.atom[k]] = 0;
                if (d.alch_on)
                    for (int sl = 0; sl < ALCH_SLOTS; ++sl) d.f_alch[((size_t)sl * d.R + r) * 3 * N + q * N + c.atom[k]] = 0;
            }
    for (int k = 0; k < c.natoms; ++k) {
        const int a = c.atom[k];
        pos[a] = make_double4(s.x[k][0], s.x[k][1], s.x[k][2], 0.0);
        vel[a] = make_double4(s.v[k][0], s.v[k][1], s.v[k][2], 0.0);
        const float4 pf = wrapped_mirror(d, s.x[k][0], s.x[k][1], s.x[k][2], d.charge[a]);
        d.posq[(size_t)r * N + a] = pf;
        { const size_t sl = (size_t)r * d.Npad + d.rank[(size_t)r * N + a]; d.posq_s[sl] = pf; }
        const float4 pr = d.pos_ref[(size_t)r * N + a];
        float ddx = pf.x - pr.x, ddy = pf.y - pr.y, ddz = pf.z - pr.z;
        if (d.periodic) {
            ddx -= d.boxf[0] * rintf(ddx * d.boxf[3]);
            ddy -= d.boxf[1] * rintf(ddy * d.boxf[4]);
            ddz -= d.boxf[2] * rintf(ddz * d.boxf[5]);
        }
        moved = moved || (ddx * ddx + ddy * ddy + ddz * ddz > lim);
        bad = bad || !(fabs(s.x[k][0]) < BLOWUP_LIMIT && fabs(s.x[k][1]) < BLOWUP_LIMIT && fabs(s.x[k][2]) < BLOWUP_LIMIT);
        for (int q = 0; q < 3; ++q) mom[q] += mass[k] * s.v[k][q];
    }
}

// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_integrate(Dev d, IntegratorConsts ic, IntegrateArgs args, const int* cm_parity) {
    cudaGridDependencySynchronize();       // (see k_cm_flip)
    const int r = blockIdx.y;
    const int cid = blockIdx.x * blockDim.x + threadIdx.x;
    Globals& g = d.g[r];
    const int parity = *cm_parity;
    double mom[3] = {0.0, 0.0, 0.0};
    double dheat = 0.0;
    bool moved = false, bad = false;
    if (cid < d.n_clusters) {
        const Cluster c = d.clusters[cid];
        const unsigned int noise0 = g.noise_counter + args.noise_offset, md0 = g.md_counter + args.md_offset;
        const int key = c.shape * 16 + c.ncons;
        switch (key) {
        case SHAPE_STAR * 16 + 0: run_cluster<1, 0, SHAPE_STAR>(d, ic, args, c, r, parity, noise0, md0, mom, dheat, moved, bad); break;
        case SHAPE_STAR * 16 + 1: run_cluster<2, 1, SHAPE_STAR>(d, ic, args, c, r, parity, noise0, md0, mom, dheat, moved, bad); break;
        case SHAPE_STAR * 16 + 2: run_cluster<3, 2, SHAPE_STAR>(d, ic, args, c, r, parity, noise0, md0, mom, dheat, moved, bad); break;
        case SHAPE_STAR * 16 + 3: run_cluster<4, 3, SHAPE_STAR>(d, ic, args, c, r, parity, noise0, md0, mom, dheat, moved, bad); break;
        case SHAPE_TRI * 16 + 3: run_cluster<3, 3, SHAPE_TRI>(d, ic, args, c, r, parity, noise0, md0, mom, dheat, moved, bad); break;
        default: break;      // generic clusters are integrated by k_integrate_generic
        }
        if (moved) g.prune_request = 1;
        if (bad) g.nan_flag = 1;
    }
    if (args.accum_cm && ic.remove_cm) {
        const int target = args.accum_cm == 1 ? parity : 1 - parity;
        for (int q = 0; q < 3; ++q) {
            const double v = warp_sum(mom[q]);
            if ((threadIdx.x & 31) == 0) fx_add(&d.cm_acc[((size_t)target * d.R + r) * 3 + q], v, FORCE_SCALE);
        }
    }
    {
        const double v = warp_sum(dheat);
        if ((threadIdx.x & 31) == 0 && v != 0.0) fx_add(&d.heat_acc[r], v, ENERGY_SCALE);
    }
    // scalar bookkeeping of the step program by one thread per walker (K9): H updates and step end.
    // (an extra CTA with no clusters: the dependent loads of the energy accumulators then overlap the constraint work
    // instead of following it in thread 0 of CTA 0)
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) {
        for (int o = 0; o < args.nops; ++o) {
            const Op op = args.ops[o];
            if (op.kind == OP_H) {
                // blues/integrators.py:217-231
                g.debug += 1;
                const double e_old = alch_energy(d, r, op.slot), e_new = alch_energy(d, r, op.slot + 1);
                g.Eold = g.e_env + e_old;
                g.lambda_step += 1;
                g.lambda = (double)g.lambda_step / (double)ic.n_lambda_steps;
                g.Enew = g.e_env + e_new;
                g.protocol_work += e_new - e_old;
            } else if (op.kind == OP_STEP_END) {
                // blues/integrators.py:205-207: unperturbed_pe = energy; step += 1; prop = 1
                if (args.energy_valid) {
                    g.e_env = env_energy(d, r);
                    g.e_total_prev = g.e_env + alch_energy(d, r, op.slot);
                    g.unperturbed_pe = g.e_total_prev;
                    g.e_valid = 1;
                } else {
                    g.e_valid = 0;
                }
                g.step += 1;
                g.prop = 1;
                if (g.nan_flag) g.protocol_work = __longlong_as_double(0x7ff8000000000000LL);   // rejected by the Metropolis test
            }
        }
    }
    if (args.pre_eval) {
        // last CTA of this walker to get here: every flag, momentum sum and energy read of the launch is complete
        __shared__ int s_last;
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            s_last = atomicAdd(&d.cta_done[r], 1) == (int)gridDim.x - 1;
        }
        __syncthreads();
        if (s_last) {
            __threadfence();
            if (threadIdx.x == 0) {
                d.cta_done[r] = 0;
                g.do_rebuild = g.rebuild_request == 2 || g.prune_request;
                g.do_prune = g.do_rebuild;
                g.rebuild_request = 0;
                g.prune_request = 0;
                g.noise_counter += args.pre_adv_noise;
                g.md_counter += args.pre_adv_md;
            }
            for (int i = threadIdx.x; i < N_ETERMS; i += blockDim.x) d.eacc[r * N_ETERMS + i] = 0;
            for (int i = threadIdx.x; i < ALCH_SLOTS * 3; i += blockDim.x) d.alch_acc[r * ALCH_SLOTS * 3 + i] = 0;
        }
    }
}

// clusters that are neither stars (<= 3 constraints) nor water triangles: dynamic-index fallback, own kernel so that
// its stack frame and code do not burden the main integrator
__global__ void __launch_bounds__(64) k_integrate_generic(Dev d, IntegratorConsts ic, IntegrateArgs args, const int* cm_parity,
                                                         int n_generic) {
    const int r = blockIdx.y;
    const int cid = blockIdx.x * blockDim.x + threadIdx.x;
    Globals& g = d.g[r];
    const int parity = *cm_parity;
    double mom[3] = {0.0, 0.0, 0.0};
    double dheat = 0.0;
    bool moved = false, bad = false;
    if (cid < n_generic) {
        const Cluster c = d.clusters[cid];
        const unsigned int noise0 = g.noise_counter + args.noise_offset, md0 = g.md_counter + args.md_offset;
        run_cluster_generic(d, ic, args, c, r, parity, noise0, md0, mom, dheat, moved, bad);
        if (moved) g.prune_request = 1;
        if (bad) g.nan_flag = 1;
    }
    if (args.accum_cm && ic.remove_cm) {
        const int target = args.accum_cm == 1 ? parity : 1 - parity;
        for (int q = 0; q < 3; ++q) {
            const double v = warp_sum(mom[q]);
            if ((threadIdx.x & 31) == 0) fx_add(&d.cm_acc[((size_t)target * d.R + r) * 3 + q], v, FORCE_SCALE);
        }
    }
    const double v = warp_sum(dheat);
    if ((threadIdx.x & 31) == 0 && v != 0.0) fx_add(&d.heat_acc[r], v, ENERGY_SCALE);
}

// Thermostat noise for the next INTEGRATE launch: one thread per (atom, set).  Same Philox counters the fused
// integrator used to evaluate inline; hoisted out so that 1k-instruction Box-Muller chains run 22k-wide instead of
// serially inside each cluster thread.
__global__ void __launch_bounds__(128) k_noise(Dev d, IntegratorConsts ic, unsigned int stream_id, int n_sets, int offset) {
    const int r = blockIdx.y;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= d.N * n_sets) return;
    const int set = idx / d.N, a = idx - set * d.N;
    if (d.invmass[a] <= 0.0) return;
    const Globals& g = d.g[r];
    const unsigned int counter = (stream_id == STREAM_MD ? g.md_counter : g.noise_counter) + offset + set;
    const double3 v = philox_normal3v(ic.seed, stream_id, (uint32_t)r, counter, (uint32_t)a);
    // stored already scaled: b sqrt(kT / m) for the O step, md_nscale sqrt(1 / m) for the MD leg
    const double im = d.invmass[a];
    const double sc = stream_id == STREAM_MD ? ic.md_nscale * sqrt(im) : ic.b * sqrt(ic.kT * im);
    double* out = d.noise + (((size_t)r * MAX_NOISE_SETS + set) * d.N + a) * 3;
    out[0] = sc * v.x; out[1] = sc * v.y; out[2] = sc * v.z;
}

// ---------------------------------------------------------------------------------------------------------
// small state kernels
// ---------------------------------------------------------------------------------------------------------
// refresh the float mirrors from the double positions (after host writes / moves); request a rebuild
// clear_replica: walker whose NaN / list-overflow latches are cleared (-1 all, -2 none)
__global__ void k_refresh_mirrors(Dev d, int request_rebuild, int clear_replica) {
    const int r = blockIdx.y;
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a == 0 && (clear_replica == -1 || clear_replica == r)) { d.g[r].nan_flag = 0; d.g[r].item_overflow = 0; }
    if (a >= d.N) return;
    const double4 p = d.pos[(size_t)r * d.N + a];
    const float4 pf = wrapped_mirror(d, p.x, p.y, p.z, d.charge[a]);
    d.posq[(size_t)r * d.N + a] = pf;
    { const size_t sl = (size_t)r * d.Npad + d.rank[(size_t)r * d.N + a]; d.posq_s[sl] = pf; }
    if (a == 0 && request_rebuild) { d.g[r].rebuild_request = 2; d.g[r].prune_request = 1; }
}

__global__ void k_momentum(Dev d, const int* cm_parity) {
    const int r = blockIdx.y;
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    double m[3] = {0.0, 0.0, 0.0};
    if (a < d.N) {
        const double4 v = d.vel[(size_t)r * d.N + a];
        const double ms = d.mass[a];
        m[0] = ms * v.x; m[1] = ms * v.y; m[2] = ms * v.z;
    }
    const int p = *cm_parity;
    for (int q = 0; q < 3; ++q) {
        const double v = warp_sum(m[q]);
        if ((threadIdx.x & 31) == 0 && v != 0.0) fx_add(&d.cm_acc[((size_t)p * d.R + r) * 3 + q], v, FORCE_SCALE);
    }
}

// zero the consumed centre-of-mass accumulator and flip the parity (single-INTEGRATE passes)
__global__ void k_cm_flip(Dev d, int* cm_parity) {
    cudaGridDependencySynchronize();       // programmatic dependent launch: no-op when launched without the attribute
    const int p = *cm_parity;
    for (int i = threadIdx.x; i < d.R * 3; i += blockDim.x) d.cm_acc[(size_t)p * d.R * 3 + i] = 0;
    __syncthreads();
    if (threadIdx.x == 0) *cm_parity = p ^ 1;
}

// total force (environment + alchemical slot) as doubles, and potential energy per walker, for the host
__global__ void k_export_forces(Dev d, int r, int slot, double* out) {
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= d.N) return;
    for (int q = 0; q < 3; ++q) {
        long long f = d.f_env[(size_t)r * 3 * d.N + q * d.N + a];
        if (d.alch_on) f += d.f_alch[((size_t)slot * d.R + r) * 3 * d.N + q * d.N + a];
        out[a * 3 + q] = (double)f * (1.0 / FORCE_SCALE);
    }
}
__global__ void k_export_energy(Dev d, int slot, double* out) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= d.R) return;
    out[r] = env_energy(d, r) + (d.alch_on ? alch_energy(d, r, slot) : 0.0);
}

__global__ void k_zero_ll(long long* p, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = 0;
}

__global__ void k_kinetic_energy(Dev d, double* out) {
    const int r = blockIdx.y;
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    double ke = 0.0;
    if (a < d.N) {
        const double4 v = d.vel[(size_t)r * d.N + a];
        ke = 0.5 * d.mass[a] * (v.x * v.x + v.y * v.y + v.z * v.z);
    }
    ke = warp_sum(ke);
    if ((threadIdx.x & 31) == 0 && ke != 0.0) atomicAdd(&out[r], ke);
}

// Maxwell-Boltzmann draw per cluster followed by the velocity constraints (setVelocitiesToTemperature)
__global__ void __launch_bounds__(128) k_velocities_to_temperature(Dev d, double kT, uint64_t seed) {
    const int r = blockIdx.y;
    const int cid = blockIdx.x * blockDim.x + threadIdx.x;
    if (cid >= d.n_clusters) return;
    const Cluster c = d.clusters[cid];
    const unsigned int counter = d.g[r].vel_counter;
    ClusterState s;
    for (int k = 0; k < c.natoms; ++k) {
        const int a = c.atom[k];
        const double4 p = d.pos[(size_t)r * d.N + a];
        s.x[k][0] = p.x; s.x[k][1] = p.y; s.x[k][2] = p.z;
        s.im[k] = d.invmass[a];
        double n0, n1, n2;
        philox_normal3(seed, STREAM_VELOCITY, (uint32_t)r, counter, (uint32_t)a, n0, n1, n2);
        const double sg = sqrt(kT * s.im[k]);
        s.v[k][0] = sg * n0; s.v[k][1] = sg * n1; s.v[k][2] = sg * n2;
    }
    constrain_velocities(c, s);
    for (int k = 0; k < c.natoms; ++k)
        d.vel[(size_t)r * d.N + c.atom[k]] = make_double4(s.v[k][0], s.v[k][1], s.v[k][2], 0.0);
}

__global__ void k_bump_counter(Dev d, int which) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= d.R) return;
    if (which == 0) d.g[r].vel_counter += 1;
    else if (which == 1) d.g[r].move_counter += 1;
    else d.g[r].accept_counter += 1;
}

// RandomLigandRotationMove.move (blues/moves.py:278-310): one warp per walker.
// COM in float32 with the supplied masses, Shoemake quaternion from three Philox uniforms, x' = (x-c) R + c.
__global__ void k_move_rotate(Dev d, int n, const int* atoms, const float* masses, uint64_t seed) {
    const int r = blockIdx.x;
    const int lane = threadIdx.x;
    double4* pos = d.pos + (size_t)r * d.N;
    float cx = 0.f, cy = 0.f, cz = 0.f, mt = 0.f;
    // sequential float32 accumulation in atom order (numpy's float32 sum over a short axis is sequential)
    if (lane == 0) {
        for (int k = 0; k < n; ++k) {
            const double4 p = pos[atoms[k]];
            const float m = masses[k];
            cx += (float)p.x * m; cy += (float)p.y * m; cz += (float)p.z * m; mt += m;
        }
        cx /= mt; cy /= mt; cz /= mt;
    }
    cx = __shfl_sync(0xffffffffu, cx, 0);
    cy = __shfl_sync(0xffffffffu, cy, 0);
    cz = __shfl_sync(0xffffffffu, cz, 0);
    Philox4 u = philox4x32_10(0u, d.g[r].move_counter, (uint32_t)r, STREAM_MOVE, (uint32_t)seed, (uint32_t)(seed >> 32));
    const double u0 = u01(u.x), u1 = u01(u.y), u2 = u01(u.z);
    const double s1 = sqrt(1.0 - u0), s2 = sqrt(u0);
    double sa, ca, sb, cb;
    sincospi(2.0 * u1, &sa, &ca);
    sincospi(2.0 * u2, &sb, &cb);
    const double w = s1 * sa, x = s1 * ca, y = s2 * sb, z = s2 * cb;
    const double R[3][3] = {{1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)},
                            {2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)},
                            {2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)}};
    for (int k = lane; k < n; k += 32) {
        const int a = atoms[k];
        const double4 p = pos[a];
        const double px = p.x - (double)cx, py = p.y - (double)cy, pz = p.z - (double)cz;
        // row vector times R
        pos[a] = make_double4(px * R[0][0] + py * R[1][0] + pz * R[2][0] + (double)cx,
                              px * R[0][1] + py * R[1][1] + pz * R[2][1] + (double)cy,
                              px * R[0][2] + py * R[1][2] + pz * R[2][2] + (double)cz, 0.0);
    }
}

// ---- WaterTranslationMove on the device (blues/moves.py:846-1083): one CTA per walker --------------------------
struct WaterMove {
    int n_atoms;  const int* alch;          // atoms of the alchemical water, first = oxygen
    int n_waters; const int* waters;        // [n_waters][n_atoms]
    int n_center; const int* center; const float* cmass;
    double radius;
    double* state;                          // [R][4]: sphere centre of beforeMove (x, y, z), go flag
};
#define WATER_BLOCK 256

// centre of mass of the protein selection: float32 coordinates times float32 masses like the reference
// (blues/moves.py:921-949), summed in double by the CTA, returned as float32
__device__ float3 water_center(const Dev& d, const WaterMove& w, int r, double* red /* shared [3*WATER_BLOCK] */) {
    const double4* pos = d.pos + (size_t)r * d.N;
    double sx = 0.0, sy = 0.0, sz = 0.0, sm = 0.0;
    for (int k = threadIdx.x; k < w.n_center; k += WATER_BLOCK) {
        const double4 p = pos[w.center[k]];
        const float m = w.cmass[k];
        sx += (double)((float)p.x * m); sy += (double)((float)p.y * m); sz += (double)((float)p.z * m); sm += (double)m;
    }
    __shared__ double tot[4];
    sx = warp_sum(sx); sy = warp_sum(sy); sz = warp_sum(sz); sm = warp_sum(sm);
    const int wid = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { red[wid * 4] = sx; red[wid * 4 + 1] = sy; red[wid * 4 + 2] = sz; red[wid * 4 + 3] = sm; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0, c = 0.0, m = 0.0;
        for (int k = 0; k < WATER_BLOCK / 32; ++k) { a += red[k * 4]; b += red[k * 4 + 1]; c += red[k * 4 + 2]; m += red[k * 4 + 3]; }
        tot[0] = a / m; tot[1] = b / m; tot[2] = c / m;
    }
    __syncthreads();
    return make_float3((float)tot[0], (float)tot[1], (float)tot[2]);
}

// periodic distance between an atom and a point in float32, as mdtraj.compute_distances(periodic=True) does
__device__ __forceinline__ float water_distance(const Dev& d, const double4 p, const float3 c) {
    float dx = (float)p.x - c.x, dy = (float)p.y - c.y, dz = (float)p.z - c.z;
    if (d.periodic) {
        const float bx = (float)d.boxd[0], by = (float)d.boxd[1], bz = (float)d.boxd[2];
        dx -= bx * rintf(dx / bx); dy -= by * rintf(dy / by); dz -= bz * rintf(dz / bz);
    }
    return sqrtf(dx * dx + dy * dy + dz * dz);
}

// beforeMove: uniform choice (Philox) among the waters inside the sphere, then swap with the alchemical water
__global__ void __launch_bounds__(WATER_BLOCK) k_water_swap(Dev d, WaterMove w, uint64_t seed) {
    __shared__ double red[4 * WATER_BLOCK / 32];
    __shared__ int cnt[WATER_BLOCK];
    __shared__ int chosen;
    const int r = blockIdx.x, t = threadIdx.x;
    double4* pos = d.pos + (size_t)r * d.N;
    double4* vel = d.vel + (size_t)r * d.N;
    const float3 c = water_center(d, w, r, red);
    // contiguous chunk of waters per thread keeps the candidates in residue order
    const int chunk = (w.n_waters + WATER_BLOCK - 1) / WATER_BLOCK;
    const int k0 = min(t * chunk, w.n_waters), k1 = min(k0 + chunk, w.n_waters);
    int mine = 0;
    for (int k = k0; k < k1; ++k)
        mine += ((double)water_distance(d, pos[w.waters[(size_t)k * w.n_atoms]], c) <= w.radius) ? 1 : 0;
    cnt[t] = mine;
    if (t == 0) chosen = -1;
    __syncthreads();
    int before = 0, total = 0;
    for (int k = 0; k < WATER_BLOCK; ++k) { if (k < t) before += cnt[k]; total += cnt[k]; }
    if (total > 0) {
        const Philox4 u = philox4x32_10(1u, d.g[r].move_counter, (uint32_t)r, STREAM_MOVE, (uint32_t)seed, (uint32_t)(seed >> 32));
        const int pick = min((int)(u01(u.x) * (double)total), total - 1);
        if (pick >= before && pick < before + mine) {
            int seen = before;
            for (int k = k0; k < k1; ++k)
                if ((double)water_distance(d, pos[w.waters[(size_t)k * w.n_atoms]], c) <= w.radius) {
                    if (seen == pick) { chosen = k; break; }
                    ++seen;
                }
        }
    }
    __syncthreads();
    const int ch = chosen;
    if (ch >= 0 && t < w.n_atoms) {
        const int a = w.alch[t], b = w.waters[(size_t)ch * w.n_atoms + t];
        if (a != b) {
            const double4 pa = pos[a], pb = pos[b], va = vel[a], vb = vel[b];
            pos[a] = pb; pos[b] = pa; vel[a] = vb; vel[b] = va;
        }
    }
    if (t == 0) {
        double* st = w.state + (size_t)r * 4;
        st[0] = (double)c.x; st[1] = (double)c.y; st[2] = (double)c.z; st[3] = ch >= 0 ? 1.0 : 0.0;
    }
}

// move: the sphere centre is the one beforeMove cached (the reference reuses that frame, blues/moves.py:1021);
// r = R u^(1/3), phi = 2 pi u, cos(theta) = 2u - 1 (blues/moves.py:899-919)
__global__ void k_water_translate(Dev d, WaterMove w, uint64_t seed) {
    const int r = blockIdx.x, t = threadIdx.x;
    const double* st = w.state + (size_t)r * 4;
    if (st[3] == 0.0) return;
    double4* pos = d.pos + (size_t)r * d.N;
    const double4 po = pos[w.alch[0]];
    const float3 c = make_float3((float)st[0], (float)st[1], (float)st[2]);
    if ((double)water_distance(d, po, c) >= w.radius) return;
    const Philox4 u = philox4x32_10(2u, d.g[r].move_counter, (uint32_t)r, STREAM_MOVE, (uint32_t)seed, (uint32_t)(seed >> 32));
    const double rr = w.radius * cbrt(u01(u.x));
    double sp, cp;
    sincospi(2.0 * u01(u.y), &sp, &cp);
    const double ct = 2.0 * u01(u.z) - 1.0, sn = sqrt(fmax(0.0, 1.0 - ct * ct));
    const double tx = st[0] + rr * sn * cp, ty = st[1] + rr * sn * sp, tz = st[2] + rr * ct;
    const double sx = po.x - tx, sy = po.y - ty, sz = po.z - tz;
    __syncwarp();                                                      // every lane has read the oxygen
    if (t < w.n_atoms) {
        const int a = w.alch[t];
        const double4 p = pos[a];
        pos[a] = make_double4(p.x - sx, p.y - sy, p.z - sz, 0.0);
    }
}

// afterMove: fresh centre of mass; outside the sphere and the move was on -> protocol_work = 999999
__global__ void __launch_bounds__(WATER_BLOCK) k_water_check(Dev d, WaterMove w) {
    __shared__ double red[4 * WATER_BLOCK / 32];
    const int r = blockIdx.x;
    const float3 c = water_center(d, w, r, red);
    if (threadIdx.x == 0) {
        const double4 po = d.pos[(size_t)r * d.N + w.alch[0]];
        if ((double)water_distance(d, po, c) > w.radius && w.state[(size_t)r * 4 + 3] != 0.0) d.g[r].protocol_work = 999999.0;
    }
}

// external work after a coordinate change between steps (blues/integrators.py:184-191):
// protocol_work += perturbed_pe - unperturbed_pe, using the energies of the evaluation that just finished
__global__ void k_external_work(Dev d, int slot, int first_step_only) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= d.R) return;
    Globals& g = d.g[r];
    g.e_env = env_energy(d, r);
    const double e = g.e_env + alch_energy(d, r, slot);
    g.perturbed_pe = e;
    if (g.first_step < 1 || first_step_only) {
        g.first_step = 1;
        g.unperturbed_pe = e;
    } else if (g.e_valid) {
        g.protocol_work += e - g.unperturbed_pe;
    }
    g.e_total_prev = e;
    g.unperturbed_pe = e;
    g.e_valid = 1;
}

// reset block of the step == 0 branch (blues/integrators.py:165-172) after the energies were evaluated
__global__ void k_reset_protocol(Dev d) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= d.R) return;
    Globals& g = d.g[r];
    g.protocol_work = 0.0;
    g.lambda = 0.0;
    g.lambda_step = 0;
}

// Metropolis test on the device: accept iff logp + correction > log(u)  (blues/simulation.py:1130-1140)
__global__ void k_accept(Dev d, double kT, const double* correction, int* accepted, double* logp_out, double* logu_out,
                         uint64_t seed) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= d.R) return;
    Globals& g = d.g[r];
    double w = -(g.protocol_work + g.shadow_work) / kT;
    if (g.nan_flag) w = __longlong_as_double(0x7ff8000000000000LL);
    Philox4 u = philox4x32_10(0u, g.accept_counter, (uint32_t)r, STREAM_ACCEPT, (uint32_t)seed, (uint32_t)(seed >> 32));
    const double lu = log(u01(u.x));
    if (!isnan(w) && correction) w += correction[r];
    accepted[r] = (w > lu) ? 1 : 0;
    logp_out[r] = w;
    logu_out[r] = lu;
}

// steepest-descent displacement with a per-atom cap, constraints re-imposed per cluster (bl_minimize)
__global__ void __launch_bounds__(128) k_minimize_step(Dev d, double step, double maxdisp, double tol, double4* saved) {
    const int r = blockIdx.y;
    const int cid = blockIdx.x * blockDim.x + threadIdx.x;
    if (cid >= d.n_clusters) return;
    const Cluster c = d.clusters[cid];
    const int N = d.N;
    double4* pos = d.pos + (size_t)r * N;
    const long long* fenv = d.f_env + (size_t)r * 3 * N;
    ClusterState s;
    double xref[MAX_CLUSTER_ATOMS][3];
    for (int k = 0; k < c.natoms; ++k) {
        const int a = c.atom[k];
        const double4 p = pos[a];
        saved[(size_t)r * N + a] = p;
        s.im[k] = d.invmass[a];
        double f[3];
        for (int q = 0; q < 3; ++q) f[q] = (double)fenv[q * N + a] * (1.0 / FORCE_SCALE);
        if (d.alch_on) {
            const long long* fa = d.f_alch + (size_t)r * 3 * N;
            for (int q = 0; q < 3; ++q) f[q] += (double)fa[q * N + a] * (1.0 / FORCE_SCALE);
        }
        double disp[3] = {step * f[0], step * f[1], step * f[2]};
        const double dn = sqrt(disp[0] * disp[0] + disp[1] * disp[1] + disp[2] * disp[2]);
        const double sc = (dn > maxdisp) ? maxdisp / dn : 1.0;
        const double mob = s.im[k] > 0.0 ? 1.0 : 0.0;
        xref[k][0] = p.x; xref[k][1] = p.y; xref[k][2] = p.z;
        s.x[k][0] = p.x + mob * sc * disp[0];
        s.x[k][1] = p.y + mob * sc * disp[1];
        s.x[k][2] = p.z + mob * sc * disp[2];
        s.v[k][0] = s.v[k][1] = s.v[k][2] = 0.0;
    }
    constrain_positions(c, s, xref, tol);
    for (int k = 0; k < c.natoms; ++k) pos[c.atom[k]] = make_double4(s.x[k][0], s.x[k][1], s.x[k][2], 0.0);
}

__global__ void k_restore_positions(Dev d, const double4* saved, const int* reject) {
    const int r = blockIdx.y;
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= d.N || !reject[r]) return;
    d.pos[(size_t)r * d.N + a] = saved[(size_t)r * d.N + a];
}

__global__ void k_max_force(Dev d, double* out) {
    const int r = blockIdx.y;
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    double f2 = 0.0;
    if (a < d.N && d.invmass[a] > 0.0) {
        const long long* fenv = d.f_env + (size_t)r * 3 * d.N;
        for (int q = 0; q < 3; ++q) {
            double f = (double)fenv[q * d.N + a] * (1.0 / FORCE_SCALE);
            if (d.alch_on) f += (double)d.f_alch[(size_t)r * 3 * d.N + q * d.N + a] * (1.0 / FORCE_SCALE);
            f2 += f * f;
        }
    }
    for (int o = 16; o > 0; o >>= 1) f2 = fmax(f2, __shfl_xor_sync(0xffffffffu, f2, o));
    if ((threadIdx.x & 31) == 0) atomicMax(reinterpret_cast<unsigned long long*>(&out[r]), (unsigned long long)__double_as_longlong(f2));
}
