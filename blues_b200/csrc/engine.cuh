// Device-side data layout of one engine handle (R independent walkers of the same N-atom system).
#pragma once
#include "common.cuh"

#define MAX_CLUSTER_ATOMS 5
#define MAX_CLUSTER_CONS 4
#define N_ETERMS 12
#define MAX_OPS 16
#define ALCH_SLOTS 3
#define MAX_NOISE_SETS 4              /* thermostat ops (O / MD) per INTEGRATE launch */
#define EWK_DEG 14
#define MAX_ALCH_SMEM 512             /* alchemical atoms staged in shared memory by k_alch                 */

enum EnergyTerm { E_BOND = 0, E_ANGLE, E_TORSION, E_RESTRAINT, E_PAIR, E_EXCEPT, E_PME, E_SELF, E_DISP,
                  E_ALCH_STERICS, E_ALCH_ELEC, E_ALCH_EXC };

enum OpKind { OP_NONE = 0, OP_CM, OP_V, OP_R, OP_O, OP_H, OP_MD, OP_CONSTRAIN, OP_STEP_BEGIN, OP_STEP_END };

struct Op { int kind; int slot; };

// Constraint cluster: atoms that share holonomic constraints (water triangle, heavy atom + its hydrogens) or a
// single unconstrained atom.  One thread integrates one cluster through the whole V/R/O sequence.
struct Cluster {
    int natoms, ncons;
    int shape;                                                // 0 star around atom 0, 1 water triangle, 2 generic
    int atom[MAX_CLUSTER_ATOMS];
    signed char ca[MAX_CLUSTER_CONS], cb[MAX_CLUSTER_CONS];   // local atom indices of each constraint
    double d2[MAX_CLUSTER_CONS];                              // squared constraint lengths
};

// Per-walker integrator globals (the CustomIntegrator global variables of blues/integrators.py:124-145 plus
// engine bookkeeping).  Doubles so host get/set round-trips are exact.
struct Globals {
    double protocol_work, shadow_work, heat, perturbed_pe, unperturbed_pe, Eold, Enew, lambda;
    double e_env;            // environment (lambda-independent) potential energy at the last energy-enabled evaluation
    double e_total_prev;     // total potential energy recorded at the end of the last completed step
    int lambda_step, step, first_step, prop, debug;
    int alch_base;           // lambda_step for which alchemical slot 0 was evaluated
    int e_valid;             // e_total_prev is valid
    int nan_flag;
    unsigned int noise_counter, vel_counter, move_counter, accept_counter, md_counter;
    int do_rebuild, rebuild_request;   // Verlet list rebuild latched for this evaluation / requested by the host (2)
    int do_prune, prune_request;       // alchemical list follows do_rebuild / some atom moved > skin / 2
    long long n_rebuilds;
    int item_overflow;        // a neighbour list ran out of capacity
    int n_groups, build_cursor;   // k_build_list work queue: groups of <= 8 sorted atoms, next group to fetch
};

struct IntegratorConsts {
    double dt, kT, gamma;
    double hV, hR, hO;                 // substep lengths dt/n_V, dt/n_R, dt/n_O
    double a, b;                       // O-step coefficients
    double md_vscale, md_fscale, md_nscale;
    double tol;
    int n_lambda_steps, nsteps, nprop;
    double total_mass;
    int remove_cm;
    uint64_t seed;
};

struct Dev {
    int N, Npad, nblocks, R;
    int periodic, pme, nb_method;
    // box (device memory so CUDA graphs survive bl_set_box): [0..2] L, [3..5] 1/L as double; floats mirror
    double* boxd;
    float* boxf;
    float cutoff, cutoff2, list_cutoff2, skin_half2, alpha, krf, crf;
    // Ewald real-space force without exp / erfc: F = qq (1/r^3 - alpha^3 k(alpha^2 r^2)), k(z) = (erf(sqrt z)/sqrt z -
    // 2/sqrt(pi) exp(-z)) / z as a degree-EWK_DEG polynomial in t = ewk_scale r^2 - 1 on [0, (alpha rc)^2] (fitted at bl_create)
    float ewk[16]; float ewk_scale, alpha3; int ewk_ok;
    float ewk2[16]; int ewk2_deg;           // the same fit at the lowest degree float rounding allows (k_pair4)
    double cutoffd, alphad;
    // static per-atom data (original order)
    double* mass; double* invmass;
    double* charge_d; double* sigma_d; double* eps_d;   // double-precision parameters for the alchemical kernel
    float* charge; float2* sigeps;          // sigeps: (sigma/2, 2 sqrt(eps)) so sigma_ij = s_i+s_j, 4 eps_ij = e_i e_j
    ull* excl_win;                          // bit (j - i + 32) set if pair (i, j) is excluded / an exception
    unsigned char* has_far;                 // atom has exclusions outside the +-32 index window
    long long* far_codes; int n_far;        // sorted i*N+j (i<j) codes of those far exclusions
    // dynamic state
    double4* pos; double4* vel;             // [R*N]
    float4* posq;                           // [R*N] single-precision mirror (x, y, z, q)
    float4* pos_ref;                        // [R*N] positions at the last neighbour rebuild
    long long* f_env;                       // [R][3][N] fixed point
    long long* f_alch;                      // [ALCH_SLOTS][R][3][N]
    long long* eacc;                        // [R][N_ETERMS]
    long long* alch_acc;                    // [R][ALCH_SLOTS][3]  (sterics, electrostatics, exceptions)
    long long* cm_acc;                      // [R][3] sum of m v
    long long* heat_acc;                    // [R]
    Globals* g;                             // [R]
    int* cta_done;                          // [R] k_integrate CTAs of the walker that have finished (pre-evaluation launches)
    double* noise;                          // [R][MAX_NOISE_SETS][N][3] standard normals for the next INTEGRATE launch
    // neighbour structures: Morton-ranked cells (edge >= list cutoff / 2), sorted mirrors, Verlet lists
    int ncell[3]; int ncells;
    int zreach;                             // cells that cover the list cutoff along z: 2, or 2 k with k-times finer z cells
    int* cell_order;                        // [ncells] Morton rank of each cell
    int* cell_start; int* cell_cursor;      // [R][ncells+1] first sorted slot of every cell (+ scatter cursor)
    int* atom_cell;                         // [R*N]
    int* group_first; int group_capacity;   // [R][group_capacity] (first sorted index << 4 | atoms) of every build group
    int* rank;                              // [R*N] position of atom a in the sorted order
    float4* posq_s; float2* sigeps_s; int* orig_s;   // [R*Npad] sorted copies (pads: NaN position, orig -1)
    int nl_M;                               // capacity of one row of the Verlet list
    int* nl_count;                          // [R*Npad]
    void* nl_list;                          // [R*Npad][nl_M] sorted indices of the neighbours within cutoff + skin
    int nl_u16;                             // indices stored as uint16 (Npad < 65536) to halve the list traffic
    unsigned char* mobile_s;                // [R*Npad] sorted atom has a mass (frozen rows are skipped by force-only pair launches)
    int n_frozen;                           // atoms with mass 0 (freeze_radius / freeze_atoms, blues/simulation.py:364-480)
    // bonded tables
    int n_bonds, n_angles, n_torsions, n_excl, n_restraints, n_alch_exc;
    int2* bonds; double2* bond_p;           // (k, r0)
    int4* angles; double2* angle_p;         // (k, theta0)   (w unused)
    int4* torsions; double4* torsion_p;     // (k, n, phase, -)
    int2* excl; double4* excl_p;            // (k_e*qq_exception, sigma, eps, k_e*q_i*q_j)
    int* restraint_atom; double4* restraint_p;   // (x0, y0, z0, k)
    int2* alch_exc; double4* alch_exc_p;    // (k_e*qq, sigma, eps, both_alchemical)
    // alchemical region
    int n_alch;
    int* alch_atom; double4* alch_p;        // (q, sigma, eps, -)
    unsigned char* is_alch;                 // [N]
    int alch_cap; int* alch_count; int* alch_list;   // per-alchemical-atom neighbour lists: [R][n_alch], [R][n_alch][alch_cap]
    double sc_alpha, sc_a, sc_b, sc_c;
    int annihilate_sterics, annihilate_elec;
    double* lam_s; double* lam_e; int n_lambda;       // tables indexed by lambda_step
    // generic Custom*Force terms (bl_topology::custom_*): evaluated per alchemical slot by k_custom
    int n_custom, custom_np;
    int4* custom_term; double* custom_cutoff; double* custom_params;
    int* custom_gstart; int* custom_gatoms; double* custom_gweights;
    int* custom_pstart; int* custom_op; double* custom_arg;
    int alch_on;                            // lambda-dependent force slots in use: n_alch > 0 or n_custom > 0
    // PME
    int gx, gy, gz; int gsize; int csize;   // real grid size, complex grid size (gx*gy*(gz/2+1))
    float* grid_r;                          // [R][gsize]
    float2* grid_c;                         // [R][csize]
    // charge grid of the frozen atoms (mass 0) in k_pme_spread's fixed point: they never move, so their share of every
    // plane is computed once per coordinate upload and the later launches start from it instead of from zero
    int* grid_frozen;                       // [R][gsize], null when nothing is frozen
    int* frozen_grid_state;                 // [R] 0: rebuild in the next spread launch, 1: valid
    float* bmod_x; float* bmod_y; float* bmod_z;
    double self_energy_coeff;               // -k_e alpha/sqrt(pi) sum q^2  (constant)
    double sumq;
    double dispersion_coeff;
    // integrator clusters
    int n_clusters;
    Cluster* clusters;
};
