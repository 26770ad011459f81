// libblues_b200.so — host side of the C ABI declared in include/blues_b200.h.
// Owns device memory, builds the per-step launch program from the splitting string, captures it into CUDA
// graphs and replays it without host round-trips.  No CPU fallback: every entry point needs a CUDA device.
#include <cuda_runtime.h>
#include <cufft.h>
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/blues_b200.h"
#include "engine.cuh"
#include "kernels_nb.cuh"
#include "kernels_bonded.cuh"
#include "kernels_pme.cuh"
#include "kernels_integrate.cuh"

static std::string g_create_error;

// cudaFuncAttributeMaxDynamicSharedMemorySize is a property of the function on a device, shared by every handle of the
// process: a later handle with a smaller need must not lower it under an earlier handle's launches (BASELINE configs[2]
// next to configs[1] in one process: the 64-walker builder uses smaller write-combining buffers than the 1-walker one)
template <class F> static void raise_dyn_smem(F* func, int device, size_t bytes) {
    static std::mutex mu;
    static std::map<std::pair<int, const void*>, size_t> cur;
    std::lock_guard<std::mutex> lock(mu);
    size_t& c = cur[{device, (const void*)func}];
    if (bytes > c) {
        cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        c = bytes;
    }
}

struct TimedLaunch { int kid; cudaEvent_t e0, e1; };

struct bl_handle {
    Dev d;
    IntegratorConsts ic;
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;   // reciprocal-space branch, forked from / joined to `stream` inside every evaluation
    cudaStream_t stream3 = nullptr, stream4 = nullptr;   // bonded branch, alchemical branch
    cudaStream_t stream5 = nullptr; cudaEvent_t ev_join5 = nullptr;   // pair kernel of the walkers that do not rebuild (many walkers)
    int pair_split = 0;          // BLUES_B200_PAIR_SPLIT=1: > 2 walkers: pair kernel of the non-rebuilding walkers beside the builder
                                 // (measured: 617 vs 610 us per 8-walker step — both kernels are issue bound, the overlap buys nothing)
    cudaEvent_t ev_fork = nullptr, ev_fork2 = nullptr, ev_join = nullptr, ev_join3 = nullptr, ev_join4 = nullptr;
    std::string error;
    std::vector<void*> allocs;
    // host copies needed after creation
    int integrator_kind = 0;
    std::vector<std::string> splitting;
    int n_H = 0;
    double prop_lambda_min = 2.0, prop_lambda_max = -1.0;
    std::vector<double> lam_s_host, lam_e_host;
    double temperature = 300.0;
    // lock-step host mirror of the per-walker program counters
    int step = 0, lambda_step = 0, first_step = 0;
    int cursor = 0;               // alchemical slot holding the energy/forces of the current lambda_step
    bool forces_valid = false;    // f_env / slots match the current positions
    bool forces_partial = false;  // ... but the last evaluation skipped the rows of the frozen atoms (enqueue_eval)
    bool skip_frozen = true;
    int zfine = 2;               // BLUES_B200_ZFINE: z resolution of the search cells (plan_cells); 2 measured +2 % over 1, 3 = 2
    bool work_pending = false;    // coordinates changed outside the integrator since the last external-work evaluation
    bool vel_dirty = true;        // cm_acc must be recomputed
    int* cm_parity = nullptr;     // device int
    int n_cons_total = 0;
    int n_generic = 0;            // clusters handled by the dynamic-index fallback kernel (sorted first)
    // cuFFT
    cufftHandle plan_r2c = 0, plan_c2r = 0;
    bool has_fft = false;
    // graphs
    bool use_graphs = true;
    std::map<std::string, cudaGraphExec_t> graphs;
    // profiling
    bool profiling = false;
    std::vector<TimedLaunch> timed;
    double ktime[BL_NUM_KERNEL_IDS] = {0};
    long long kcount[BL_NUM_KERNEL_IDS] = {0};
    unsigned long long launches = 0;
    bool capturing = false;
    unsigned long long capture_launches = 0;
    // scratch
    double* d_scratch = nullptr;   // [R*4] doubles
    int* d_iscratch = nullptr;     // [R*2]
    double4* d_saved = nullptr;    // minimizer
    int* d_move_atoms = nullptr; float* d_move_masses = nullptr; int move_capacity = 0;
    // WaterTranslationMove: candidate waters, protein selection, per-walker {sphere centre, go}
    int* d_water_atoms = nullptr; size_t water_capacity = 0;
    int* d_center_atoms = nullptr; float* d_center_masses = nullptr; int center_capacity = 0;
    double* d_water_state = nullptr;
    std::vector<double> host_tmp;
    double skin = 0.0; int cell_capacity = 0;
    int build_cq = 0, build_ctas = 0;
    bool debug_sync = false, debug_reported = false;   // BLUES_B200_DEBUG_SYNC
    int int_block = 32;          // BLUES_B200_INT_BLOCK: threads per k_integrate CTA (one constraint cluster per thread)
    bool fold_zero = true;       // step programs: force zeroing + rebuild latch inside the INTEGRATE launch before an evaluation
    int spread_split = 0;        // BLUES_B200_SPREAD_SPLIT: y-bands per x-plane of k_pme_spread at <= 2 walkers (0: one wave, see bl_create)
    int spread_threads = 1024;   // BLUES_B200_SPREAD_THREADS: 512 or 1024
    int pair_per_sm = 0, n_sm = 148;   // BLUES_B200_PAIR_PER_SM: resident k_pair4 CTAs per SM (0: one CTA per row block)
    int pair_lanes = 8;          // BLUES_B200_PAIR_LANES: lanes per i-atom in k_pair4 (8, 16, 32)
    int pair_x2 = 2;             // BLUES_B200_PAIR_X2: 0 off, 2 / 4 = k_pair4 (packed FFMA2 arithmetic) with that many entries per trip
    int graph_steps = 4;         // plain NCMC steps captured per CUDA graph
    bool pdl = true;             // programmatic dependent launch on the B -> flip -> A -> sort edges (BLUES_B200_PDL=0: off)
    // diagnostic timeline (BLUES_B200_TIMELINE=1): events recorded inside the step graphs, read after every replay
    bool timeline = false; cudaEvent_t tl_ev[24] = {}; double tl_sum[24] = {}; long tl_n[24] = {}; int tl_int = 0;
    double4* pinned = nullptr;     // pinned staging for state uploads / downloads ([N] double4)
};

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            char buf_[512];                                                                        \
            snprintf(buf_, sizeof buf_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            h->error = buf_;                                                                       \
            return BL_ERR_CUDA;                                                                    \
        }                                                                                          \
    } while (0)

template <typename T>
static T* dalloc(bl_handle* h, size_t n) {
    void* p = nullptr;
    if (n == 0) n = 1;
    if (cudaMalloc(&p, n * sizeof(T)) != cudaSuccess) return nullptr;
    // cudaMemset on device memory is asynchronous and runs in the legacy stream, with which the handle's non-blocking
    // streams are NOT ordered: without the synchronisation a buffer allocated lazily (move staging, water state, grown
    // cell tables) could be zeroed AFTER the first asynchronous upload into it.  Seen as NaN work of every walker of a rank
    // in the first iteration when two processes shared one GPU (tests/test_gpu_two_ranks.py).
    cudaMemset(p, 0, n * sizeof(T));
    cudaStreamSynchronize(cudaStreamLegacy);
    h->allocs.push_back(p);
    return static_cast<T*>(p);
}
static void dfree(bl_handle* h, void* p) {
    if (!p) return;
    auto it = std::find(h->allocs.begin(), h->allocs.end(), p);
    if (it != h->allocs.end()) h->allocs.erase(it);
    cudaFree(p);
}
template <typename T>
static T* dupload(bl_handle* h, const std::vector<T>& v) {
    T* p = dalloc<T>(h, v.size());
    if (p && !v.empty()) cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
    return p;
}

// ---- launch helper with optional per-kernel event timing -------------------------------------------------
struct LaunchTimer {
    bl_handle* h; int kid; cudaStream_t st; cudaEvent_t e0 = nullptr, e1 = nullptr; int line;
    LaunchTimer(bl_handle* h_, int kid_, cudaStream_t st_ = nullptr, int line_ = __builtin_LINE())
        : h(h_), kid(kid_), st(st_ ? st_ : h_->stream), line(line_) {
        if (h->capturing) h->capture_launches++; else h->launches++;
        if (h->profiling && !h->capturing && kid >= 0) {
            cudaEventCreate(&e0); cudaEventCreate(&e1);
            cudaEventRecord(e0, st);
        }
    }
    ~LaunchTimer() {
        if (e0) { cudaEventRecord(e1, st); h->timed.push_back({kid, e0, e1}); }
        if (h->debug_sync && !h->capturing) {
            // BLUES_B200_DEBUG_SYNC=1 (diagnostic): direct launches, every one followed by a synchronisation, so that a
            // device fault is reported at the launch that caused it
            const cudaError_t e = cudaStreamSynchronize(st);
            if (e != cudaSuccess && !h->debug_reported) {
                h->debug_reported = true;
                fprintf(stderr, "[blues_b200 debug] launch at engine.cu:%d (timer id %d, launch #%llu, step %d) failed: %s\n", line,
                        kid, h->launches, h->step, cudaGetErrorString(e));
            }
        }
    }
};
static void collect_timings(bl_handle* h) {
    for (auto& t : h->timed) {
        float ms = 0.f;
        cudaEventSynchronize(t.e1);
        cudaEventElapsedTime(&ms, t.e0, t.e1);
        h->ktime[t.kid] += ms;
        h->kcount[t.kid] += 1;
        cudaEventDestroy(t.e0); cudaEventDestroy(t.e1);
    }
    h->timed.clear();
}

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

enum { TL_START = 0, TL_SORT, TL_ZERO, TL_BUILD, TL_PAIR, TL_SPREAD, TL_R2C, TL_CONV, TL_C2R, TL_GATHER, TL_BONDED, TL_ALCH,
       TL_JOINED, TL_INT0, TL_INT1, TL_INT2, TL_COUNT };
static const char* TL_NAMES[] = {"step start", "sort done", "zero done", "build done", "pair done", "pme spread done",
                                 "pme r2c done", "pme convolve done", "pme c2r done", "pme gather done", "bonded+noise done",
                                 "alch done", "eval joined", "integrate #1 done", "integrate #2 done", "integrate #3 done"};
static void tl_mark(bl_handle* h, cudaStream_t st, int id) {
    if (!h->timeline || id >= TL_COUNT) return;
    if (!h->tl_ev[id]) cudaEventCreate(&h->tl_ev[id]);
    if (h->capturing) cudaEventRecordWithFlags(h->tl_ev[id], st, cudaEventRecordExternal);
    else cudaEventRecord(h->tl_ev[id], st);
}
static void tl_collect(bl_handle* h) {
    if (!h->timeline || !h->tl_ev[TL_START]) return;
    cudaStreamSynchronize(h->stream);
    for (int id = 1; id < TL_COUNT; ++id) {
        if (!h->tl_ev[id]) continue;
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, h->tl_ev[TL_START], h->tl_ev[id]) == cudaSuccess && ms >= 0.f) {
            h->tl_sum[id] += ms * 1e3;
            h->tl_n[id] = labs(h->tl_n[id]) + 1;
        }
    }
    cudaGetLastError();
}
static void tl_report(bl_handle* h) {
    if (!h->timeline) return;
    fprintf(stderr, "[blues_b200 timeline] mean microseconds after step start (graph replays, one step per graph)\n");
    for (int id = 1; id < TL_COUNT; ++id)
        if (labs(h->tl_n[id]) > 0) fprintf(stderr, "    %-22s %8.1f   (n = %ld)\n", TL_NAMES[id], h->tl_sum[id] / labs(h->tl_n[id]), labs(h->tl_n[id]));
}

// Launch with the programmatic-stream-serialization attribute: the kernel may be scheduled while its stream
// predecessor is still running and blocks in cudaGridDependencySynchronize() until that one has completed, which takes
// the launch latency off the dependent chain.  Only used on edges whose consumer waits at its very first instruction.
template <typename... KArgs, typename... Args>
static void launch_pdl(bl_handle* h, void (*kernel)(KArgs...), dim3 grid, dim3 block, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = 0; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = h->pdl ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, args...);
}

// k_pair2 launch of an evaluation that k_pair4 does not take.  PME uses the polynomial Ewald force (EWALD 1) wherever
// its fit holds (Dev::ewk_ok); reaction field and no-cutoff have no Ewald term.
template <int METHOD, bool ENERGY>
static void launch_pair2(const Dev& d, cudaStream_t st, int skip) {
    const dim3 grid(cdiv((long long)d.Npad * NL_LANES, NL_BLOCK), d.R);
    if constexpr (METHOD == NB_PME) {
        if (d.ewk_ok) {
            if (d.nl_u16) k_pair2<METHOD, ENERGY, unsigned short, 1><<<grid, NL_BLOCK, 0, st>>>(d, skip);
            else k_pair2<METHOD, ENERGY, int, 1><<<grid, NL_BLOCK, 0, st>>>(d, skip);
            return;
        }
    }
    if (d.nl_u16) k_pair2<METHOD, ENERGY, unsigned short, 0><<<grid, NL_BLOCK, 0, st>>>(d, skip);
    else k_pair2<METHOD, ENERGY, int, 0><<<grid, NL_BLOCK, 0, st>>>(d, skip);
}

// ---- force / energy evaluation at the current positions ---------------------------------------------------
// energy: also accumulate energies; cm_mode: forwarded to k_begin_eval
// pre_zeroed: the preceding INTEGRATE launch ran with IntegrateArgs::pre_eval (forces cleared, rebuild latched, counters
// advanced): no k_begin_eval
static void enqueue_eval(bl_handle* h, bool energy, int adv_noise, int adv_md, int cm_mode, int prefetch_noise = 0,
                         bool pre_zeroed = false, bool in_program = false) {
    Dev& d = h->d;
    cudaStream_t st = h->stream;
    const int R = d.R, N = d.N;
    // frozen atoms (mass 0): force-only evaluations inside a step program leave their rows out (BLUES_B200_SKIP_FROZEN=0:
    // off).  The forces then cover the mobile atoms only; a host force query re-evaluates in full (forces_partial).
    const int skip = (in_program && !energy && h->skip_frozen && d.n_frozen > 0) ? 1 : 0;
    h->forces_partial = skip != 0;
    {
        // latches the rebuild request (unless the integrator did), then (only if due) the cell sort
        LaunchTimer t(h, BL_K_NEIGHBOR);
        launch_pdl(h, k_sort_atoms, dim3(SORT_CTAS, R), dim3(1024), st, d, pre_zeroed ? 1 : 0, cm_mode, h->cm_parity);
    }
    tl_mark(h, st, TL_SORT);
    // Fork 1: reciprocal space (stream2) depends only on the cell-sorted positions; its gather waits for fork 2.
    cudaEventRecord(h->ev_fork, st);
    if (!pre_zeroed) {
        LaunchTimer t(h, -1);
        long long nf = (long long)R * 3 * N * (d.alch_on ? 1 + ALCH_SLOTS : 1);
        int blocks = std::max(1, std::min(cdiv(nf, 256 * 4), 148 * 8));
        k_begin_eval<<<blocks, 256, 0, st>>>(d, adv_noise, adv_md, cm_mode, h->cm_parity);
    }
    // Fork 2: force accumulators are zeroed and the noise counters advanced.  Branches: bonded terms + noise prefetch
    // (stream3), alchemical lists + kernel (stream4); the main stream keeps the list build and the pair kernel.  All
    // branches accumulate into the same fixed-point buffers with atomics.
    cudaEventRecord(h->ev_fork2, st);
    tl_mark(h, st, TL_ZERO);
    const bool pme = d.pme && h->has_fft;
    const int nterms = d.n_bonds + d.n_angles + d.n_torsions + d.n_excl + d.n_restraints + d.n_alch_exc;
    if (pme) {
        cudaStream_t s2 = h->profiling ? st : h->stream2;
        cufftSetStream(h->plan_r2c, s2);
        cufftSetStream(h->plan_c2r, s2);
        cudaStreamWaitEvent(s2, h->ev_fork, 0);
        const int fcache = d.grid_frozen ? 1 : 0;      // frozen atoms' share of the charge grid is kept (k_pme_spread)
        { LaunchTimer t(h, BL_K_PME_SPREAD, s2);
          // few walkers: latency bound, many wide CTAs; many walkers: throughput bound, fewer duplicate B-splines
          if (R <= 2) {
              const int ys = h->spread_split;
              const size_t sm = (size_t)(d.gy / ys + 1) * d.gz * sizeof(int) * (fcache ? 2 : 1);
              if (h->spread_threads == 1024) k_pme_spread<1024><<<dim3(d.gx, ys, R), 1024, sm, s2>>>(d, fcache);
              else k_pme_spread<512><<<dim3(d.gx, ys, R), 512, sm, s2>>>(d, fcache);
          } else k_pme_spread<256><<<dim3(d.gx, 4, R), 256, (size_t)(d.gy / 4 + 1) * d.gz * sizeof(int) * (fcache ? 2 : 1), s2>>>(d, fcache); }
        tl_mark(h, s2, TL_SPREAD);
        { LaunchTimer t(h, BL_K_FFT, s2); cufftExecR2C(h->plan_r2c, d.grid_r, reinterpret_cast<cufftComplex*>(d.grid_c)); }
        tl_mark(h, s2, TL_R2C);
        { LaunchTimer t(h, BL_K_PME_CONVOLVE, s2);
          if (energy) k_pme_convolve<true><<<dim3(cdiv(d.csize, 256), R), 256, 0, s2>>>(d);
          else k_pme_convolve<false><<<dim3(cdiv(d.csize, 256), R), 256, 0, s2>>>(d); }
        tl_mark(h, s2, TL_CONV);
        { LaunchTimer t(h, BL_K_FFT, s2); cufftExecC2R(h->plan_c2r, reinterpret_cast<cufftComplex*>(d.grid_c), d.grid_r); }
        tl_mark(h, s2, TL_C2R);
        if (!h->profiling) cudaStreamWaitEvent(s2, h->ev_fork2, 0);      // the gather adds to the cleared force accumulators
        { LaunchTimer t(h, BL_K_PME_GATHER, s2);
          if (R <= 2) k_pme_gather5<<<dim3(cdiv(cdiv(N, 6) * 32, 128), R), 128, 0, s2>>>(d, skip);
          else k_pme_gather<<<dim3(cdiv(N, 128), R), 128, 0, s2>>>(d, skip); }
        tl_mark(h, s2, TL_GATHER);
        cudaEventRecord(h->ev_join, s2);
    }
    if (nterms > 0 || prefetch_noise > 0) {
        cudaStream_t s3 = h->profiling ? st : h->stream3;
        cudaStreamWaitEvent(s3, h->ev_fork2, 0);
        if (nterms > 0) { LaunchTimer t(h, BL_K_BONDED, s3); k_bonded<<<dim3(cdiv(nterms, 128), R), 128, 0, s3>>>(d); }
        if (prefetch_noise > 0) {
            // thermostat kicks of the next INTEGRATE launch with O steps: k_begin_eval above has advanced the noise
            // counter past everything consumed so far, so sets 0.. at offset 0 are exactly what that launch will read
            LaunchTimer t(h, BL_K_INTEGRATE, s3);
            k_noise<<<dim3(cdiv((long long)N * prefetch_noise, 128), R), 128, 0, s3>>>(d, h->ic, STREAM_LANGEVIN, prefetch_noise, 0);
        }
        tl_mark(h, s3, TL_BONDED);
        cudaEventRecord(h->ev_join3, s3);
    }
    if (d.alch_on) {
        cudaStream_t s4 = h->profiling ? st : h->stream4;
        cudaStreamWaitEvent(s4, h->ev_fork2, 0);
        if (d.n_alch > 0) {
            { LaunchTimer t(h, BL_K_NEIGHBOR, s4); k_alch_reset<<<cdiv(R * d.n_alch, 128), 128, 0, s4>>>(d); }
            { LaunchTimer t(h, BL_K_NEIGHBOR, s4);
              k_alch_list<<<dim3(cdiv(N, 128), R), 128, d.n_alch * sizeof(float4), s4>>>(d); }
            { LaunchTimer t(h, BL_K_NEIGHBOR, s4); k_alch_sort<<<dim3(d.n_alch, R), 512, 0, s4>>>(d); }
            { LaunchTimer t(h, BL_K_ALCH, s4); k_alch<<<dim3(cdiv(d.alch_cap, 128), d.n_alch, R), 128, 0, s4>>>(d); }
        }
        if (d.n_custom > 0) { LaunchTimer t(h, BL_K_ALCH, s4); k_custom<<<dim3(cdiv(d.n_custom, 64), R), 64, 0, s4>>>(d); }
        tl_mark(h, s4, TL_ALCH);
        cudaEventRecord(h->ev_join4, s4);
    }
    // packed-pair FP32 kernel (FFMA2): PME force-only evaluations, i.e. every evaluation of a plain NCMC / MD step
    const bool use_x2 = h->pair_x2 && !energy && d.nb_method == 4 && d.ewk_ok && d.ewk2_deg <= 12;
    auto launch_pair4 = [&](cudaStream_t ps, int phase) {
        LaunchTimer t(h, BL_K_PAIR, ps);
        const int U = h->pair_x2 == 4 ? 4 : 2;
        const int lanes = h->pair_lanes;
        dim3 grid(cdiv((long long)d.Npad * lanes, NL_BLOCK), R);
        if (h->pair_per_sm > 0) grid.x = std::min<unsigned>(grid.x, (unsigned)std::max(1, h->pair_per_sm * h->n_sm / R));
#define PX3(T, L, UU, DG) k_pair4<T, L, UU, DG><<<grid, NL_BLOCK, 0, ps>>>(d, skip, phase)
#define PX2(T, UU, DG) if (lanes == 16) PX3(T, 16, UU, DG); else if (lanes == 32) PX3(T, 32, UU, DG); else if (lanes == 4) PX3(T, 4, UU, DG); else PX3(T, 8, UU, DG)
#define PX1(T, UU) if (d.ewk2_deg == 10) { PX2(T, UU, 10); } else { PX2(T, UU, 12); }
#define PX0(T) if (U == 4) { PX1(T, 4) } else { PX1(T, 2) }
        if (d.nl_u16) { PX0(unsigned short) } else { PX0(int) }
#undef PX3
#undef PX2
#undef PX1
#undef PX0
    };
    // many walkers: each rebuilds its list on its own schedule (every ~4 steps), so in a typical evaluation a quarter of the
    // walkers wait for the builder and the others do not — their pair kernel runs beside the builder on its own stream
    const bool split = use_x2 && R > 2 && h->pair_split && !h->profiling;
    if (split) {
        cudaStreamWaitEvent(h->stream5, h->ev_fork2, 0);
        launch_pair4(h->stream5, 1);
        cudaEventRecord(h->ev_join5, h->stream5);
    }
    {
        LaunchTimer t(h, BL_K_NEIGHBOR);
        dim3 grid(h->build_ctas);                          // persistent single-warp CTAs shared by all walkers
        const size_t smem = build_smem_bytes(h->build_cq, d.nl_u16 ? 2 : 4);
        if (d.nl_u16) k_build_list<unsigned short><<<grid, 32, smem, st>>>(d, h->build_cq);
        else k_build_list<int><<<grid, 32, smem, st>>>(d, h->build_cq);
    }
    tl_mark(h, st, TL_BUILD);
    if (use_x2) {
        launch_pair4(st, split ? 2 : 0);
        if (split) cudaStreamWaitEvent(st, h->ev_join5, 0);
    } else {
        LaunchTimer t(h, BL_K_PAIR);
        if (d.nb_method == NB_PME) { if (energy) launch_pair2<NB_PME, true>(d, st, skip); else launch_pair2<NB_PME, false>(d, st, skip); }
        else if (d.nb_method == NB_RF) { if (energy) launch_pair2<NB_RF, true>(d, st, skip); else launch_pair2<NB_RF, false>(d, st, skip); }
        else { if (energy) launch_pair2<NB_NOCUT, true>(d, st, skip); else launch_pair2<NB_NOCUT, false>(d, st, skip); }
    }
    tl_mark(h, st, TL_PAIR);
    if (pme) cudaStreamWaitEvent(st, h->ev_join, 0);
    if (nterms > 0 || prefetch_noise > 0) cudaStreamWaitEvent(st, h->ev_join3, 0);
    if (d.alch_on) cudaStreamWaitEvent(st, h->ev_join4, 0);
    tl_mark(h, st, TL_JOINED);
}

static void enqueue_integrate(bl_handle* h, const IntegrateArgs& a, bool noise_prefetched) {
    int n_o = 0, n_md = 0;
    for (int k = 0; k < a.nops; ++k) { if (a.ops[k].kind == OP_O) n_o++; if (a.ops[k].kind == OP_MD) n_md++; }
    if (n_o > 0 && !noise_prefetched) {
        LaunchTimer t(h, BL_K_INTEGRATE);
        k_noise<<<dim3(cdiv((long long)h->d.N * n_o, 128), h->d.R), 128, 0, h->stream>>>(h->d, h->ic, STREAM_LANGEVIN, n_o, a.noise_offset);
    }
    if (n_md > 0) {
        LaunchTimer t(h, BL_K_INTEGRATE);
        k_noise<<<dim3(cdiv((long long)h->d.N * n_md, 128), h->d.R), 128, 0, h->stream>>>(h->d, h->ic, STREAM_MD, n_md, a.md_offset);
    }
    if (h->n_generic > 0) {
        // generic clusters are sorted first; they must not also run the bookkeeping ops of the main kernel
        LaunchTimer t(h, BL_K_INTEGRATE);
        k_integrate_generic<<<dim3(cdiv(h->n_generic, 64), h->d.R), 64, 0, h->stream>>>(h->d, h->ic, a, h->cm_parity, h->n_generic);
    }
    LaunchTimer t(h, BL_K_INTEGRATE);
    // + 1: the last CTA holds no clusters (n_clusters is passed to the bounds check) and does the scalar bookkeeping
    launch_pdl(h, k_integrate, dim3(cdiv(h->d.n_clusters, h->int_block) + 1, h->d.R), dim3(h->int_block), h->stream, h->d, h->ic, a,
               (const int*)h->cm_parity);
    tl_mark(h, h->stream, TL_INT0 + std::min(h->tl_int++, 2));
}

static void enqueue_momentum(bl_handle* h) {
    if (!h->ic.remove_cm) return;
    Dev& d = h->d;
    { LaunchTimer t(h, -1); k_zero_ll<<<1, 64, 0, h->stream>>>(d.cm_acc, (size_t)2 * d.R * 3); }
    { LaunchTimer t(h, -1); k_momentum<<<dim3(cdiv(d.N, 128), d.R), 128, 0, h->stream>>>(d, h->cm_parity); }
}

// ---- step-program compilation -----------------------------------------------------------------------------
struct Launch { bool is_eval; bool energy; int cm_mode; int adv_noise; IntegrateArgs args; bool flip_after; };

// Build the launch list of one pass over the splitting string (blues/integrators.py:192,200 → openmmtools
// LangevinIntegrator._add_integrator_steps).  cursor: alchemical slot of the current lambda_step.
static void compile_pass(bl_handle* h, std::vector<Launch>& out, int& cursor, bool h_active, bool last_pass,
                         bool energy_at_end) {
    std::vector<Launch> pass;
    IntegrateArgs cur;
    memset(&cur, 0, sizeof cur);
    auto push_op = [&](int kind, int slot) {
        if (cur.nops >= MAX_OPS) return;
        cur.ops[cur.nops].kind = kind;
        cur.ops[cur.nops].slot = slot;
        cur.nops++;
    };
    auto emit_integrate = [&]() {
        Launch l;
        memset(&l, 0, sizeof l);
        l.is_eval = false;
        l.args = cur;
        pass.push_back(l);
        memset(&cur, 0, sizeof cur);
    };
    auto emit_eval = [&](bool energy) {
        Launch l;
        memset(&l, 0, sizeof l);
        l.is_eval = true;
        l.energy = energy;
        pass.push_back(l);
        cursor = 0;
    };
    push_op(OP_CM, 0);
    bool x_dirty = false;
    for (const std::string& tok : h->splitting) {
        if (tok == "V") {
            if (x_dirty) { emit_integrate(); emit_eval(false); x_dirty = false; }
            push_op(OP_V, cursor);
        } else if (tok == "R") {
            push_op(OP_R, 0);
            x_dirty = true;
        } else if (tok == "O") {
            push_op(OP_O, 0);
        } else if (tok == "H") {
            if (!h_active) continue;
            if (x_dirty) { emit_integrate(); emit_eval(false); x_dirty = false; }
            if (cursor + 1 >= ALCH_SLOTS) { emit_integrate(); emit_eval(false); }
            push_op(OP_H, cursor);
            cursor++;
        }
    }
    if (x_dirty) { emit_integrate(); emit_eval(energy_at_end && last_pass); x_dirty = false; }
    else if (energy_at_end && last_pass) {
        // the last evaluation of this pass must carry energies: mark it
        for (int k = (int)pass.size() - 1; k >= 0; --k)
            if (pass[k].is_eval) { pass[k].energy = true; break; }
    }
    if (last_pass) push_op(OP_STEP_END, cursor);
    emit_integrate();      // every pass ends with an INTEGRATE launch (momentum accumulation lives there)
    // energy_valid for STEP_END: true if the most recent EVAL of the pass carried energies and no H with a
    // re-evaluation invalidated it — alchemical slot energies are always present, e_env only with `energy`
    bool last_eval_energy = false;
    int first_int = -1, last_int = -1;
    for (size_t k = 0; k < pass.size(); ++k) {
        if (pass[k].is_eval) last_eval_energy = pass[k].energy;
        else { if (first_int < 0) first_int = (int)k; last_int = (int)k; }
    }
    pass[last_int].args.energy_valid = last_eval_energy ? 1 : 0;
    // centre-of-mass momentum plumbing
    if (h->ic.remove_cm) {
        bool between = false;
        for (int k = first_int + 1; k < last_int; ++k) if (pass[k].is_eval) between = true;
        if (between && first_int != last_int) {
            for (int k = first_int + 1; k < last_int; ++k) if (pass[k].is_eval) pass[k].cm_mode = 1;
            pass[last_int].args.accum_cm = 1;
        } else {
            pass[last_int].args.accum_cm = 2;
            pass[last_int].flip_after = true;
        }
    }
    for (auto& l : pass) out.push_back(l);
}

// ---- issuing launches, CUDA-graph caching -------------------------------------------------------------------
struct HostCounters {
    int pending_noise = 0, pending_md = 0;
    int noise_ready = 0;      // thermostat noise sets prefetched by the last evaluation, valid at offset 0
};
static std::map<bl_handle*, HostCounters>& counter_map() {
    static std::map<bl_handle*, HostCounters> m;
    return m;
}
static HostCounters& counters(bl_handle* h) { return counter_map()[h]; }

static int count_ops(const IntegrateArgs& a, int kind) {
    int n = 0;
    for (int k = 0; k < a.nops; ++k) n += a.ops[k].kind == kind;
    return n;
}

// O steps of the first noise-consuming INTEGRATE launch after evaluation `k` (wrapping to the start of the list: a step
// program repeats), or 0 if another evaluation or an MD step comes first.  A wrong guess costs nothing: the consumer
// checks hc.noise_ready and falls back to generating its noise inline.
static int noise_lookahead(const std::vector<Launch>& ls, size_t k) {
    for (size_t j = 1; j <= ls.size(); ++j) {
        const Launch& l = ls[(k + j) % ls.size()];
        if (l.is_eval) return 0;
        if (count_ops(l.args, OP_MD) > 0) return 0;
        const int n_o = count_ops(l.args, OP_O);
        if (n_o > 0) return n_o;
    }
    return 0;
}

// Enqueue the launches (dry = false) or only replay their host-side bookkeeping (dry = true, after a graph launch).
static void issue(bl_handle* h, const std::vector<Launch>& ls, HostCounters& hc, bool dry = false) {
    if (!dry) { h->tl_int = 0; tl_mark(h, h->stream, TL_START); }
    for (size_t k = 0; k < ls.size(); ++k) {
        const Launch& l = ls[k];
        if (l.is_eval) {
            if (hc.pending_noise != 0 || hc.pending_md != 0) hc.noise_ready = 0;    // counters move: stale
            const int prefetch = hc.noise_ready > 0 ? 0 : noise_lookahead(ls, k);
            const bool pre_zeroed = h->fold_zero && k > 0 && !ls[k - 1].is_eval;
            if (!dry) enqueue_eval(h, l.energy, hc.pending_noise, hc.pending_md, l.cm_mode, prefetch, pre_zeroed, true);
            else h->forces_partial = !l.energy && h->skip_frozen && h->d.n_frozen > 0;
            if (prefetch > 0) hc.noise_ready = prefetch;
            hc.pending_noise = 0;
            hc.pending_md = 0;
        } else {
            IntegrateArgs a = l.args;
            a.noise_offset = hc.pending_noise;
            a.md_offset = hc.pending_md;
            const int n_o = count_ops(a, OP_O), n_md = count_ops(a, OP_MD);
            if (h->fold_zero && k + 1 < ls.size() && ls[k + 1].is_eval) {
                a.pre_eval = 1;
                a.pre_cm_mode = ls[k + 1].cm_mode;
                a.pre_adv_noise = hc.pending_noise + n_o;
                a.pre_adv_md = hc.pending_md + n_md;
            }
            const bool prefetched = n_o > 0 && n_md == 0 && hc.pending_noise == 0 && hc.noise_ready >= n_o;
            if (!dry) enqueue_integrate(h, a, prefetched);
            if (n_o > 0 || n_md > 0) hc.noise_ready = 0;        // consumed, or overwritten by the inline kernels
            hc.pending_noise += n_o;
            hc.pending_md += n_md;
            if (l.flip_after && !dry) {
                LaunchTimer t(h, -1);
                launch_pdl(h, k_cm_flip, dim3(1), dim3(64), h->stream, h->d, h->cm_parity);
            }
        }
    }
}

// run `ls` either directly or through a cached graph keyed by `key`
static int run_launches(bl_handle* h, const std::string& key, const std::vector<Launch>& ls) {
    HostCounters& hc = counters(h);
    if (!h->use_graphs || h->profiling) {
        issue(h, ls, hc);
        return BL_OK;
    }
    char suffix[64];
    snprintf(suffix, sizeof suffix, "|n%d|m%d|p%d", hc.pending_noise, hc.pending_md, hc.noise_ready);
    const std::string k = key + suffix;
    auto it = h->graphs.find(k);
    if (it == h->graphs.end()) {
        cudaGraph_t graph = nullptr;
        HostCounters tmp = hc;
        CK(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
        h->capturing = true;
        h->capture_launches = 0;
        issue(h, ls, tmp);
        h->capturing = false;
        CK(cudaStreamEndCapture(h->stream, &graph));
        cudaGraphExec_t exec = nullptr;
        CK(cudaGraphInstantiate(&exec, graph, 0));
        cudaGraphDestroy(graph);
        it = h->graphs.emplace(k, exec).first;
        // remember how many kernels one replay launches
        h->graphs.emplace(k + "#n", reinterpret_cast<cudaGraphExec_t>((uintptr_t)h->capture_launches));
    }
    CK(cudaGraphLaunch(it->second, h->stream));
    h->launches += (unsigned long long)(uintptr_t)h->graphs[k + "#n"];
    issue(h, ls, hc, true);      // advance the host mirror of the counters exactly as the captured launches did
    tl_collect(h);
    return BL_OK;
}

static void invalidate_graphs(bl_handle* h) {
    for (auto& kv : h->graphs)
        if (kv.first.find("#n") == std::string::npos && kv.second) cudaGraphExecDestroy(kv.second);
    h->graphs.clear();
}

// nan_is_error: the stepping entry points report a walker whose coordinates went non-finite (OpenMM raises "Particle
// coordinate is nan" from step()); state queries do not, so that the caller can still read the state and reject the move
static int check_flags(bl_handle* h, bool nan_is_error = true) {
    Dev& d = h->d;
    std::vector<Globals> g(d.R);
    CK(cudaMemcpyAsync(g.data(), d.g, sizeof(Globals) * d.R, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (h->profiling) collect_timings(h);
    for (int r = 0; r < d.R; ++r) {
        // a walker that blew up also overflows its list rows (its runaway atoms are parked at the origin): report the cause
        if (g[r].item_overflow && !g[r].nan_flag) {
            h->error = "neighbour work-item list overflow";
            return BL_ERR_CAPACITY;
        }
        if (g[r].nan_flag && nan_is_error) {
            char b[96];
            snprintf(b, sizeof b, "Particle coordinate is nan (walker %d)", r);
            h->error = b;
            return BL_ERR_NAN;
        }
    }
    return BL_OK;
}

// evaluate forces (and energies) at the current positions outside the step program
static void eval_now(bl_handle* h, bool energy) {
    HostCounters& hc = counters(h);
    if (hc.pending_noise != 0 || hc.pending_md != 0) hc.noise_ready = 0;
    enqueue_eval(h, energy, hc.pending_noise, hc.pending_md, 0);
    hc.pending_noise = hc.pending_md = 0;
    h->forces_valid = true;
    h->cursor = 0;
}

// ---- topology preprocessing ---------------------------------------------------------------------------------
static bool build_clusters(bl_handle* h, const bl_topology* t, std::vector<Cluster>& out) {
    const int N = t->n_atoms;
    std::vector<int> parent(N);
    for (int i = 0; i < N; ++i) parent[i] = i;
    auto find = [&](int a) { while (parent[a] != a) { parent[a] = parent[parent[a]]; a = parent[a]; } return a; };
    for (int k = 0; k < t->n_constraints; ++k) {
        int a = find(t->constraints[2 * k]), b = find(t->constraints[2 * k + 1]);
        if (a != b) parent[a] = b;
    }
    std::map<int, int> root_to_cluster;
    std::vector<Cluster> cl;
    std::vector<int> atom_cluster(N, -1);
    for (int k = 0; k < t->n_constraints; ++k) {
        const int i = t->constraints[2 * k], j = t->constraints[2 * k + 1];
        const int root = find(i);
        auto it = root_to_cluster.find(root);
        if (it == root_to_cluster.end()) {
            Cluster c;
            memset(&c, 0, sizeof c);
            cl.push_back(c);
            it = root_to_cluster.emplace(root, (int)cl.size() - 1).first;
        }
        Cluster& c = cl[it->second];
        int li = -1, lj = -1;
        for (int q = 0; q < c.natoms; ++q) { if (c.atom[q] == i) li = q; if (c.atom[q] == j) lj = q; }
        if (li < 0) { if (c.natoms >= MAX_CLUSTER_ATOMS) return false; li = c.natoms; c.atom[c.natoms++] = i; }
        if (lj < 0) { if (c.natoms >= MAX_CLUSTER_ATOMS) return false; lj = c.natoms; c.atom[c.natoms++] = j; }
        if (c.ncons >= MAX_CLUSTER_CONS) return false;
        c.ca[c.ncons] = (signed char)li;
        c.cb[c.ncons] = (signed char)lj;
        c.d2[c.ncons] = t->constraint_d[k] * t->constraint_d[k];
        c.ncons++;
        atom_cluster[i] = atom_cluster[j] = it->second;
    }
    // canonical layouts: star (every constraint touches one hub atom → hub first, constraint a = (0, a+1)) or
    // water triangle ((0,1),(0,2),(1,2)); anything else takes the generic path
    for (Cluster& c : cl) {
        c.shape = 2;
        int hub = -1;
        for (int k = 0; k < c.natoms && hub < 0; ++k) {
            bool all = true;
            for (int a = 0; a < c.ncons; ++a) if (c.ca[a] != k && c.cb[a] != k) all = false;
            if (all) hub = k;
        }
        if (hub >= 0 && c.natoms == c.ncons + 1) {
            Cluster n = c;
            n.atom[0] = c.atom[hub];
            for (int a = 0; a < c.ncons; ++a) {
                const int other = c.ca[a] == hub ? c.cb[a] : c.ca[a];
                n.atom[a + 1] = c.atom[other];
                n.ca[a] = 0; n.cb[a] = (signed char)(a + 1);
                n.d2[a] = c.d2[a];
            }
            n.shape = 0;
            c = n;
        } else if (c.natoms == 3 && c.ncons == 3) {
            Cluster n = c;
            double d01 = -1, d02 = -1, d12 = -1;
            for (int a = 0; a < 3; ++a) {
                const int lo = std::min(c.ca[a], c.cb[a]), hi = std::max(c.ca[a], c.cb[a]);
                if (lo == 0 && hi == 1) d01 = c.d2[a];
                if (lo == 0 && hi == 2) d02 = c.d2[a];
                if (lo == 1 && hi == 2) d12 = c.d2[a];
            }
            if (d01 > 0 && d02 > 0 && d12 > 0) {
                n.ca[0] = 0; n.cb[0] = 1; n.d2[0] = d01;
                n.ca[1] = 0; n.cb[1] = 2; n.d2[1] = d02;
                n.ca[2] = 1; n.cb[2] = 2; n.d2[2] = d12;
                n.shape = 1;
                c = n;
            }
        }
    }
    // homogeneous warps: order constrained clusters by (shape, ncons), then the free atoms
    for (Cluster& c : cl) if (c.shape == 0 && c.ncons > 3) c.shape = 2;      // stars with > 3 constraints: generic path
    std::stable_sort(cl.begin(), cl.end(), [](const Cluster& a, const Cluster& b) {
        return a.shape != b.shape ? a.shape > b.shape : a.ncons > b.ncons;
    });
    for (int i = 0; i < N; ++i) {
        if (atom_cluster[i] >= 0) continue;
        Cluster c;
        memset(&c, 0, sizeof c);
        c.natoms = 1;
        c.atom[0] = i;
        cl.push_back(c);
    }
    out.swap(cl);
    return true;
}

static void bspline_moduli_host(int K, std::vector<float>& out) {
    // M5 at the integer nodes 1..4: 1/24, 11/24, 11/24, 1/24
    const double data[PME_ORDER] = {0.0, 1.0 / 24, 11.0 / 24, 11.0 / 24, 1.0 / 24};
    std::vector<double> mod(K);
    for (int m = 0; m < K; ++m) {
        double sc = 0, ss = 0;
        for (int k = 0; k < PME_ORDER; ++k) {
            double arg = 2.0 * M_PI * m * k / K;
            sc += data[k] * cos(arg);
            ss += data[k] * sin(arg);
        }
        mod[m] = sc * sc + ss * ss;
    }
    for (int m = 0; m < K; ++m)
        if (mod[m] < 1e-7) mod[m] = 0.5 * (mod[(m - 1 + K) % K] + mod[(m + 1) % K]);
    out.resize(K);
    for (int m = 0; m < K; ++m) out[m] = (float)mod[m];
}

// k(z) = (erf(sqrt z) / sqrt z - 2 / sqrt(pi) exp(-z)) / z: the smooth part of the Ewald real-space force,
// F(r) = qq (1 / r^3 - alpha^3 k(alpha^2 r^2)) r_vec
static double ewald_k(double z) {
    if (z < 1e-3) return 4.0 / (3.0 * sqrt(M_PI)) * (1.0 - 3.0 * z / 5.0 + 3.0 * z * z / 14.0 - z * z * z / 18.0);
    const double s = sqrt(z);
    return (erf(s) / s - 2.0 / sqrt(M_PI) * exp(-z)) / z;
}
// Chebyshev interpolant of k on [0, zmax] of degree `deg` (<= 15), returned as monomial coefficients in t = 2 z / zmax - 1
// (sum of |c| ~ 0.75: a Horner evaluation in float is accurate to ~2e-7 absolute; interpolation error 1e-8 at zmax 11.5)
static void fit_ewald_k(double zmax, float out[16], int deg = EWK_DEG) {
    const int n = deg + 1;
    double f[17], c[17];
    for (int j = 0; j < n; ++j) f[j] = ewald_k(0.5 * zmax * (cos(M_PI * (j + 0.5) / n) + 1.0));
    for (int m = 0; m < n; ++m) {
        double acc = 0;
        for (int j = 0; j < n; ++j) acc += f[j] * cos(M_PI * m * (j + 0.5) / n);
        c[m] = acc * 2.0 / n;
    }
    c[0] *= 0.5;
    double mono[17] = {0}, tm1[17] = {0}, tm[17] = {0};     // T_{m-1}, T_m as monomial coefficient arrays
    tm1[0] = 1.0;                                         // T_0
    tm[1] = 1.0;                                          // T_1
    mono[0] += c[0];
    mono[1] += c[1];
    for (int m = 2; m < n; ++m) {
        double tn[17] = {0};
        for (int k = 0; k + 1 < n; ++k) tn[k + 1] += 2.0 * tm[k];
        for (int k = 0; k < n; ++k) tn[k] -= tm1[k];
        for (int k = 0; k < n; ++k) { mono[k] += c[m] * tn[k]; tm1[k] = tm[k]; tm[k] = tn[k]; }
    }
    for (int k = 0; k < 16; ++k) out[k] = k < n ? (float)mono[k] : 0.f;
}

static uint32_t morton3(uint32_t x, uint32_t y, uint32_t z) {
    auto part = [](uint32_t v) {
        uint64_t r = v & 0x1fffff;
        r = (r | r << 32) & 0x1f00000000ffffULL;
        r = (r | r << 16) & 0x1f0000ff0000ffULL;
        r = (r | r << 8) & 0x100f00f00f00f00fULL;
        r = (r | r << 4) & 0x10c30c30c30c30c3ULL;
        r = (r | r << 2) & 0x1249249249249249ULL;
        return r;
    };
    return (uint32_t)(part(x) | (part(y) << 1) | (part(z) << 2));
}

static int setup_box(bl_handle* h, const double box[3]) {
    Dev& d = h->d;
    double bd[6] = {box[0], box[1], box[2], 0, 0, 0};
    float bf[6];
    for (int k = 0; k < 3; ++k) {
        bd[3 + k] = box[k] > 0 ? 1.0 / box[k] : 0.0;
        bf[k] = (float)bd[k];
        bf[3 + k] = (float)bd[3 + k];
    }
    if (h->stream) CK(cudaStreamSynchronize(h->stream));     // blocking copies are not ordered with the non-blocking streams
    CK(cudaMemcpy(d.boxd, bd, sizeof bd, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d.boxf, bf, sizeof bf, cudaMemcpyHostToDevice));
    return BL_OK;
}

// cell grid for the neighbour search: cell edge >= list cutoff / 2 in x and y (so +-2 columns cover it), row-major order
// zfine: z cells finer by that factor (a cell column is one run of the sorted order whatever its z resolution; finer z
// cells trim the scanned z range of a column, and the z extent of a build group, more tightly)
static void plan_cells(const double box[3], bool periodic, double list_cutoff, int zfine, int nc[3], std::vector<int>& order) {
    nc[0] = nc[1] = nc[2] = 1;
    if (periodic && box[0] > 0)
        for (int k = 0; k < 3; ++k)
            nc[k] = std::max(1, std::min(256, (int)floor(box[k] / (0.5 * list_cutoff / (k == 2 ? zfine : 1)))));
    const int n = nc[0] * nc[1] * nc[2];
    std::vector<std::pair<uint32_t, int>> keys(n);
    for (int x = 0; x < nc[0]; ++x)
        for (int y = 0; y < nc[1]; ++y)
            for (int z = 0; z < nc[2]; ++z) {
                int lin = (x * nc[1] + y) * nc[2] + z;
                keys[lin] = {morton3(x, y, z), lin};
            }
    std::sort(keys.begin(), keys.end());
    order.assign(n, 0);
    for (int rnk = 0; rnk < n; ++rnk) order[rnk] = rnk;      // row-major cell order (z-columns contiguous)
}

// (re)plan the cell grid for a box; cell tables are reallocated when the cell count grows
static int setup_cells(bl_handle* h, const double box[3]) {
    Dev& d = h->d;
    std::vector<int> order;
    int nc[3];
    plan_cells(box, d.periodic, d.cutoffd + h->skin, h->zfine, nc, order);
    d.zreach = 2 * h->zfine;
    const int n = nc[0] * nc[1] * nc[2];
    if (n > h->cell_capacity) {
        h->cell_capacity = n + n / 4 + 8;
        d.cell_order = dalloc<int>(h, h->cell_capacity);
        d.cell_start = dalloc<int>(h, (size_t)d.R * (h->cell_capacity + 1));
        d.cell_cursor = dalloc<int>(h, (size_t)d.R * (h->cell_capacity + 1));
        d.group_capacity = d.Npad / BUILD_GROUP + h->cell_capacity + 8;
        d.group_first = dalloc<int>(h, (size_t)d.R * d.group_capacity);
        if (!d.cell_order || !d.cell_start || !d.cell_cursor || !d.group_first) { h->error = "device allocation failed"; return BL_ERR_CUDA; }
        invalidate_graphs(h);          // kernels captured the old pointers by value
    }
    if (n != d.ncells) invalidate_graphs(h);
    d.ncell[0] = nc[0]; d.ncell[1] = nc[1]; d.ncell[2] = nc[2];
    d.ncells = n;
    CK(cudaMemcpy(d.cell_order, order.data(), sizeof(int) * n, cudaMemcpyHostToDevice));
    return BL_OK;
}

// ---- C ABI ----------------------------------------------------------------------------------------------------
extern "C" {

const char* bl_version(void) { return "blues_b200 0.1.0 (sm_100a)"; }

const char* bl_last_error(const bl_handle* h) { return h ? h->error.c_str() : g_create_error.c_str(); }

int bl_num_replicas(const bl_handle* h) { return h ? h->d.R : 0; }
int bl_num_atoms(const bl_handle* h) { return h ? h->d.N : 0; }
uint64_t bl_launch_count(const bl_handle* h) { return h ? h->launches : 0; }
void* bl_stream(bl_handle* h) { return h ? (void*)h->stream : nullptr; }

int bl_destroy(bl_handle* h) {
    if (!h) return BL_OK;
    tl_report(h);
    for (auto& e : h->tl_ev) if (e) cudaEventDestroy(e);
    counter_map().erase(h);
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    invalidate_graphs(h);
    if (h->has_fft) { cufftDestroy(h->plan_r2c); cufftDestroy(h->plan_c2r); }
    for (void* p : h->allocs) cudaFree(p);
    if (h->pinned) cudaFreeHost(h->pinned);
    if (h->stream) cudaStreamDestroy(h->stream);
    if (h->stream2) cudaStreamDestroy(h->stream2);
    if (h->stream3) cudaStreamDestroy(h->stream3);
    if (h->stream4) cudaStreamDestroy(h->stream4);
    if (h->stream5) cudaStreamDestroy(h->stream5);
    if (h->ev_join5) cudaEventDestroy(h->ev_join5);
    if (h->ev_join3) cudaEventDestroy(h->ev_join3);
    if (h->ev_join4) cudaEventDestroy(h->ev_join4);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_fork2) cudaEventDestroy(h->ev_fork2);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    delete h;
    return BL_OK;
}

int bl_create(const bl_topology* t, int device, int n_replicas, uint64_t seed, bl_handle** out) {
    if (!t || !out || n_replicas < 1 || t->n_atoms < 1) { g_create_error = "invalid arguments"; return BL_ERR_INVALID; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        g_create_error = "no CUDA device available: blues_b200 has no CPU fallback";
        cudaGetLastError();
        return BL_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= ndev) { g_create_error = "invalid device index"; return BL_ERR_INVALID; }
    if (t->nb_method != 0 && t->nb_method != 2 && t->nb_method != 4) { g_create_error = "unsupported nonbonded method"; return BL_ERR_INVALID; }
    bl_handle* h = new bl_handle();
    if (getenv("BLUES_B200_PDL")) h->pdl = atoi(getenv("BLUES_B200_PDL")) != 0;
    if (getenv("BLUES_B200_GRAPH_STEPS")) h->graph_steps = std::max(1, atoi(getenv("BLUES_B200_GRAPH_STEPS")));
    if (getenv("BLUES_B200_TIMELINE")) { h->timeline = true; h->graph_steps = 1; }
    if (getenv("BLUES_B200_PAIR_SPLIT")) h->pair_split = atoi(getenv("BLUES_B200_PAIR_SPLIT"));
    if (getenv("BLUES_B200_PAIR_PER_SM")) h->pair_per_sm = std::max(0, atoi(getenv("BLUES_B200_PAIR_PER_SM")));
    cudaDeviceGetAttribute(&h->n_sm, cudaDevAttrMultiProcessorCount, device);
    if (getenv("BLUES_B200_PAIR_LANES")) { const int l = atoi(getenv("BLUES_B200_PAIR_LANES")); h->pair_lanes = l == 16 || l == 32 || l == 4 ? l : 8; }
    if (getenv("BLUES_B200_PAIR_X2")) h->pair_x2 = atoi(getenv("BLUES_B200_PAIR_X2"));
    if (getenv("BLUES_B200_DEBUG_SYNC") && atoi(getenv("BLUES_B200_DEBUG_SYNC"))) { h->debug_sync = true; h->use_graphs = false; h->pdl = false; }
    if (getenv("BLUES_B200_SPREAD_SPLIT")) h->spread_split = atoi(getenv("BLUES_B200_SPREAD_SPLIT"));
    if (getenv("BLUES_B200_SPREAD_THREADS")) h->spread_threads = atoi(getenv("BLUES_B200_SPREAD_THREADS")) == 1024 ? 1024 : 512;
    if (getenv("BLUES_B200_SKIP_FROZEN")) h->skip_frozen = atoi(getenv("BLUES_B200_SKIP_FROZEN")) != 0;
    if (getenv("BLUES_B200_ZFINE")) h->zfine = std::max(1, std::min(4, atoi(getenv("BLUES_B200_ZFINE"))));
    if (getenv("BLUES_B200_INT_BLOCK")) h->int_block = std::max(32, std::min(256, atoi(getenv("BLUES_B200_INT_BLOCK")) / 32 * 32));
    if (getenv("BLUES_B200_FOLD_ZERO")) h->fold_zero = atoi(getenv("BLUES_B200_FOLD_ZERO")) != 0;
    counter_map().erase(h);      // a recycled address must not inherit another handle's bookkeeping
    auto fail = [&](int code, const std::string& msg) { g_create_error = msg; bl_destroy(h); return code; };
    h->device = device;
    if (cudaSetDevice(device) != cudaSuccess) return fail(BL_ERR_CUDA, "cudaSetDevice failed");
    // the reciprocal-space chain (seven short dependent kernels) is the critical path of most steps and loses against
    // the wide pair kernel when they compete for SMs: its stream gets the highest priority
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    if (getenv("BLUES_B200_NO_PRIORITY")) prio_hi = prio_lo;
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithPriority(&h->stream2, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->stream3, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->stream4, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->stream5, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_join5, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_join3, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_join4, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_fork2, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming) != cudaSuccess)
        return fail(BL_ERR_CUDA, "stream creation failed");
    Dev& d = h->d;
    memset(&d, 0, sizeof d);
    const int N = t->n_atoms, R = n_replicas;
    d.N = N; d.R = R;
    d.nblocks = (N + 31) / 32;
    d.Npad = d.nblocks * 32;
    d.nb_method = t->nb_method;
    d.periodic = t->nb_method != 0;
    d.pme = t->nb_method == 4;
    if (d.periodic) {
        const double minbox = std::min(t->box[0], std::min(t->box[1], t->box[2]));
        if (!(minbox > 0) || t->cutoff * 2.0 > minbox) return fail(BL_ERR_INVALID, "cutoff must be at most half the smallest box edge");
    }
    d.cutoffd = t->cutoff; d.alphad = t->ewald_alpha;
    d.cutoff = (float)t->cutoff; d.cutoff2 = (float)(t->cutoff * t->cutoff);
    // Verlet skin: 0.14 x cutoff balances list rebuilds (every ~6 steps at 4 fs) against extra pair work (measured)
    double skin = d.periodic ? 0.14 * t->cutoff : 0.0;
    if (d.periodic && getenv("BLUES_B200_SKIN")) skin = std::max(0.01, atof(getenv("BLUES_B200_SKIN")));
    d.list_cutoff2 = d.periodic ? (float)((t->cutoff + skin) * (t->cutoff + skin)) : 3.0e38f;
    d.skin_half2 = d.periodic ? (float)(0.25 * skin * skin) : 3.0e38f;
    d.alpha = (float)t->ewald_alpha;
    if (t->nb_method == 4) {
        const double zmax = 1.02 * t->ewald_alpha * t->ewald_alpha * t->cutoff * t->cutoff;
        d.ewk_ok = zmax <= 11.5;          // beyond that (ewaldErrorTolerance < 5e-6) the erfc form is used
        fit_ewald_k(std::min(zmax, 11.5), d.ewk);
        d.ewk2_deg = zmax <= 4.8 ? 10 : (zmax <= 11.5 ? 12 : EWK_DEG);
        fit_ewald_k(std::min(zmax, 11.5), d.ewk2, d.ewk2_deg);
        d.ewk_scale = (float)(2.0 * t->ewald_alpha * t->ewald_alpha / std::min(zmax, 11.5));
        d.alpha3 = (float)(t->ewald_alpha * t->ewald_alpha * t->ewald_alpha);
    }
    if (t->nb_method == 2) {
        const double eps_rf = 78.3, rc = t->cutoff;
        d.krf = (float)((1.0 / (rc * rc * rc)) * (eps_rf - 1.0) / (2.0 * eps_rf + 1.0));
        d.crf = (float)((1.0 / rc) * 3.0 * eps_rf / (2.0 * eps_rf + 1.0));
    }
    // per-atom tables
    std::vector<double> mass(t->mass, t->mass + N), invmass(N);
    std::vector<float> charge(N);
    std::vector<float2> sigeps(N);
    double total_mass = 0, sumq = 0, sumq2 = 0;
    for (int i = 0; i < N; ++i) {
        invmass[i] = mass[i] > 0 ? 1.0 / mass[i] : 0.0;
        total_mass += mass[i];
        charge[i] = (float)t->charge[i];
        sumq += t->charge[i];
        sumq2 += t->charge[i] * t->charge[i];
        sigeps[i] = make_float2((float)(0.5 * t->sigma[i]), (float)(2.0 * sqrt(t->epsilon[i])));
    }
    d.mass = dupload(h, mass); d.invmass = dupload(h, invmass);
    d.charge = dupload(h, charge); d.sigeps = dupload(h, sigeps);
    d.charge_d = dupload(h, std::vector<double>(t->charge, t->charge + N));
    d.sigma_d = dupload(h, std::vector<double>(t->sigma, t->sigma + N));
    d.eps_d = dupload(h, std::vector<double>(t->epsilon, t->epsilon + N));
    d.sumq = sumq;
    d.self_energy_coeff = -ONE_4PI_EPS0 * t->ewald_alpha / sqrt(M_PI) * sumq2;
    d.dispersion_coeff = t->dispersion_coeff;
    // exclusion windows
    std::vector<ull> win(N, 0ull);
    std::vector<unsigned char> hasfar(N, 0);
    std::vector<long long> far;
    for (int k = 0; k < t->n_excl; ++k) {
        int i = t->excl_pairs[2 * k], j = t->excl_pairs[2 * k + 1];
        if (i < 0 || j < 0 || i >= N || j >= N || i == j) return fail(BL_ERR_INVALID, "bad exclusion pair");
        int dd = j - i + 32;
        if (dd >= 0 && dd < 64 && (i - j + 32) >= 0 && (i - j + 32) < 64) {
            win[i] |= 1ull << dd;
            win[j] |= 1ull << (i - j + 32);
        } else {
            hasfar[i] = hasfar[j] = 1;
            far.push_back(i < j ? (long long)i * N + j : (long long)j * N + i);
        }
    }
    std::sort(far.begin(), far.end());
    d.excl_win = dupload(h, win); d.has_far = dupload(h, hasfar);
    d.far_codes = dupload(h, far); d.n_far = (int)far.size();
    // bonded tables
    d.n_bonds = t->n_bonds; d.n_angles = t->n_angles; d.n_torsions = t->n_torsions;
    d.n_excl = t->n_excl; d.n_restraints = t->n_restraints; d.n_alch_exc = t->n_alch_exc;
    {
        std::vector<int2> ix(t->n_bonds); std::vector<double2> p(t->n_bonds);
        for (int k = 0; k < t->n_bonds; ++k) { ix[k] = make_int2(t->bonds[2 * k], t->bonds[2 * k + 1]); p[k] = make_double2(t->bond_k[k], t->bond_r0[k]); }
        d.bonds = dupload(h, ix); d.bond_p = dupload(h, p);
    }
    {
        std::vector<int4> ix(t->n_angles); std::vector<double2> p(t->n_angles);
        for (int k = 0; k < t->n_angles; ++k) { ix[k] = make_int4(t->angles[3 * k], t->angles[3 * k + 1], t->angles[3 * k + 2], 0); p[k] = make_double2(t->angle_k[k], t->angle_t0[k]); }
        d.angles = dupload(h, ix); d.angle_p = dupload(h, p);
    }
    {
        std::vector<int4> ix(t->n_torsions); std::vector<double4> p(t->n_torsions);
        for (int k = 0; k < t->n_torsions; ++k) {
            ix[k] = make_int4(t->torsions[4 * k], t->torsions[4 * k + 1], t->torsions[4 * k + 2], t->torsions[4 * k + 3]);
            p[k] = make_double4(t->torsion_k[k], (double)t->torsion_n[k], t->torsion_phase[k], 0.0);
        }
        d.torsions = dupload(h, ix); d.torsion_p = dupload(h, p);
    }
    {
        std::vector<int2> ix(t->n_excl); std::vector<double4> p(t->n_excl);
        for (int k = 0; k < t->n_excl; ++k) {
            int i = t->excl_pairs[2 * k], j = t->excl_pairs[2 * k + 1];
            ix[k] = make_int2(i, j);
            p[k] = make_double4(ONE_4PI_EPS0 * t->excl_qq[k], t->excl_sigma[k], t->excl_eps[k],
                                ONE_4PI_EPS0 * t->charge[i] * t->charge[j]);
        }
        d.excl = dupload(h, ix); d.excl_p = dupload(h, p);
    }
    {
        std::vector<int> ix(t->n_restraints); std::vector<double4> p(t->n_restraints);
        for (int k = 0; k < t->n_restraints; ++k) {
            ix[k] = t->restraint_atoms[k];
            p[k] = make_double4(t->restraint_x0[3 * k], t->restraint_x0[3 * k + 1], t->restraint_x0[3 * k + 2], t->restraint_k[k]);
        }
        d.restraint_atom = dupload(h, ix); d.restraint_p = dupload(h, p);
    }
    // alchemical region
    d.n_alch = t->n_alch;
    if (d.n_alch > MAX_ALCH_SMEM) return fail(BL_ERR_INVALID, "too many alchemical atoms");
    std::vector<unsigned char> is_alch(N, 0);
    {
        std::vector<int> at(t->n_alch); std::vector<double4> p(t->n_alch);
        for (int k = 0; k < t->n_alch; ++k) {
            at[k] = t->alch_atoms[k];
            is_alch[at[k]] = 1;
            p[k] = make_double4(t->alch_charge[k], t->alch_sigma[k], t->alch_eps[k], 0.0);
        }
        d.alch_atom = dupload(h, at); d.alch_p = dupload(h, p);
        d.is_alch = dupload(h, is_alch);
        std::vector<int2> ix(t->n_alch_exc); std::vector<double4> pe(t->n_alch_exc);
        for (int k = 0; k < t->n_alch_exc; ++k) {
            int i = t->alch_exc_pairs[2 * k], j = t->alch_exc_pairs[2 * k + 1];
            ix[k] = make_int2(i, j);
            pe[k] = make_double4(ONE_4PI_EPS0 * t->alch_exc_qq[k], t->alch_exc_sigma[k], t->alch_exc_eps[k],
                                 (is_alch[i] && is_alch[j]) ? 1.0 : 0.0);
        }
        d.alch_exc = dupload(h, ix); d.alch_exc_p = dupload(h, pe);
    }
    // generic Custom*Force terms
    d.n_custom = t->n_custom_terms; d.custom_np = std::max(1, t->custom_n_params);
    if (d.n_custom > 0) {
        if (!t->custom_term || !t->custom_cutoff || !t->custom_group_start || !t->custom_group_atoms || !t->custom_group_weights ||
            !t->custom_prog_start || !t->custom_code_op || !t->custom_code_arg || t->n_custom_groups < 1 || t->n_custom_progs < 1)
            return fail(BL_ERR_INVALID, "incomplete custom force tables");
        std::vector<int4> ct(d.n_custom);
        for (int k = 0; k < d.n_custom; ++k) {
            ct[k] = make_int4(t->custom_term[4 * k], t->custom_term[4 * k + 1], t->custom_term[4 * k + 2], t->custom_term[4 * k + 3]);
            if (ct[k].x < 0 || ct[k].x >= t->n_custom_groups || ct[k].y < 0 || ct[k].y >= t->n_custom_groups || ct[k].z < 0 ||
                ct[k].z >= t->n_custom_progs)
                return fail(BL_ERR_INVALID, "custom force term refers to a missing group or program");
        }
        const int n_ga = t->custom_group_start[t->n_custom_groups], n_code = t->custom_prog_start[t->n_custom_progs];
        for (int k = 0; k < n_ga; ++k)
            if (t->custom_group_atoms[k] < 0 || t->custom_group_atoms[k] >= N) return fail(BL_ERR_INVALID, "custom force group atom out of range");
        // stack discipline of every program, checked once here so that the device interpreter needs no guards
        for (int p = 0; p < t->n_custom_progs; ++p) {
            int sp = 0;
            for (int pc = t->custom_prog_start[p]; pc < t->custom_prog_start[p + 1]; ++pc) {
                const int op = t->custom_code_op[pc];
                int pops = 1, pushes = 1;
                if (op <= BL_OP_GLOBAL) pops = 0;
                else if (op == BL_OP_ADD || op == BL_OP_SUB || op == BL_OP_MUL || op == BL_OP_DIV || op == BL_OP_POW ||
                         op == BL_OP_MIN || op == BL_OP_MAX) pops = 2;
                else if (op == BL_OP_SELECT) pops = 3;
                else if (op > BL_OP_ATAN) return fail(BL_ERR_INVALID, "unknown opcode in a custom force program");
                if (op == BL_OP_PARAM && ((int)t->custom_code_arg[pc] < 0 || (int)t->custom_code_arg[pc] >= d.custom_np))
                    return fail(BL_ERR_INVALID, "custom force program reads a missing parameter");
                if (sp < pops) return fail(BL_ERR_INVALID, "custom force program underflows its stack");
                sp += pushes - pops;
                if (sp > BL_CUSTOM_STACK) return fail(BL_ERR_INVALID, "custom force expression too deep");
            }
            if (sp != 1) return fail(BL_ERR_INVALID, "custom force program must leave one value");
        }
        d.custom_term = dupload(h, ct);
        d.custom_cutoff = dupload(h, std::vector<double>(t->custom_cutoff, t->custom_cutoff + d.n_custom));
        d.custom_params = dupload(h, t->custom_params && t->custom_n_params > 0
                                         ? std::vector<double>(t->custom_params, t->custom_params + (size_t)d.n_custom * t->custom_n_params)
                                         : std::vector<double>((size_t)d.n_custom, 0.0));
        d.custom_gstart = dupload(h, std::vector<int>(t->custom_group_start, t->custom_group_start + t->n_custom_groups + 1));
        d.custom_gatoms = dupload(h, std::vector<int>(t->custom_group_atoms, t->custom_group_atoms + n_ga));
        d.custom_gweights = dupload(h, std::vector<double>(t->custom_group_weights, t->custom_group_weights + n_ga));
        d.custom_pstart = dupload(h, std::vector<int>(t->custom_prog_start, t->custom_prog_start + t->n_custom_progs + 1));
        d.custom_op = dupload(h, std::vector<int>(t->custom_code_op, t->custom_code_op + n_code));
        d.custom_arg = dupload(h, std::vector<double>(t->custom_code_arg, t->custom_code_arg + n_code));
    }
    d.alch_on = (d.n_alch > 0 || d.n_custom > 0) ? 1 : 0;
    d.alch_cap = std::min(N, 2048);
    d.alch_count = dalloc<int>(h, (size_t)R * std::max(1, d.n_alch));
    d.alch_list = dalloc<int>(h, (size_t)R * std::max(1, d.n_alch) * d.alch_cap);
    d.sc_alpha = t->softcore_alpha; d.sc_a = t->softcore_a; d.sc_b = t->softcore_b; d.sc_c = t->softcore_c;
    d.annihilate_sterics = t->annihilate_sterics; d.annihilate_elec = t->annihilate_electrostatics;
    {
        std::vector<double> one(2, 1.0);
        d.lam_s = dupload(h, one); d.lam_e = dupload(h, one); d.n_lambda = 2;
        h->lam_s_host = one; h->lam_e_host = one;
    }
    // clusters
    std::vector<Cluster> clusters;
    if (!build_clusters(h, t, clusters)) return fail(BL_ERR_INVALID, "constraint cluster too large (max 5 atoms / 4 constraints per cluster)");
    // water triangles have 3 constraints among 3 atoms; everything else is a star — both fit
    d.n_clusters = (int)clusters.size();
    for (const Cluster& c : clusters) if (c.shape == 2 || (c.shape == 0 && c.ncons > 3)) h->n_generic++;
    d.clusters = dupload(h, clusters);
    h->n_cons_total = t->n_constraints;
    // dynamic state
    const size_t RN = (size_t)R * N;
    d.boxd = dalloc<double>(h, 6); d.boxf = dalloc<float>(h, 6);
    d.pos = dalloc<double4>(h, RN); d.vel = dalloc<double4>(h, RN);
    d.posq = dalloc<float4>(h, RN); d.pos_ref = dalloc<float4>(h, RN);
    d.f_env = dalloc<long long>(h, RN * 3);
    d.f_alch = dalloc<long long>(h, d.alch_on ? RN * 3 * ALCH_SLOTS : 1);
    d.eacc = dalloc<long long>(h, (size_t)R * N_ETERMS);
    d.alch_acc = dalloc<long long>(h, (size_t)R * ALCH_SLOTS * 3);
    d.cm_acc = dalloc<long long>(h, (size_t)2 * R * 3);
    d.heat_acc = dalloc<long long>(h, R);
    d.g = dalloc<Globals>(h, R);
    d.cta_done = dalloc<int>(h, R);
    d.noise = dalloc<double>(h, (size_t)R * MAX_NOISE_SETS * N * 3);
    h->cm_parity = dalloc<int>(h, 1);
    h->d_scratch = dalloc<double>(h, std::max((size_t)R * 4, (size_t)N * 3));
    h->d_iscratch = dalloc<int>(h, (size_t)R * 2);
    // neighbour structures
    h->skin = skin;           // the cell grid serves the list cutoff (cutoff + skin)
    {
        int rc = setup_cells(h, t->box);
        if (rc != BL_OK) return fail(rc, h->error);
    }
    d.atom_cell = dalloc<int>(h, RN); d.rank = dalloc<int>(h, RN);
    d.posq_s = dalloc<float4>(h, (size_t)R * d.Npad);
    d.sigeps_s = dalloc<float2>(h, (size_t)R * d.Npad);
    d.orig_s = dalloc<int>(h, (size_t)R * d.Npad);
    {
        // row capacity per atom: 1.5 x the mean number of atoms inside the list-cutoff sphere (+ margin)
        long long M = N;
        if (d.periodic) {
            const double V = t->box[0] * t->box[1] * t->box[2], rl = t->cutoff + skin;
            M = std::min<long long>(N, (long long)(1.5 * 4.0 / 3.0 * M_PI * rl * rl * rl * N / V) + 96);
        }
        d.nl_M = (int)((M + 7) / 8 * 8);
    }
    d.nl_u16 = d.Npad < 65536 ? 1 : 0;
    d.nl_count = dalloc<int>(h, (size_t)R * d.Npad);
    if (SORT_CTAS > 8) cudaFuncSetAttribute(k_sort_atoms, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    d.mobile_s = dalloc<unsigned char>(h, (size_t)R * d.Npad);
    d.n_frozen = 0;
    for (int i = 0; i < N; ++i) d.n_frozen += t->mass[i] == 0.0 ? 1 : 0;
    d.nl_list = dalloc<unsigned char>(h, ((size_t)R * d.Npad * d.nl_M + PAIR_SLACK_ENTRIES) * (d.nl_u16 ? 2 : 4));
    {
        // k_build_list: per-lane sub-lists in shared memory are write-combining buffers flushed to the rows whenever one
        // of them passes build_cq entries (a chunk adds at most BUILD_SLACK): ~8 KB (u16) / ~10 KB (int32) per single-warp
        // CTA, so that registers, not shared memory, bound the number of resident CTAs; then the number of persistent
        // CTAs that fit on the device
        h->build_cq = (d.nl_u16 && R <= 2) ? 88 : 56;      // measured: 8 walkers 657 us per step at 56 against 690 at 88
        if (getenv("BLUES_B200_BUILD_CQ")) h->build_cq = std::max(8, std::min(d.nl_M / 4 + 48, atoi(getenv("BLUES_B200_BUILD_CQ"))));
        const size_t smem = build_smem_bytes(h->build_cq, d.nl_u16 ? 2 : 4);
        if (smem > 200 * 1024) return fail(BL_ERR_CAPACITY, "neighbour list rows do not fit the builder's shared memory");
        int per_sm = 0, n_sm = 148;
        cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device);
        if (d.nl_u16) {
            raise_dyn_smem(k_build_list<unsigned short>, device, smem);
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_build_list<unsigned short>, 32, smem);
        } else {
            raise_dyn_smem(k_build_list<int>, device, smem);
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_build_list<int>, 32, smem);
        }
        per_sm = std::max(1, per_sm);
        // With many walkers the builder runs next to the other streams' kernels (PME spread, cuFFT) most of the time and
        // would take all the shared memory of every SM: leave one CTA's worth (measured: 745 vs 770 us per 8-walker step)
        if (R > 2 && per_sm > 2) per_sm -= 1;
        if (getenv("BLUES_B200_BUILD_PER_SM")) per_sm = std::max(1, std::min(per_sm, atoi(getenv("BLUES_B200_BUILD_PER_SM"))));
        h->build_ctas = std::max(32, std::min(R * (cdiv(d.Npad, BUILD_GROUP) + 64), per_sm * n_sm));
    }
    // PME
    if (d.pme) {
        d.gx = t->pme_grid[0]; d.gy = t->pme_grid[1]; d.gz = t->pme_grid[2];
        if (d.gx < PME_ORDER || d.gy < PME_ORDER || d.gz < PME_ORDER) return fail(BL_ERR_INVALID, "PME grid too small");
        d.gsize = d.gx * d.gy * d.gz;
        // k_pme_spread at <= 2 walkers: as many y-bands per x-plane as keep the launch within one wave of one CTA per SM
        if (h->spread_split <= 0) h->spread_split = std::max(1, std::min(12, h->n_sm / std::max(1, d.gx * std::min(R, 2))));
        h->spread_split = std::max(1, std::min(h->spread_split, d.gy / 2));
        d.csize = d.gx * d.gy * (d.gz / 2 + 1);
        {
            const bool fcache = h->skip_frozen && d.n_frozen > 0;
            const size_t plane_bytes = (size_t)(d.gy / std::min(4, h->spread_split) + 1) * d.gz * sizeof(int) * (fcache ? 2 : 1);
            if (plane_bytes > 200 * 1024) return fail(BL_ERR_INVALID, "PME grid plane does not fit in shared memory");
            if (plane_bytes > 48 * 1024)
            {
                raise_dyn_smem(k_pme_spread<256>, device, plane_bytes);
                raise_dyn_smem(k_pme_spread<512>, device, plane_bytes);
                raise_dyn_smem(k_pme_spread<1024>, device, plane_bytes);
            }
        }
        d.grid_r = dalloc<float>(h, (size_t)R * d.gsize);
        if (h->skip_frozen && d.n_frozen > 0) {
            d.grid_frozen = dalloc<int>(h, (size_t)R * d.gsize);
            d.frozen_grid_state = dalloc<int>(h, R);             // zeroed: the first spread launch fills the cache
        }
        d.grid_c = dalloc<float2>(h, (size_t)R * d.csize);
        std::vector<float> mx, my, mz;
        bspline_moduli_host(d.gx, mx); bspline_moduli_host(d.gy, my); bspline_moduli_host(d.gz, mz);
        d.bmod_x = dupload(h, mx); d.bmod_y = dupload(h, my); d.bmod_z = dupload(h, mz);
        int n[3] = {d.gx, d.gy, d.gz};
        if (cufftPlanMany(&h->plan_r2c, 3, n, nullptr, 1, d.gsize, nullptr, 1, d.csize, CUFFT_R2C, R) != CUFFT_SUCCESS ||
            cufftPlanMany(&h->plan_c2r, 3, n, nullptr, 1, d.csize, nullptr, 1, d.gsize, CUFFT_C2R, R) != CUFFT_SUCCESS)
            return fail(BL_ERR_CUDA, "cufftPlanMany failed");
        h->has_fft = true;
        cufftSetStream(h->plan_r2c, h->stream2);
        cufftSetStream(h->plan_c2r, h->stream2);
    }
    for (void* p : h->allocs) if (!p) return fail(BL_ERR_CUDA, "device allocation failed");
    if (setup_box(h, t->box) != BL_OK) return fail(BL_ERR_CUDA, h->error);
    // integrator defaults
    memset(&h->ic, 0, sizeof h->ic);
    h->ic.total_mass = total_mass;
    h->ic.remove_cm = t->remove_cm && total_mass > 0;
    h->ic.seed = seed;
    h->ic.tol = 1e-8;
    h->ic.kT = 0.0083144720 * 300.0;
    // initial globals
    std::vector<Globals> g0(R);
    memset(g0.data(), 0, sizeof(Globals) * R);
    for (auto& g : g0) { g.prop = 1; g.rebuild_request = 2; g.prune_request = 1; }
    cudaMemcpy(d.g, g0.data(), sizeof(Globals) * R, cudaMemcpyHostToDevice);
    // identity ordering so that mirrors can be written before the first rebuild
    {
        std::vector<int> rk(RN);
        for (size_t i = 0; i < RN; ++i) rk[i] = (int)(i % N);
        cudaMemcpy(d.rank, rk.data(), RN * sizeof(int), cudaMemcpyHostToDevice);
    }
    if (cudaDeviceSynchronize() != cudaSuccess) return fail(BL_ERR_CUDA, "device initialisation failed");
    *out = h;
    return BL_OK;
}

int bl_set_seed(bl_handle* h, uint64_t seed) {
    if (!h) return BL_ERR_INVALID;
    h->ic.seed = seed;
    counters(h).noise_ready = 0;
    invalidate_graphs(h);
    return BL_OK;
}

int bl_use_graphs(bl_handle* h, int on) { if (!h) return BL_ERR_INVALID; h->use_graphs = on != 0; return BL_OK; }
int bl_set_profiling(bl_handle* h, int on) {
    if (!h) return BL_ERR_INVALID;
    cudaStreamSynchronize(h->stream);
    collect_timings(h);
    h->profiling = on != 0;
    if (on) for (int k = 0; k < BL_NUM_KERNEL_IDS; ++k) { h->ktime[k] = 0; h->kcount[k] = 0; }
    return BL_OK;
}
int bl_get_kernel_time(bl_handle* h, int kid, double* total_ms, int64_t* launches) {
    if (!h || kid < 0 || kid >= BL_NUM_KERNEL_IDS) return BL_ERR_INVALID;
    cudaStreamSynchronize(h->stream);
    collect_timings(h);
    if (total_ms) *total_ms = h->ktime[kid];
    if (launches) *launches = h->kcount[kid];
    return BL_OK;
}
int bl_synchronize(bl_handle* h) { if (!h) return BL_ERR_INVALID; CK(cudaStreamSynchronize(h->stream)); return BL_OK; }

int bl_set_integrator(bl_handle* h, const bl_integrator_params* p) {
    if (!h || !p) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    IntegratorConsts& ic = h->ic;
    h->integrator_kind = p->kind;
    h->temperature = p->temperature;
    ic.kT = 0.0083144720036 * p->temperature;   // kB*NA = 1.3806504e-23 * 6.02214179e23 / 1000
    ic.kT = 1.3806504e-23 * 6.02214179e23 / 1000.0 * p->temperature;
    ic.gamma = p->friction;
    ic.dt = p->timestep;
    ic.tol = p->constraint_tol > 0 ? p->constraint_tol : 1e-8;
    h->splitting.clear();
    if (p->kind == BL_INTEGRATOR_NCMC) {
        std::string s = p->splitting ? p->splitting : "H V R O R V H";
        size_t pos = 0;
        while (pos < s.size()) {
            while (pos < s.size() && s[pos] == ' ') pos++;
            size_t e = pos;
            while (e < s.size() && s[e] != ' ') e++;
            if (e > pos) h->splitting.push_back(s.substr(pos, e - pos));
            pos = e;
        }
        int nV = 0, nR = 0, nO = 0, nH = 0;
        for (auto& tok : h->splitting) {
            if (tok == "V") nV++; else if (tok == "R") nR++; else if (tok == "O") nO++; else if (tok == "H") nH++;
            else { h->error = "unsupported splitting token '" + tok + "' (supported: H V R O)"; return BL_ERR_INVALID; }
        }
        if ((int)h->splitting.size() + 2 > MAX_OPS) { h->error = "splitting string too long"; return BL_ERR_INVALID; }
        if (nO > MAX_NOISE_SETS) { h->error = "too many O steps in the splitting"; return BL_ERR_INVALID; }
        h->n_H = nH;
        ic.hV = nV ? ic.dt / nV : 0; ic.hR = nR ? ic.dt / nR : 0; ic.hO = nO ? ic.dt / nO : 0;
        ic.a = exp(-ic.gamma * ic.hO);
        ic.b = sqrt(1.0 - exp(-2.0 * ic.gamma * ic.hO));
        ic.nsteps = p->nsteps_neq;
        ic.nprop = std::max(1, p->nprop);
        ic.n_lambda_steps = p->nsteps_neq * nH;
        h->prop_lambda_min = p->prop_lambda_min;
        h->prop_lambda_max = p->prop_lambda_max;
        const int need = ic.n_lambda_steps + 1;
        if (p->n_lambda != need || !p->lambda_sterics || !p->lambda_electrostatics) {
            h->error = "lambda tables must have nsteps_neq * n_H + 1 entries";
            return BL_ERR_INVALID;
        }
        h->lam_s_host.assign(p->lambda_sterics, p->lambda_sterics + need);
        h->lam_e_host.assign(p->lambda_electrostatics, p->lambda_electrostatics + need);
        // pad so that slot indices beyond the end stay in range
        for (int k = 0; k < ALCH_SLOTS; ++k) { h->lam_s_host.push_back(h->lam_s_host[need - 1]); h->lam_e_host.push_back(h->lam_e_host[need - 1]); }
        h->d.lam_s = dupload(h, h->lam_s_host);
        h->d.lam_e = dupload(h, h->lam_e_host);
        h->d.n_lambda = (int)h->lam_s_host.size();
    } else if (p->kind == BL_INTEGRATOR_LANGEVIN) {
        ic.md_vscale = exp(-ic.dt * ic.gamma);
        ic.md_fscale = ic.gamma > 0 ? (1.0 - ic.md_vscale) / ic.gamma : ic.dt;
        ic.md_nscale = sqrt(ic.kT * (1.0 - ic.md_vscale * ic.md_vscale));
    } else {
        h->error = "unknown integrator kind";
        return BL_ERR_INVALID;
    }
    invalidate_graphs(h);
    counters(h).noise_ready = 0;
    h->forces_valid = false;
    return BL_OK;
}

// ---- state ---------------------------------------------------------------------------------------------------
static int upload_vec3(bl_handle* h, double4* dst, int replica, const double* xyz) {
    Dev& d = h->d;
    if (replica >= d.R) { h->error = "replica index out of range"; return BL_ERR_INVALID; }
    if (!h->pinned) CK(cudaMallocHost(&h->pinned, sizeof(double4) * d.N));
    CK(cudaStreamSynchronize(h->stream));
    double4* tmp = h->pinned;
    for (int i = 0; i < d.N; ++i) tmp[i] = make_double4(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], 0.0);
    const int r0 = replica < 0 ? 0 : replica, r1 = replica < 0 ? d.R : replica + 1;
    for (int r = r0; r < r1; ++r)
        CK(cudaMemcpyAsync(dst + (size_t)r * d.N, tmp, sizeof(double4) * d.N, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return BL_OK;
}
static int download_vec3(bl_handle* h, const double4* src, int replica, double* xyz) {
    Dev& d = h->d;
    if (replica < 0 || replica >= d.R) { h->error = "replica index out of range"; return BL_ERR_INVALID; }
    if (!h->pinned) CK(cudaMallocHost(&h->pinned, sizeof(double4) * d.N));
    double4* tmp = h->pinned;
    CK(cudaMemcpyAsync(tmp, src + (size_t)replica * d.N, sizeof(double4) * d.N, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < d.N; ++i) { xyz[3 * i] = tmp[i].x; xyz[3 * i + 1] = tmp[i].y; xyz[3 * i + 2] = tmp[i].z; }
    return BL_OK;
}

// replica: the walker whose coordinates were written by the host (-1: all) — its NaN / overflow latches are cleared,
// fresh coordinates make the walker usable again (a NaN in one NCMC leg must not poison the next iteration)
static void positions_changed(bl_handle* h, int replica = -2) {
    Dev& d = h->d;
    LaunchTimer t(h, -1);
    k_refresh_mirrors<<<dim3(cdiv(d.N, 128), d.R), 128, 0, h->stream>>>(d, 1, replica);
    // any coordinate may have been written, frozen atoms included: their stored charge grid is recomputed by the next
    // evaluation (stream order: the evaluation's reciprocal-space branch forks from this stream)
    if (d.grid_frozen) cudaMemsetAsync(d.frozen_grid_state, 0, sizeof(int) * d.R, h->stream);
    h->forces_valid = false;
    h->work_pending = true;      // consumed by k_external_work only (blues/integrators.py:184-191)
}

int bl_set_positions(bl_handle* h, int replica, const double* xyz) {
    if (!h || !xyz) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    int rc = upload_vec3(h, h->d.pos, replica, xyz);
    if (rc != BL_OK) return rc;
    positions_changed(h, replica);
    return BL_OK;
}
int bl_set_velocities(bl_handle* h, int replica, const double* v) {
    if (!h || !v) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    h->vel_dirty = true;
    return upload_vec3(h, h->d.vel, replica, v);
}
int bl_set_box(bl_handle* h, const double box[3]) {
    if (!h || !box) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    Dev& d = h->d;
    if (d.periodic) {
        const double minbox = std::min(box[0], std::min(box[1], box[2]));
        if (d.cutoffd * 2.0 > minbox) { h->error = "cutoff must be at most half the smallest box edge"; return BL_ERR_INVALID; }
    }
    CK(cudaStreamSynchronize(h->stream));
    int rc = setup_box(h, box);
    if (rc != BL_OK) return rc;
    if (d.periodic) { rc = setup_cells(h, box); if (rc != BL_OK) return rc; }
    positions_changed(h);
    return BL_OK;
}
int bl_get_box(bl_handle* h, double box[3]) {
    if (!h || !box) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(box, h->d.boxd, 3 * sizeof(double), cudaMemcpyDeviceToHost));
    return BL_OK;
}
int bl_get_positions(bl_handle* h, int replica, double* xyz) {
    if (!h || !xyz) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    return download_vec3(h, h->d.pos, replica, xyz);
}
int bl_get_velocities(bl_handle* h, int replica, double* v) {
    if (!h || !v) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    return download_vec3(h, h->d.vel, replica, v);
}

int bl_get_forces(bl_handle* h, int replica, double* f) {
    if (!h || !f || replica < 0 || replica >= h->d.R) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    Dev& d = h->d;
    if (!h->forces_valid || h->forces_partial) eval_now(h, true);
    { LaunchTimer t(h, -1); k_export_forces<<<cdiv(d.N, 128), 128, 0, h->stream>>>(d, replica, h->cursor, h->d_scratch); }
    CK(cudaMemcpyAsync(f, h->d_scratch, sizeof(double) * 3 * d.N, cudaMemcpyDeviceToHost, h->stream));
    return check_flags(h, false);
}

int bl_get_energy(bl_handle* h, double* epot, double* ekin) {
    if (!h) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    Dev& d = h->d;
    if (epot) {
        eval_now(h, true);     // energies are only accumulated on request
        { LaunchTimer t(h, -1); k_export_energy<<<cdiv(d.R, 64), 64, 0, h->stream>>>(d, h->cursor, h->d_scratch); }
        CK(cudaMemcpyAsync(epot, h->d_scratch, sizeof(double) * d.R, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    if (ekin) {
        CK(cudaMemsetAsync(h->d_scratch, 0, sizeof(double) * d.R, h->stream));
        { LaunchTimer t(h, -1); k_kinetic_energy<<<dim3(cdiv(d.N, 128), d.R), 128, 0, h->stream>>>(d, h->d_scratch); }
        CK(cudaMemcpyAsync(ekin, h->d_scratch, sizeof(double) * d.R, cudaMemcpyDeviceToHost, h->stream));
    }
    return check_flags(h, false);
}

int bl_get_energy_terms(bl_handle* h, int replica, double terms[BL_NUM_ENERGY_TERMS]) {
    if (!h || !terms || replica < 0 || replica >= h->d.R) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    Dev& d = h->d;
    eval_now(h, true);
    long long e[N_ETERMS], a[ALCH_SLOTS * 3];
    double box[3];
    CK(cudaMemcpyAsync(e, d.eacc + (size_t)replica * N_ETERMS, sizeof e, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(a, d.alch_acc + (size_t)replica * ALCH_SLOTS * 3, sizeof a, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(box, d.boxd, sizeof box, cudaMemcpyDeviceToHost, h->stream));
    int rc = check_flags(h, false);
    if (rc != BL_OK) return rc;
    for (int k = 0; k < N_ETERMS; ++k) terms[k] = (double)e[k] / ENERGY_SCALE;
    const double V = d.periodic ? box[0] * box[1] * box[2] : 1.0;
    terms[E_SELF] = d.pme ? d.self_energy_coeff - ONE_4PI_EPS0 * M_PI * d.sumq * d.sumq / (2.0 * d.alphad * d.alphad * V) : 0.0;
    terms[E_DISP] = d.periodic ? d.dispersion_coeff / V : 0.0;
    terms[E_ALCH_STERICS] = (double)a[h->cursor * 3 + 0] / ENERGY_SCALE;
    terms[E_ALCH_ELEC] = (double)a[h->cursor * 3 + 1] / ENERGY_SCALE;
    terms[E_ALCH_EXC] = (double)a[h->cursor * 3 + 2] / ENERGY_SCALE;
    return BL_OK;
}

int bl_copy_state(bl_handle* dst, const bl_handle* src, int flags) {
    if (!dst || !src) return BL_ERR_INVALID;
    bl_handle* h = dst;
    if (dst->d.N != src->d.N || dst->device != src->device) { h->error = "handles are not compatible"; return BL_ERR_INVALID; }
    cudaSetDevice(h->device);
    CK(cudaStreamSynchronize(src->stream));
    CK(cudaStreamSynchronize(dst->stream));            // the box / cell tables below are rewritten with blocking copies
    const int R = std::min(dst->d.R, src->d.R);
    const size_t n = sizeof(double4) * (size_t)R * dst->d.N;
    if (flags & 4) {
        double box[3];
        CK(cudaMemcpy(box, src->d.boxd, sizeof box, cudaMemcpyDeviceToHost));
        int rc = setup_box(h, box);
        if (rc != BL_OK) return rc;
        if (h->d.periodic) { rc = setup_cells(h, box); if (rc != BL_OK) return rc; }
    }
    if (flags & 1) CK(cudaMemcpyAsync(dst->d.pos, src->d.pos, n, cudaMemcpyDeviceToDevice, h->stream));
    if (flags & 2) { CK(cudaMemcpyAsync(dst->d.vel, src->d.vel, n, cudaMemcpyDeviceToDevice, h->stream)); h->vel_dirty = true; }
    if (flags & 5) positions_changed(h, (flags & 1) ? -1 : -2);
    return BL_OK;
}

int bl_copy_state_masked(bl_handle* dst, const bl_handle* src, int flags, const int32_t* mask) {
    if (!dst || !src) return BL_ERR_INVALID;
    if (!mask) return bl_copy_state(dst, src, flags);
    bl_handle* h = dst;
    if (dst->d.N != src->d.N || dst->device != src->device || dst->d.R != src->d.R) { h->error = "handles are not compatible"; return BL_ERR_INVALID; }
    cudaSetDevice(h->device);
    CK(cudaStreamSynchronize(src->stream));
    const size_t n = sizeof(double4) * (size_t)dst->d.N;
    bool any = false;
    for (int r = 0; r < dst->d.R; ++r) {
        if (!mask[r]) continue;
        any = true;
        if (flags & 1) CK(cudaMemcpyAsync(dst->d.pos + (size_t)r * dst->d.N, src->d.pos + (size_t)r * dst->d.N, n, cudaMemcpyDeviceToDevice, h->stream));
        if (flags & 2) { CK(cudaMemcpyAsync(dst->d.vel + (size_t)r * dst->d.N, src->d.vel + (size_t)r * dst->d.N, n, cudaMemcpyDeviceToDevice, h->stream)); h->vel_dirty = true; }
    }
    if (any && (flags & 1)) {
        // clear the latches of the walkers that received coordinates; all mirrors are refreshed
        positions_changed(h, -2);
        std::vector<Globals> g(dst->d.R);
        CK(cudaStreamSynchronize(h->stream));
        CK(cudaMemcpy(g.data(), dst->d.g, sizeof(Globals) * dst->d.R, cudaMemcpyDeviceToHost));
        for (int r = 0; r < dst->d.R; ++r) if (mask[r]) { g[r].nan_flag = 0; g[r].item_overflow = 0; }
        CK(cudaMemcpy(dst->d.g, g.data(), sizeof(Globals) * dst->d.R, cudaMemcpyHostToDevice));
    }
    return BL_OK;
}

int bl_velocities_to_temperature(bl_handle* h, double temperature) {
    if (!h) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    Dev& d = h->d;
    const double kT = 1.3806504e-23 * 6.02214179e23 / 1000.0 * temperature;
    { LaunchTimer t(h, -1);
      k_velocities_to_temperature<<<dim3(cdiv(d.n_clusters, 128), d.R), 128, 0, h->stream>>>(d, kT, h->ic.seed); }
    { LaunchTimer t(h, -1); k_bump_counter<<<cdiv(d.R, 64), 64, 0, h->stream>>>(d, 0); }
    h->vel_dirty = true;
    return BL_OK;
}

// ---- globals -------------------------------------------------------------------------------------------------
int bl_get_global(bl_handle* h, int replica, const char* name, double* value) {
    if (!h || !name || !value || replica < 0 || replica >= h->d.R) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    Globals g;
    long long heat = 0;
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(&g, h->d.g + replica, sizeof g, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(&heat, h->d.heat_acc + replica, sizeof heat, cudaMemcpyDeviceToHost));
    const std::string n = name;
    const int li = std::min(std::max(g.lambda_step, 0), (int)h->lam_s_host.size() - 1);
    if (n == "lambda") *value = g.lambda;
    else if (n == "lambda_step") *value = g.lambda_step;
    else if (n == "step") *value = g.step;
    else if (n == "protocol_work") *value = g.nan_flag ? NAN : g.protocol_work;     // a blown-up walker can never be accepted
    else if (n == "shadow_work") *value = g.shadow_work;
    else if (n == "heat") *value = g.heat + (double)heat / ENERGY_SCALE;
    else if (n == "first_step") *value = g.first_step;
    else if (n == "perturbed_pe") *value = g.perturbed_pe;
    else if (n == "unperturbed_pe") *value = g.unperturbed_pe;
    else if (n == "prop") *value = g.prop;
    else if (n == "nprop") *value = h->ic.nprop;
    else if (n == "prop_lambda_min") *value = h->prop_lambda_min;
    else if (n == "prop_lambda_max") *value = h->prop_lambda_max;
    else if (n == "Eold") *value = g.Eold;
    else if (n == "Enew") *value = g.Enew;
    else if (n == "debug") *value = g.debug;
    else if (n == "lambda_sterics") *value = h->lam_s_host[li];
    else if (n == "lambda_electrostatics") *value = h->lam_e_host[li];
    else if (n == "n_lambda_steps") *value = h->ic.n_lambda_steps;
    else if (n == "nsteps") *value = h->ic.nsteps;
    else if (n == "kT") *value = h->ic.kT;
    else if (n == "n_rebuilds") *value = (double)g.n_rebuilds;
    else if (n == "noise_counter") *value = (double)g.noise_counter;       // diagnostic: position in the thermostat's Philox stream
    else { h->error = "unknown global variable '" + n + "'"; return BL_ERR_INVALID; }
    return BL_OK;
}

int bl_set_global(bl_handle* h, int replica, const char* name, double value) {
    if (!h || !name || replica >= h->d.R) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    CK(cudaStreamSynchronize(h->stream));
    std::vector<Globals> g(h->d.R);
    CK(cudaMemcpy(g.data(), h->d.g, sizeof(Globals) * h->d.R, cudaMemcpyDeviceToHost));
    const std::string n = name;
    const int r0 = replica < 0 ? 0 : replica, r1 = replica < 0 ? h->d.R : replica + 1;
    for (int r = r0; r < r1; ++r) {
        Globals& x = g[r];
        if (n == "lambda") x.lambda = value;
        else if (n == "lambda_step") { x.lambda_step = (int)value; h->lambda_step = (int)value; h->forces_valid = false; }
        else if (n == "step") { x.step = (int)value; h->step = (int)value; }
        else if (n == "protocol_work") x.protocol_work = value;
        else if (n == "shadow_work") x.shadow_work = value;
        else if (n == "heat") x.heat = value;
        else if (n == "first_step") { x.first_step = (int)value; h->first_step = (int)value; }
        else if (n == "perturbed_pe") x.perturbed_pe = value;
        else if (n == "unperturbed_pe") x.unperturbed_pe = value;
        else if (n == "prop") x.prop = (int)value;
        else if (n == "Eold") x.Eold = value;
        else if (n == "Enew") x.Enew = value;
        else if (n == "debug") x.debug = (int)value;
        else if (n == "noise_counter") { x.noise_counter = (unsigned int)value; counters(h).noise_ready = 0; }   // diagnostic: replay a run from a later point of its noise stream
        else if (n == "nprop") { h->ic.nprop = std::max(1, (int)value); invalidate_graphs(h); }
        else if (n == "prop_lambda_min") h->prop_lambda_min = value;
        else if (n == "prop_lambda_max") h->prop_lambda_max = value;
        else { h->error = "global variable '" + n + "' cannot be set"; return BL_ERR_INVALID; }
    }
    CK(cudaMemcpy(h->d.g, g.data(), sizeof(Globals) * h->d.R, cudaMemcpyHostToDevice));
    return BL_OK;
}

int bl_reset_ncmc(bl_handle* h) {
    if (!h) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    CK(cudaStreamSynchronize(h->stream));
    std::vector<Globals> g(h->d.R);
    CK(cudaMemcpy(g.data(), h->d.g, sizeof(Globals) * h->d.R, cudaMemcpyDeviceToHost));
    for (auto& x : g) {
        x.step = 0; x.lambda = 0.0; x.protocol_work = 0.0; x.shadow_work = 0.0; x.first_step = 0;
        x.perturbed_pe = 0.0; x.unperturbed_pe = 0.0; x.prop = 1; x.lambda_step = 0; x.e_valid = 0;
        x.nan_flag = 0; x.item_overflow = 0;
    }
    CK(cudaMemcpy(h->d.g, g.data(), sizeof(Globals) * h->d.R, cudaMemcpyHostToDevice));
    h->step = 0; h->lambda_step = 0; h->first_step = 0;
    h->forces_valid = false;
    return BL_OK;
}

// ---- moves -----------------------------------------------------------------------------------------------------
static bool is_water_move(int kind) {
    return kind == BL_MOVE_WATER_SWAP || kind == BL_MOVE_WATER_TRANSLATE || kind == BL_MOVE_WATER_CHECK;
}
static int stage_move(bl_handle* h, const bl_move* m) {
    const bool water = is_water_move(m->kind);
    if (m->n_atoms <= 0 || !m->atoms || (!water && !m->masses)) { h->error = "move needs atoms and masses"; return BL_ERR_INVALID; }
    for (int k = 0; k < m->n_atoms; ++k)
        if (m->atoms[k] < 0 || m->atoms[k] >= h->d.N) { h->error = "move atom index out of range"; return BL_ERR_INVALID; }
    if (m->n_atoms > h->move_capacity) {
        CK(cudaStreamSynchronize(h->stream));
        dfree(h, h->d_move_atoms); dfree(h, h->d_move_masses);
        h->d_move_atoms = dalloc<int>(h, m->n_atoms);
        h->d_move_masses = dalloc<float>(h, m->n_atoms);
        h->move_capacity = m->n_atoms;
    }
    std::vector<float> mf(m->n_atoms, 0.f);
    if (m->masses) for (int k = 0; k < m->n_atoms; ++k) mf[k] = (float)m->masses[k];
    CK(cudaMemcpyAsync(h->d_move_atoms, m->atoms, sizeof(int) * m->n_atoms, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_move_masses, mf.data(), sizeof(float) * m->n_atoms, cudaMemcpyHostToDevice, h->stream));
    std::vector<float> cf;
    if (water) {
        if (m->n_atoms > 32) { h->error = "water move: at most 32 atoms per water"; return BL_ERR_INVALID; }
        if (m->n_center <= 0 || !m->center_atoms || !m->center_masses || !(m->radius > 0.0)) {
            h->error = "water move needs the protein selection (center_atoms, center_masses) and a radius";
            return BL_ERR_INVALID;
        }
        for (int k = 0; k < m->n_center; ++k)
            if (m->center_atoms[k] < 0 || m->center_atoms[k] >= h->d.N) { h->error = "water move: centre atom index out of range"; return BL_ERR_INVALID; }
        if (m->n_center > h->center_capacity) {
            CK(cudaStreamSynchronize(h->stream));
            dfree(h, h->d_center_atoms); dfree(h, h->d_center_masses);
            h->d_center_atoms = dalloc<int>(h, m->n_center);
            h->d_center_masses = dalloc<float>(h, m->n_center);
            h->center_capacity = m->n_center;
        }
        cf.resize(m->n_center);
        for (int k = 0; k < m->n_center; ++k) cf[k] = (float)m->center_masses[k];
        CK(cudaMemcpyAsync(h->d_center_atoms, m->center_atoms, sizeof(int) * m->n_center, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(h->d_center_masses, cf.data(), sizeof(float) * m->n_center, cudaMemcpyHostToDevice, h->stream));
        if (!h->d_water_state) h->d_water_state = dalloc<double>(h, (size_t)h->d.R * 4);
        if (m->kind == BL_MOVE_WATER_SWAP) {
            if (m->n_waters <= 0 || !m->water_atoms) { h->error = "water swap needs the candidate waters"; return BL_ERR_INVALID; }
            const size_t n = (size_t)m->n_waters * m->n_atoms;
            for (size_t k = 0; k < n; ++k)
                if (m->water_atoms[k] < 0 || m->water_atoms[k] >= h->d.N) { h->error = "water move: water atom index out of range"; return BL_ERR_INVALID; }
            if (n > h->water_capacity) {
                CK(cudaStreamSynchronize(h->stream));
                dfree(h, h->d_water_atoms);
                h->d_water_atoms = dalloc<int>(h, n); h->water_capacity = n;
            }
            CK(cudaMemcpyAsync(h->d_water_atoms, m->water_atoms, sizeof(int) * n, cudaMemcpyHostToDevice, h->stream));
        }
    }
    CK(cudaStreamSynchronize(h->stream));
    return BL_OK;
}
static int enqueue_move(bl_handle* h, const bl_move* m) {
    Dev& d = h->d;
    if (m->kind == BL_MOVE_ROTATE) {
        { LaunchTimer t(h, -1); k_move_rotate<<<d.R, 32, 0, h->stream>>>(d, m->n_atoms, h->d_move_atoms, h->d_move_masses, h->ic.seed); }
        { LaunchTimer t(h, -1); k_bump_counter<<<cdiv(d.R, 64), 64, 0, h->stream>>>(d, 1); }
    } else if (is_water_move(m->kind)) {
        WaterMove w;
        w.n_atoms = m->n_atoms; w.alch = h->d_move_atoms;
        w.n_waters = m->n_waters; w.waters = h->d_water_atoms;
        w.n_center = m->n_center; w.center = h->d_center_atoms; w.cmass = h->d_center_masses;
        w.radius = m->radius; w.state = h->d_water_state;
        if (m->kind == BL_MOVE_WATER_SWAP) {
            { LaunchTimer t(h, -1); k_water_swap<<<d.R, WATER_BLOCK, 0, h->stream>>>(d, w, h->ic.seed); }
            { LaunchTimer t(h, -1); k_bump_counter<<<cdiv(d.R, 64), 64, 0, h->stream>>>(d, 1); }
            h->vel_dirty = true;
        } else if (m->kind == BL_MOVE_WATER_TRANSLATE) {
            { LaunchTimer t(h, -1); k_water_translate<<<d.R, 32, 0, h->stream>>>(d, w, h->ic.seed); }
            { LaunchTimer t(h, -1); k_bump_counter<<<cdiv(d.R, 64), 64, 0, h->stream>>>(d, 1); }
        } else {
            LaunchTimer t(h, -1);
            k_water_check<<<d.R, WATER_BLOCK, 0, h->stream>>>(d, w);
            return BL_OK;                                   // coordinates untouched
        }
    } else {
        h->error = "unknown move kind";
        return BL_ERR_INVALID;
    }
    positions_changed(h);
    return BL_OK;
}

int bl_apply_move(bl_handle* h, const bl_move* m) {
    if (!h || !m) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    int rc = stage_move(h, m);
    if (rc != BL_OK) return rc;
    return enqueue_move(h, m);
}

// ---- the hot path ----------------------------------------------------------------------------------------------
static void external_work_eval(bl_handle* h, bool first_only) {
    eval_now(h, true);
    LaunchTimer t(h, -1);
    k_external_work<<<cdiv(h->d.R, 64), 64, 0, h->stream>>>(h->d, 0, first_only ? 1 : 0);
    h->first_step = 1;
    h->work_pending = false;
}

int bl_ncmc_run(bl_handle* h, int n_steps, const bl_move* move) {
    if (!h || n_steps < 0) return BL_ERR_INVALID;
    if (h->integrator_kind != BL_INTEGRATOR_NCMC) { h->error = "bl_ncmc_run needs an NCMC integrator"; return BL_ERR_INVALID; }
    cudaSetDevice(h->device);
    Dev& d = h->d;
    const bool has_move = move && move->kind != BL_MOVE_NONE;
    if (has_move) { int rc = stage_move(h, move); if (rc != BL_OK) return rc; }
    for (int i = 0; i < n_steps; ++i) {
        if (h->step >= h->ic.nsteps) break;        // `if step < nsteps` (blues/integrators.py:183)
        if (h->step == 0) {
            // reset block (blues/integrators.py:165-172): constrain, zero the work, lambda = 0
            IntegrateArgs a;
            memset(&a, 0, sizeof a);
            a.nops = 1;
            a.ops[0].kind = OP_CONSTRAIN;
            enqueue_integrate(h, a, false);
            { LaunchTimer t(h, -1); k_reset_protocol<<<cdiv(d.R, 64), 64, 0, h->stream>>>(d); }
            h->lambda_step = 0;
            h->forces_valid = false;
            h->vel_dirty = true;
        }
        if (has_move && i == move->step) {
            int rc = enqueue_move(h, move);
            if (rc != BL_OK) return rc;
        }
        if (h->vel_dirty) { enqueue_momentum(h); h->vel_dirty = false; }
        // forces_valid alone is not enough: an energy query between a host-side coordinate change and this step made the
        // forces current without booking perturbed_pe - unperturbed_pe
        if (!h->forces_valid || h->work_pending) external_work_eval(h, false);
        // one integrator step = main pass + optional extra propagation passes
        const int ls_after = h->lambda_step + h->n_H;
        const double lam_after = (double)ls_after / (double)h->ic.n_lambda_steps;
        int n_extra = 0;
        if (h->ic.nprop > 1 && lam_after > h->prop_lambda_min && lam_after <= h->prop_lambda_max) n_extra = h->ic.nprop - 1;
        const bool energy_end = (i == n_steps - 1) || (h->step + 1 >= h->ic.nsteps) || (has_move && i + 1 == move->step);
        // several plain steps (no move, no extra propagation, no energy needed at their end) go into one graph: fewer
        // graph launches and no inter-graph gap between them
        int batch = 1;
        if (h->ic.nprop == 1 && !energy_end && h->graph_steps > 1) {
            batch = h->graph_steps;
            batch = std::min(batch, n_steps - 1 - i);                          // the last step of the call carries energies
            batch = std::min(batch, h->ic.nsteps - 1 - h->step);              // so does the last step of the protocol
            if (has_move && move->step > i) batch = std::min(batch, move->step - 1 - i);   // and the step before a move
            if (batch < h->graph_steps) batch = 1;                             // only full batches: few distinct graphs
        }
        std::vector<Launch> ls;
        int cursor = h->cursor;
        for (int b = 0; b < batch; ++b) {
            compile_pass(h, ls, cursor, true, n_extra == 0, energy_end);
            for (int p = 0; p < n_extra; ++p) compile_pass(h, ls, cursor, false, p == n_extra - 1, energy_end);
        }
        char key[96];
        snprintf(key, sizeof key, "ncmc|c%d|e%d|x%d|b%d", h->cursor, energy_end ? 1 : 0, n_extra, batch);
        int rc = run_launches(h, key, ls);
        if (rc != BL_OK) return rc;
        h->cursor = cursor;
        h->step += batch;
        h->lambda_step = h->lambda_step + batch * h->n_H;
        h->forces_valid = true;
        i += batch - 1;
    }
    return check_flags(h);
}

int bl_md_run(bl_handle* h, int n_steps) {
    if (!h || n_steps < 0) return BL_ERR_INVALID;
    if (h->integrator_kind != BL_INTEGRATOR_LANGEVIN) { h->error = "bl_md_run needs a Langevin integrator"; return BL_ERR_INVALID; }
    cudaSetDevice(h->device);
    for (int i = 0; i < n_steps; ++i) {
        if (h->vel_dirty) { enqueue_momentum(h); h->vel_dirty = false; }
        if (!h->forces_valid) eval_now(h, false);
        std::vector<Launch> ls(2);
        memset(&ls[0], 0, sizeof(Launch));
        memset(&ls[1], 0, sizeof(Launch));
        ls[0].is_eval = false;
        ls[0].args.nops = 2;
        ls[0].args.ops[0].kind = OP_CM;
        ls[0].args.ops[1].kind = OP_MD;
        ls[0].args.ops[1].slot = h->cursor;
        ls[0].args.accum_cm = h->ic.remove_cm ? 2 : 0;
        ls[1].is_eval = true;
        ls[1].energy = false;
        ls[1].cm_mode = h->ic.remove_cm ? 2 : 0;
        char key[64];
        snprintf(key, sizeof key, "md|c%d", h->cursor);
        int rc = run_launches(h, key, ls);
        if (rc != BL_OK) return rc;
        h->cursor = 0;
        h->forces_valid = true;
    }
    return check_flags(h);
}

int bl_accept_reject(bl_handle* h, const double* correction, int32_t* accepted, double* logp, double* log_u) {
    if (!h || !accepted) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    Dev& d = h->d;
    double* dcorr = nullptr;
    if (correction) {
        dcorr = h->d_scratch + 2 * d.R;
        CK(cudaMemcpyAsync(dcorr, correction, sizeof(double) * d.R, cudaMemcpyHostToDevice, h->stream));
    }
    { LaunchTimer t(h, -1);
      k_accept<<<cdiv(d.R, 64), 64, 0, h->stream>>>(d, h->ic.kT, dcorr, h->d_iscratch, h->d_scratch, h->d_scratch + d.R, h->ic.seed); }
    { LaunchTimer t(h, -1); k_bump_counter<<<cdiv(d.R, 64), 64, 0, h->stream>>>(d, 2); }
    std::vector<double> tmp(2 * d.R);
    CK(cudaMemcpyAsync(accepted, h->d_iscratch, sizeof(int) * d.R, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(tmp.data(), h->d_scratch, sizeof(double) * 2 * d.R, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (logp) memcpy(logp, tmp.data(), sizeof(double) * d.R);
    if (log_u) memcpy(log_u, tmp.data() + d.R, sizeof(double) * d.R);
    return BL_OK;
}

int bl_minimize(bl_handle* h, int max_iterations, double tolerance) {
    if (!h) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    Dev& d = h->d;
    if (max_iterations <= 0) max_iterations = 1000;
    if (tolerance <= 0) tolerance = 10.0;
    if (!h->d_saved) h->d_saved = dalloc<double4>(h, (size_t)d.R * d.N);
    // constrain first, then adaptive steepest descent: accept a trial if the energy went down (step *= 1.2),
    // otherwise restore and halve the step.  One host round-trip per iteration (not a hot path).
    {
        IntegrateArgs a; memset(&a, 0, sizeof a); a.nops = 1; a.ops[0].kind = OP_CONSTRAIN;
        enqueue_integrate(h, a, false);
        positions_changed(h);
    }
    std::vector<double> e0(d.R), e1(d.R), step(d.R, 1e-6);
    std::vector<int> reject(d.R);
    int rc = bl_get_energy(h, e0.data(), nullptr);
    if (rc != BL_OK) return rc;
    double gstep = 1e-5;   // nm per (kJ/mol/nm): displacement = gstep * F, capped at 0.01 nm per atom
    for (int it = 0; it < max_iterations; ++it) {
        { LaunchTimer t(h, -1);
          k_minimize_step<<<dim3(cdiv(d.n_clusters, 128), d.R), 128, 0, h->stream>>>(d, gstep, 0.01, h->ic.tol, h->d_saved); }
        positions_changed(h);
        rc = bl_get_energy(h, e1.data(), nullptr);
        if (rc != BL_OK && rc != BL_ERR_NAN) return rc;
        bool any_reject = false, all_up = true;
        for (int r = 0; r < d.R; ++r) {
            reject[r] = !(e1[r] < e0[r]);
            if (reject[r]) any_reject = true; else { all_up = false; e0[r] = e1[r]; }
        }
        if (any_reject) {
            CK(cudaMemcpyAsync(h->d_iscratch, reject.data(), sizeof(int) * d.R, cudaMemcpyHostToDevice, h->stream));
            { LaunchTimer t(h, -1);
              k_restore_positions<<<dim3(cdiv(d.N, 128), d.R), 128, 0, h->stream>>>(d, h->d_saved, h->d_iscratch); }
            positions_changed(h);
            CK(cudaStreamSynchronize(h->stream));
            // forces must be re-evaluated at the restored coordinates
            eval_now(h, true);
        }
        gstep = all_up ? gstep * 0.5 : gstep * 1.2;
        if (gstep < 1e-12) break;
        if (!any_reject && (it % 10) == 9) {
            CK(cudaMemsetAsync(h->d_scratch, 0, sizeof(double) * d.R, h->stream));
            { LaunchTimer t(h, -1); k_max_force<<<dim3(cdiv(d.N, 128), d.R), 128, 0, h->stream>>>(d, h->d_scratch); }
            std::vector<double> f2(d.R);
            CK(cudaMemcpyAsync(f2.data(), h->d_scratch, sizeof(double) * d.R, cudaMemcpyDeviceToHost, h->stream));
            CK(cudaStreamSynchronize(h->stream));
            double worst = 0;
            for (double v : f2) worst = std::max(worst, sqrt(v));
            if (worst < tolerance) break;
        }
    }
    // clear a NaN flag possibly raised by rejected trial steps
    std::vector<Globals> g(d.R);
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaMemcpy(g.data(), d.g, sizeof(Globals) * d.R, cudaMemcpyDeviceToHost));
    for (auto& x : g) x.nan_flag = 0;
    CK(cudaMemcpy(d.g, g.data(), sizeof(Globals) * d.R, cudaMemcpyHostToDevice));
    return BL_OK;
}

// ---- introspection ----------------------------------------------------------------------------------------------
}  // extern "C"

// FP32 FMA throughput microbenchmark: the roofline denominator of the pair kernel (MEASURED_PEAKS.json carries HBM and
// bf16 tensor figures only).  16 independent FMA chains per thread, 8 warps x 8 CTAs per SM, no memory traffic.
__global__ void __launch_bounds__(256) k_fma_peak(float* out, int iters, float a, float b) {
    float x[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) x[k] = (float)(threadIdx.x + k) * 1e-3f;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int k = 0; k < 16; ++k) x[k] = fmaf(x[k], a, b);
    }
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) s += x[k];
    if (s == 123.456f) out[blockIdx.x * blockDim.x + threadIdx.x] = s;      // never true: keeps the chains alive
}

extern "C" {

int bl_measure_fp32_peak(int device, double* tflops) {
    if (!tflops) return BL_ERR_INVALID;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) { cudaGetLastError(); return BL_ERR_NO_DEVICE; }
    cudaSetDevice(device);
    cudaGetLastError();                                   // a stale error of an unrelated earlier call is not ours
    int n_sm = 148;
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, device);
    float* out = nullptr;
    const int blocks = n_sm * 8, threads = 256, iters = 4096;
    if (cudaMalloc(&out, sizeof(float) * blocks * threads) != cudaSuccess) return BL_ERR_CUDA;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    double best = 0.0;
    for (int rep = 0; rep < 12; ++rep) {                 // first repeats warm the clocks up; best of the rest
        cudaEventRecord(e0, 0);
        k_fma_peak<<<blocks, threads>>>(out, iters, 0.999f, 1e-3f);
        cudaEventRecord(e1, 0);
        cudaEventSynchronize(e1);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        const double flops = 2.0 * 16.0 * (double)iters * (double)blocks * threads;
        if (rep >= 2 && ms > 0.f) best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    const cudaError_t err = cudaDeviceSynchronize();
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(out);
    if (err != cudaSuccess || best <= 0.0) { cudaGetLastError(); return BL_ERR_CUDA; }
    *tflops = best;
    return BL_OK;
}

int bl_neighbor_pairs(bl_handle* h, int replica, int64_t* codes, size_t capacity, size_t* n_pairs) {
    if (!h || !n_pairs || replica < 0 || replica >= h->d.R) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    Dev& d = h->d;
    // coordinates changed by the host since the last evaluation: build a fresh list.  Otherwise report the list the
    // last evaluation used (tests use this to check the skin / prune / rebuild logic after dynamics).
    if (!h->forces_valid) {
        { LaunchTimer t(h, -1); k_refresh_mirrors<<<dim3(cdiv(d.N, 128), d.R), 128, 0, h->stream>>>(d, 1, -2); }
        eval_now(h, false);
    }
    long long* dcodes = nullptr;
    unsigned long long* dn = nullptr;
    CK(cudaMalloc(&dcodes, sizeof(long long) * std::max<size_t>(capacity, 1)));
    CK(cudaMalloc(&dn, sizeof(unsigned long long)));
    CK(cudaMemsetAsync(dn, 0, sizeof(unsigned long long), h->stream));
    { LaunchTimer t(h, -1);
      if (d.nl_u16) k_neighbor_pairs<unsigned short><<<148 * 4, 128, 0, h->stream>>>(d, replica, dcodes, capacity, dn);
      else k_neighbor_pairs<int><<<148 * 4, 128, 0, h->stream>>>(d, replica, dcodes, capacity, dn); }
    unsigned long long n = 0;
    CK(cudaMemcpyAsync(&n, dn, sizeof n, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    *n_pairs = (size_t)n;
    if (codes && n <= capacity) {
        CK(cudaMemcpy(codes, dcodes, sizeof(long long) * n, cudaMemcpyDeviceToHost));
        std::sort(codes, codes + n);
    }
    cudaFree(dcodes);
    cudaFree(dn);
    return check_flags(h, false);
}

int bl_neighbor_stats(bl_handle* h, int replica, int64_t* n_tiles, int64_t* n_rebuilds) {
    if (!h || replica < 0 || replica >= h->d.R) return BL_ERR_INVALID;
    cudaSetDevice(h->device);
    CK(cudaStreamSynchronize(h->stream));
    Globals g;
    CK(cudaMemcpy(&g, h->d.g + replica, sizeof g, cudaMemcpyDeviceToHost));
    if (n_tiles) *n_tiles = (int64_t)h->d.nl_M;
    if (n_rebuilds) *n_rebuilds = g.n_rebuilds;
    return BL_OK;
}

}  // extern "C"
