// rx_internal.cuh -- shared declarations of librx_b200.so (not part of the public ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>
#include <utility>
#include "../../include/rx_b200.h"

#define RX_KB 8.31446261815324e-3 /* kJ/mol/K, openmmtools/constants.py:7 with OpenMM >= 7.6 CODATA-2018 values */
#define RX_MAX_PROGRAM 32

// ---- per-state table as the kernels see it ---------------------------------------------------------
struct StateDev {
    double beta;     // 1/(kB T)
    double kT;       // kB T
    double lambda;   // lambda_sterics
    double la;       // lambda^a            (alchemy.py:1385)
    double ob;       // alpha (1-lambda)^b  (alchemy.py:1388)
    double offset;   // kJ/mol
    double ho_K;
    double ho_x0[3];
};

// ---- MT19937 stream resident on the device (numba's / numpy's generator restated) ---------------------
struct MTStream {
    uint32_t *d_window = nullptr;  // last 624 raw words x_n .. x_{n+623}
    uint32_t *d_words = nullptr;   // tempered outputs not yet consumed: d_words[0..avail)
    uint32_t *d_words_alt = nullptr;
    size_t cap = 0;
    size_t avail = 0;
    uint64_t consumed = 0;  // words consumed since seeding
    bool seeded = false;
};

struct SlotRec {        // one 2-word "slot" of the stream, state independent (pow2 K fast path)
    uint32_t ij;        // i | j << 16 (masked replica indices)
    uint32_t backmask;  // bit 31-b: slot s-1-b shares a replica index with slot s (b = 0..30)
    double logU;        // log of the uniform the two words of THIS slot would produce
};

struct MixCtl {          // device-resident control block of the resumable mixing kernels
    long long head;      // in: first unconsumed word (serial) / slot (pow2);  out: same after the call
    long long remaining; // attempts still to do
    int status;          // 0 done, 1 need more words
    int rounds;          // statistics: speculation rounds executed
    long long slow_exp;  // statistics: exact exp() fallbacks
    long long log_count; // entries written to the commit log by this launch
    long long aux;       // k_mix_walk2c: candidate index reached (extent of its sparse commit log)
};

// One Langevin move: timestep, friction, steps per launch, splitting program and velocity reassignment.
struct rx_state_move {
    double dt = 0, gamma = 0;
    int n_steps = 0, reassign = 0;
    char program[RX_MAX_PROGRAM] = {0};
};

struct rx_engine {
    rx_config cfg;
    int k0 = 0, kloc = 0;  // owned replicas [k0, k0+kloc)
    int n_sms = 0;         // streaming multiprocessors of cfg.device
    cudaStream_t stream = nullptr, stream_rng = nullptr;
    cudaEvent_t ev[8] = {};
    cudaEvent_t ev_user[2] = {};
    long long mix_stats[6] = {0, 0, 0, 0, 0, 0};   // rounds, exact-exp, passes, words, walker us, prepare-wait us
    cudaEvent_t ev_walk[2] = {};
    // particles
    float4 *d_atom = nullptr;     // (sigma, sqrt_eps, inv_mass, alch ? 1 : 0)
    double4 *d_atom_d = nullptr;  // (sigma, eps, mass, alch)
    int n_alch = 0;
    int *d_alch_list = nullptr;   // indices of the alchemical atoms
    bool have_particles = false, have_states = false, have_integrator = false;
    StateDev *d_states = nullptr;
    std::vector<StateDev> h_states;
    // replica state
    float4 *d_pos = nullptr, *d_vel = nullptr;  // [kloc][N]
    float4 *d_pos_snap = nullptr, *d_vel_snap = nullptr;   // start-of-iteration copy for the NaN restart policy
    int *d_retry = nullptr;                     // [K] replicas to propagate again
    bool have_snapshot = false;
    double *d_io = nullptr;                     // staging for set/get: [kloc][N][3]
    double *h_io = nullptr;                     // pinned host staging of the same size
    std::vector<std::pair<const char *, size_t>> pinned;   // caller buffers registered with rx_pin_host_memory
    int *d_perm = nullptr;                      // [K] replica -> state
    double *d_u = nullptr;                      // [K][M]
    unsigned long long *d_nacc = nullptr, *d_nprop = nullptr;  // [M][M]
    double *d_pot = nullptr, *d_kin = nullptr;  // [K]
    int *d_nan = nullptr;                       // [K]
    int *d_err = nullptr;                       // device error flag (capacity overflow, ...)
    // energy kernel scratch: lambda-controlled pairs per owned replica
    double4 *d_pairs = nullptr;  // (r, sigma, eps, S) ... see rx_dynamics.cu
    int pair_cap = 0;
    rx_state_move move;                      // the move of every state (rx_set_integrator; its reassign is unused)
    void *mol_dev = nullptr;                 // MolDev (host copy of the device table of a RX_SYSTEM_MOLECULE engine)
    std::vector<void *> mol_allocs;
    std::vector<rx_state_move> state_moves;   // per-state moves (empty: one move for all states)
    bool state_moves_dirty = false;
    void *d_moves = nullptr;
    // mixing
    MTStream streams[2];
    SlotRec *d_slots = nullptr;
    size_t slots_cap = 0;
    MixCtl *d_ctl = nullptr;
    uint32_t *d_log = nullptr;   // commit log of the walker: packed (si, sj, accepted)
    size_t log_cap = 0;
    uint32_t *d_slotlog = nullptr;   // sparse commit log of k_mix_walk2: one word per slot
    uint32_t *d_cpos = nullptr;      // k_mix_walk2c: word position of every candidate of the pass
    uint32_t *d_ctile = nullptr;     // ... candidates per tile / their exclusive scan, then [last] = number of candidates
    size_t ctile_cap = 0;
    unsigned char *d_filt = nullptr;   // 24-bit row image of u for the K=256 walker
    double *d_filt_scale = nullptr;    // [K] scales + [K] row abs-max
    int prepared_plan = 0;        // walker plan (WalkPlan of rx_mix.cu) the prepared records were built for
    bool prepared = false;        // words + slot records for the next swap-all call were produced on stream_rng
    size_t last_consumed = 0;     // words the previous swap-all call consumed (sizes the generate-ahead)
    size_t slots_for_avail = 0;   // S.avail the slot records were built for
    cudaEvent_t ev_prepared = nullptr, ev_consumed = nullptr;
    void *sams = nullptr;         // SamsState (rx_sams.cuh): device-resident logZ / weights / histogram of a SAMSSampler
    // timing
    double phase_ms[4] = {0, 0, 0, 0};
    long long phase_launches[4] = {0, 0, 0, 0};
    // nccl
    void *nccl_lib = nullptr;
    void *nccl_comm = nullptr;
    std::string err;
};

extern thread_local std::string g_rx_create_error;

#define RX_CHECK_CUDA(h, call)                                                                     \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            (h)->err = std::string(#call) + ": " + cudaGetErrorString(_e);                         \
            return RX_ERR_CUDA;                                                                    \
        }                                                                                          \
    } while (0)

#define RX_FAIL(h, code, msg)     \
    do {                          \
        (h)->err = (msg);         \
        return (code);            \
    } while (0)

// phase timing helper: records events around a phase on h->stream
struct PhaseTimer {
    rx_engine *h;
    int phase;
    PhaseTimer(rx_engine *h_, int p) : h(h_), phase(p) { cudaEventRecord(h->ev[2 * p], h->stream); }
    void stop(int launches) {
        cudaEventRecord(h->ev[2 * phase + 1], h->stream);
        h->phase_launches[phase] += launches;
    }
    void accumulate() {  // call after a stream sync
        float ms = 0;
        if (cudaEventElapsedTime(&ms, h->ev[2 * phase], h->ev[2 * phase + 1]) == cudaSuccess) h->phase_ms[phase] += ms;
    }
};

// ---- implemented in rx_mix.cu ----
int rxi_mix_seed(rx_engine *h, int stream, uint32_t seed);
int rxi_mix_skip(rx_engine *h, int stream, unsigned long long n);
int rxi_selftest_exp(rx_engine *h, const double *x, double *y, int n);
int rxi_mix_swap_all(rx_engine *h, long long nswap, int *launches);
int rxi_mix_swap_neighbors(rx_engine *h, int *launches);
void rxi_mix_free(rx_engine *h);
int rxi_sams_set(rx_engine *h, const rx_sams_config *c, const double *log_target, const double *logZ, const int64_t *histogram);
int rxi_sams_step(rx_engine *h, long long iteration, int update, int *launches);
int rxi_sams_get(rx_engine *h, double *logZ, double *log_weights, int64_t *histogram, int32_t *stage, int64_t *t0, double *gamma,
                 int64_t *states, int64_t *previous_states);
int rxi_sams_set_histogram(rx_engine *h, const int64_t *histogram);
void rxi_sams_free(rx_engine *h);

// ---- implemented in rx_dynamics.cu ----
int rxi_propagate(rx_engine *h, uint64_t seed, uint64_t iteration, int reassign, int *launches, const int *d_only = nullptr);
int rxi_upload_state_moves(rx_engine *h);
int rxi_set_molecule(rx_engine *h, const rx_molecule *mol);
void rxi_free_molecule(rx_engine *h);
int rxi_snapshot_state(rx_engine *h);   // positions + velocities at the start of a propagation
int rxi_restore_failed(rx_engine *h);   // replicas with a NaN flag go back to the snapshot; d_retry = the flags
int rxi_compute_energy_rows(rx_engine *h, int *launches);  // fills d_u rows [k0, k0+kloc)
int rxi_compute_energy_rows_at(rx_engine *h, const StateDev *d_states, int n_states, double *d_out, int *launches);
int rxi_randomize_velocities(rx_engine *h, uint64_t seed, uint64_t stream_id);
int rxi_minimize(rx_engine *h, double tolerance, int max_iterations, double *d_rms, int *d_iters);  // [K] each
int rxi_convert_in(rx_engine *h, float4 *dst, int first_local, int count, const double *host_xyz, bool is_vel);
int rxi_convert_out(rx_engine *h, const float4 *src, int first_local, int count, double *host_xyz, bool wrap);

// ---- implemented in rx_api.cu ----
bool rxi_is_pinned(const rx_engine *h, const void *p, size_t bytes);
int rxi_allgather_energies(rx_engine *h);
int rxi_allgather_rows(rx_engine *h, double *d_matrix, int n_cols);
