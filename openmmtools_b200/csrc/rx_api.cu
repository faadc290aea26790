// rx_api.cu -- the C ABI of librx_b200.so (include/rx_b200.h): lifecycle, tables, replica I/O, phase calls,
// the fused iteration loop, NCCL (dlopen) energy-row all-gather.
#include "rx_internal.cuh"
#include <dlfcn.h>
#include <math.h>
#include <string.h>

thread_local std::string g_rx_create_error;

extern "C" int rx_abi_version(void) { return RX_ABI_VERSION; }

extern "C" const char *rx_last_error(const rx_engine *h) { return h ? h->err.c_str() : g_rx_create_error.c_str(); }

#define CREATE_FAIL(code, msg)       \
    do {                             \
        g_rx_create_error = (msg);   \
        if (h) rx_destroy(h);        \
        return (code);               \
    } while (0)
#define CREATE_CUDA(call)                                                                 \
    do {                                                                                  \
        cudaError_t _e = (call);                                                          \
        if (_e != cudaSuccess) CREATE_FAIL(RX_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e)); \
    } while (0)

extern "C" int rx_create(const rx_config *cfg, rx_engine **out) {
    rx_engine *h = nullptr;
    if (!cfg || !out) CREATE_FAIL(RX_ERR_INVALID, "rx_create: null argument");
    if (cfg->abi_version != RX_ABI_VERSION) CREATE_FAIL(RX_ERR_INVALID, "rx_create: ABI version mismatch");
    if (cfg->n_replicas < 1 || cfg->n_states < 1) CREATE_FAIL(RX_ERR_INVALID, "rx_create: n_replicas and n_states must be >= 1");
    if (cfg->system_kind < RX_SYSTEM_NONE || cfg->system_kind > RX_SYSTEM_MOLECULE) CREATE_FAIL(RX_ERR_INVALID, "rx_create: unknown system_kind");
    if (cfg->system_kind != RX_SYSTEM_NONE && cfg->n_atoms < 1) CREATE_FAIL(RX_ERR_INVALID, "rx_create: n_atoms must be >= 1");
    if (cfg->system_kind == RX_SYSTEM_MOLECULE && cfg->n_atoms > 32) CREATE_FAIL(RX_ERR_UNSUPPORTED, "rx_create: a molecule has at most 32 atoms");
    if (cfg->world_size < 1 || cfg->rank < 0 || cfg->rank >= cfg->world_size) CREATE_FAIL(RX_ERR_INVALID, "rx_create: bad rank/world_size");
    if (cfg->system_kind == RX_SYSTEM_LJ_ALCH) {
        for (int d = 0; d < 3; d++)
            if (!(cfg->box[d] > 0) || cfg->r_cutoff > 0.5 * cfg->box[d])
                CREATE_FAIL(RX_ERR_INVALID, "rx_create: cutoff must not exceed half the box edge (minimum image)");
        if (!(cfg->r_cutoff > 0)) CREATE_FAIL(RX_ERR_INVALID, "rx_create: r_cutoff must be > 0");
        if (cfg->use_switch && !(cfg->r_switch >= 0 && cfg->r_switch < cfg->r_cutoff))
            CREATE_FAIL(RX_ERR_INVALID, "rx_create: need 0 <= r_switch < r_cutoff");
        if (!(cfg->softcore_c > 0)) CREATE_FAIL(RX_ERR_INVALID, "rx_create: softcore_c must be > 0");
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) CREATE_FAIL(RX_ERR_CUDA, std::string("rx_create: no CUDA device available (") + cudaGetErrorString(e) + "); this engine has no CPU fallback");
    if (cfg->device < 0 || cfg->device >= ndev) CREATE_FAIL(RX_ERR_INVALID, "rx_create: device ordinal out of range");
    CREATE_CUDA(cudaSetDevice(cfg->device));
    h = new rx_engine();
    h->cfg = *cfg;
    CREATE_CUDA(cudaDeviceGetAttribute(&h->n_sms, cudaDevAttrMultiProcessorCount, cfg->device));
    const int K = cfg->n_replicas, M = cfg->n_states, N = cfg->n_atoms, W = cfg->world_size, R = cfg->rank;
    h->k0 = (int)(((long long)R * K) / W);
    h->kloc = (int)(((long long)(R + 1) * K) / W) - h->k0;
    {
        // The side stream prepares the NEXT mixing call (random words, slot records) while the replicas propagate on the main
        // stream: it gets the lowest priority, so that its thread blocks only fill what k_propagate leaves free.
        int prio_lo = 0, prio_hi = 0;
        CREATE_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        CREATE_CUDA(cudaStreamCreateWithPriority(&h->stream, cudaStreamNonBlocking, prio_hi));
        CREATE_CUDA(cudaStreamCreateWithPriority(&h->stream_rng, cudaStreamNonBlocking, prio_lo));
    }
    for (int i = 0; i < 8; i++) CREATE_CUDA(cudaEventCreate(&h->ev[i]));
    for (int i = 0; i < 2; i++) CREATE_CUDA(cudaEventCreate(&h->ev_user[i]));
    for (int i = 0; i < 2; i++) CREATE_CUDA(cudaEventCreate(&h->ev_walk[i]));
    CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_prepared, cudaEventDisableTiming));
    CREATE_CUDA(cudaEventCreateWithFlags(&h->ev_consumed, cudaEventDisableTiming));
    CREATE_CUDA(cudaMalloc(&h->d_perm, sizeof(int) * K));
    CREATE_CUDA(cudaMalloc(&h->d_u, sizeof(double) * (size_t)K * M));
    CREATE_CUDA(cudaMemset(h->d_u, 0, sizeof(double) * (size_t)K * M));
    CREATE_CUDA(cudaMalloc(&h->d_nacc, sizeof(unsigned long long) * (size_t)M * M));
    CREATE_CUDA(cudaMalloc(&h->d_nprop, sizeof(unsigned long long) * (size_t)M * M));
    CREATE_CUDA(cudaMemset(h->d_nacc, 0, sizeof(unsigned long long) * (size_t)M * M));
    CREATE_CUDA(cudaMemset(h->d_nprop, 0, sizeof(unsigned long long) * (size_t)M * M));
    CREATE_CUDA(cudaMalloc(&h->d_pot, sizeof(double) * K));
    CREATE_CUDA(cudaMalloc(&h->d_kin, sizeof(double) * K));
    CREATE_CUDA(cudaMemset(h->d_pot, 0, sizeof(double) * K));
    CREATE_CUDA(cudaMemset(h->d_kin, 0, sizeof(double) * K));
    CREATE_CUDA(cudaMalloc(&h->d_nan, sizeof(int) * K));
    CREATE_CUDA(cudaMemset(h->d_nan, 0, sizeof(int) * K));
    CREATE_CUDA(cudaMalloc(&h->d_err, sizeof(int)));
    CREATE_CUDA(cudaMemset(h->d_err, 0, sizeof(int)));
    CREATE_CUDA(cudaMalloc(&h->d_ctl, sizeof(MixCtl)));
    CREATE_CUDA(cudaMalloc(&h->d_states, sizeof(StateDev) * M));
    {
        std::vector<int> perm(K);
        for (int k = 0; k < K; k++) perm[k] = k % M;
        CREATE_CUDA(cudaMemcpy(h->d_perm, perm.data(), sizeof(int) * K, cudaMemcpyHostToDevice));
    }
    if (cfg->system_kind != RX_SYSTEM_NONE) {
        const size_t n = (size_t)(h->kloc > 0 ? h->kloc : 1) * N;
        // (a molecule keeps its state as double[3] per atom, the other systems as float4)
        const size_t per_atom = cfg->system_kind == RX_SYSTEM_MOLECULE ? 3 * sizeof(double) : sizeof(float4);
        CREATE_CUDA(cudaMalloc(&h->d_pos, per_atom * n));
        CREATE_CUDA(cudaMalloc(&h->d_vel, per_atom * n));
        CREATE_CUDA(cudaMemset(h->d_pos, 0, per_atom * n));
        CREATE_CUDA(cudaMemset(h->d_vel, 0, per_atom * n));
        CREATE_CUDA(cudaMalloc(&h->d_io, sizeof(double) * 3 * n));
        CREATE_CUDA(cudaHostAlloc(&h->h_io, sizeof(double) * 3 * n, cudaHostAllocDefault));
        CREATE_CUDA(cudaMalloc(&h->d_atom, sizeof(float4) * N));
        CREATE_CUDA(cudaMalloc(&h->d_atom_d, sizeof(double4) * N));
        CREATE_CUDA(cudaMalloc(&h->d_alch_list, sizeof(int) * N));
    }
    *out = h;
    return RX_OK;
}

extern "C" void rx_destroy(rx_engine *h) {
    if (!h) return;
    cudaSetDevice(h->cfg.device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->stream_rng) cudaStreamSynchronize(h->stream_rng);
    if (h->ev_prepared) cudaEventDestroy(h->ev_prepared);
    if (h->ev_consumed) cudaEventDestroy(h->ev_consumed);
    if (h->nccl_comm && h->nccl_lib) {
        typedef int (*destroy_t)(void *);
        destroy_t f = (destroy_t)dlsym(h->nccl_lib, "ncclCommDestroy");
        if (f) f(h->nccl_comm);
    }
    rxi_sams_free(h);
    rxi_mix_free(h);
    cudaFree(h->d_atom); cudaFree(h->d_atom_d); cudaFree(h->d_alch_list); cudaFree(h->d_states);
    cudaFree(h->d_pos_snap); cudaFree(h->d_vel_snap); cudaFree(h->d_retry);
    cudaFree(h->d_pos); cudaFree(h->d_vel); cudaFree(h->d_io); cudaFree(h->d_perm); cudaFree(h->d_u);
    cudaFree(h->d_nacc); cudaFree(h->d_nprop); cudaFree(h->d_pot); cudaFree(h->d_kin); cudaFree(h->d_nan);
    cudaFree(h->d_err); cudaFree(h->d_pairs);
    for (int i = 0; i < 8; i++) if (h->ev[i]) cudaEventDestroy(h->ev[i]);
    for (int i = 0; i < 2; i++) if (h->ev_user[i]) cudaEventDestroy(h->ev_user[i]);
    for (int i = 0; i < 2; i++) if (h->ev_walk[i]) cudaEventDestroy(h->ev_walk[i]);
    for (const auto &r : h->pinned) cudaHostUnregister((void *)r.first);
    cudaFree(h->d_moves);
    rxi_free_molecule(h);
    if (h->h_io) cudaFreeHost(h->h_io);
    if (h->stream) cudaStreamDestroy(h->stream);
    if (h->stream_rng) cudaStreamDestroy(h->stream_rng);
    delete h;
}

#define ENTER(h)                                  \
    if (!(h)) return RX_ERR_INVALID;              \
    (h)->err.clear();                             \
    RX_CHECK_CUDA(h, cudaSetDevice((h)->cfg.device))

extern "C" int rx_set_particles(rx_engine *h, const double *sigma, const double *epsilon, const double *mass,
                                const uint8_t *alch) {
    ENTER(h);
    if (h->cfg.system_kind == RX_SYSTEM_NONE) RX_FAIL(h, RX_ERR_INVALID, "rx_set_particles: engine has no particle system");
    if (h->cfg.system_kind == RX_SYSTEM_MOLECULE) RX_FAIL(h, RX_ERR_INVALID, "rx_set_particles: use rx_set_molecule for RX_SYSTEM_MOLECULE");
    if (!mass) RX_FAIL(h, RX_ERR_INVALID, "rx_set_particles: mass is required");
    const int N = h->cfg.n_atoms;
    const bool lj = h->cfg.system_kind == RX_SYSTEM_LJ_ALCH;
    if (lj && (!sigma || !epsilon)) RX_FAIL(h, RX_ERR_INVALID, "rx_set_particles: sigma and epsilon are required");
    std::vector<float4> a(N);
    std::vector<double4> ad(N);
    std::vector<int> al;
    for (int i = 0; i < N; i++) {
        const double s = lj ? sigma[i] : 1.0, e = lj ? epsilon[i] : 0.0, m = mass[i];
        const bool isal = lj && alch && alch[i];
        if (!(m > 0)) RX_FAIL(h, RX_ERR_INVALID, "rx_set_particles: masses must be > 0");
        if (lj && (!(s > 0) || e < 0)) RX_FAIL(h, RX_ERR_INVALID, "rx_set_particles: need sigma > 0 and epsilon >= 0");
        a[i] = make_float4((float)s, (float)sqrt(e), (float)(1.0 / m), isal ? 1.f : 0.f);
        ad[i] = make_double4(s, e, m, isal ? 1.0 : 0.0);
        if (isal) al.push_back(i);
    }
    h->n_alch = (int)al.size();
    RX_CHECK_CUDA(h, cudaMemcpy(h->d_atom, a.data(), sizeof(float4) * N, cudaMemcpyHostToDevice));
    RX_CHECK_CUDA(h, cudaMemcpy(h->d_atom_d, ad.data(), sizeof(double4) * N, cudaMemcpyHostToDevice));
    if (h->n_alch) RX_CHECK_CUDA(h, cudaMemcpy(h->d_alch_list, al.data(), sizeof(int) * h->n_alch, cudaMemcpyHostToDevice));
    // scratch for the lambda-controlled pair list of each owned replica
    long long cap = (long long)h->n_alch * (N - 1);
    if (cap > (1 << 18)) cap = 1 << 18;
    if (cap < 1) cap = 1;
    cudaFree(h->d_pairs);
    h->d_pairs = nullptr;
    h->pair_cap = (int)cap;
    RX_CHECK_CUDA(h, cudaMalloc(&h->d_pairs, sizeof(double2) * (size_t)cap * (h->kloc > 0 ? h->kloc : 1)));
    h->have_particles = true;
    return RX_OK;
}

extern "C" int rx_set_molecule(rx_engine *h, const rx_molecule *molecule) {
    ENTER(h);
    if (h->cfg.system_kind != RX_SYSTEM_MOLECULE) RX_FAIL(h, RX_ERR_INVALID, "rx_set_molecule: the engine was not created with RX_SYSTEM_MOLECULE");
    if (!molecule) RX_FAIL(h, RX_ERR_INVALID, "rx_set_molecule: null");
    if (molecule->n_bonds < 0 || molecule->n_angles < 0 || molecule->n_torsions < 0 || molecule->n_exclusions < 0 ||
        molecule->n_exceptions < 0 || molecule->n_constraints < 0)
        RX_FAIL(h, RX_ERR_INVALID, "rx_set_molecule: negative count");
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    return rxi_set_molecule(h, molecule);
}

static int convert_states(rx_engine *h, const rx_state_params *s, int n, std::vector<StateDev> &out, const char *who) {
    out.resize(n);
    for (int l = 0; l < n; l++) {
        if (!(s[l].temperature > 0)) RX_FAIL(h, RX_ERR_INVALID, std::string(who) + ": temperature must be > 0");
        if (h->cfg.system_kind == RX_SYSTEM_LJ_ALCH && !(s[l].lambda_sterics >= 0.0 && s[l].lambda_sterics <= 1.0))
            RX_FAIL(h, RX_ERR_INVALID, std::string(who) + ": lambda_sterics must be in [0, 1]");
        StateDev &d = out[l];
        d.kT = RX_KB * s[l].temperature;
        d.beta = 1.0 / d.kT;
        d.lambda = s[l].lambda_sterics;
        d.la = pow(s[l].lambda_sterics, h->cfg.softcore_a);
        d.ob = h->cfg.softcore_alpha * pow(1.0 - s[l].lambda_sterics, h->cfg.softcore_b);
        d.offset = s[l].energy_offset;
        d.ho_K = s[l].ho_K;
        for (int q = 0; q < 3; q++) d.ho_x0[q] = s[l].ho_x0[q];
    }
    return RX_OK;
}

extern "C" int rx_set_states(rx_engine *h, const rx_state_params *s) {
    ENTER(h);
    if (!s) RX_FAIL(h, RX_ERR_INVALID, "rx_set_states: null");
    const int M = h->cfg.n_states;
    int rc = convert_states(h, s, M, h->h_states, "rx_set_states");
    if (rc) return rc;
    RX_CHECK_CUDA(h, cudaMemcpy(h->d_states, h->h_states.data(), sizeof(StateDev) * M, cudaMemcpyHostToDevice));
    h->have_states = true;
    return RX_OK;
}

// Checks the arguments of a move (messages start with `who`) and stores it in *out; *out is untouched on failure.
static int make_move(rx_engine *h, const char *who, double timestep, double collision_rate, int32_t n_steps,
                     const char *splitting, int reassign, rx_state_move *out) {
    const std::string w(who);
    if (!(timestep > 0) || collision_rate < 0 || n_steps < 0) RX_FAIL(h, RX_ERR_INVALID, w + ": bad timestep/collision_rate/n_steps");
    if (!splitting) RX_FAIL(h, RX_ERR_INVALID, w + ": null splitting");
    const size_t n = strlen(splitting);
    if (n == 0 || n >= RX_MAX_PROGRAM) RX_FAIL(h, RX_ERR_INVALID, w + ": splitting must have 1..31 substeps");
    bool hasV = false, hasR = false, hasO = false;
    for (size_t i = 0; i < n; i++) {
        const char c = splitting[i];
        if (c == 'V') hasV = true; else if (c == 'R') hasR = true; else if (c == 'O') hasO = true;
        else RX_FAIL(h, RX_ERR_UNSUPPORTED, w + ": only R, V and O substeps are supported (no force groups / Metropolization)");
    }
    if (!(hasV && hasR && hasO)) RX_FAIL(h, RX_ERR_INVALID, w + ": splitting must contain R, V and O (integrators.py:1360-1363)");
    rx_state_move m;
    m.dt = timestep; m.gamma = collision_rate; m.n_steps = n_steps; m.reassign = reassign ? 1 : 0;
    memcpy(m.program, splitting, n);
    *out = m;
    return RX_OK;
}

extern "C" int rx_set_integrator(rx_engine *h, double timestep, double collision_rate, int32_t n_steps,
                                 const char *splitting) {
    ENTER(h);
    int rc = make_move(h, "rx_set_integrator", timestep, collision_rate, n_steps, splitting, 0, &h->move);
    if (rc) return rc;
    h->have_integrator = true;
    h->state_moves.clear();   // one move for every state again
    return RX_OK;
}

/* One MCMCMove per thermodynamic state (openmmtools/multistate/multistatesampler.py:906-910; a replica is propagated with
 * the move of the state it is in, :1311-1322).  Call after rx_set_integrator (which provides the move of every state not
 * set here) for each state whose move differs; rx_set_integrator again returns to one move for all states. */
extern "C" int rx_set_state_integrator(rx_engine *h, int32_t state, double timestep, double collision_rate, int32_t n_steps,
                                       const char *splitting, int32_t reassign_velocities) {
    ENTER(h);
    if (!h->have_integrator) RX_FAIL(h, RX_ERR_INVALID, "rx_set_state_integrator: rx_set_integrator must be called first");
    if (state < 0 || state >= h->cfg.n_states) RX_FAIL(h, RX_ERR_INVALID, "rx_set_state_integrator: state out of range");
    rx_state_move m;
    int rc = make_move(h, "rx_set_state_integrator", timestep, collision_rate, n_steps, splitting, reassign_velocities, &m);
    if (rc) return rc;
    if (h->state_moves.empty()) h->state_moves.assign((size_t)h->cfg.n_states, h->move);   // start from the common move
    h->state_moves[(size_t)state] = m;
    h->state_moves_dirty = true;
    return RX_OK;
}

static int local_range(rx_engine *h, int first, int count, int *lo, int *n, int *skip) {
    const int K = h->cfg.n_replicas;
    if (first < 0 || count < 0 || first + count > K) RX_FAIL(h, RX_ERR_INVALID, "replica range out of bounds");
    int a = first > h->k0 ? first : h->k0;
    int b = (first + count) < (h->k0 + h->kloc) ? (first + count) : (h->k0 + h->kloc);
    if (b < a) b = a;
    *lo = a - h->k0; *n = b - a; *skip = a - first;
    return RX_OK;
}

static int set_xyz(rx_engine *h, float4 *dst, int first, int count, const double *xyz, const char *what) {
    if (h->cfg.system_kind == RX_SYSTEM_NONE) RX_FAIL(h, RX_ERR_INVALID, "engine has no particle system");
    if (!xyz) RX_FAIL(h, RX_ERR_INVALID, std::string(what) + ": null buffer");
    int lo, n, skip;
    int rc = local_range(h, first, count, &lo, &n, &skip);
    if (rc) return rc;
    return rxi_convert_in(h, dst, lo, n, xyz + (size_t)skip * h->cfg.n_atoms * 3, false);
}
static int get_xyz(rx_engine *h, const float4 *src, int first, int count, double *xyz, bool wrap, const char *what) {
    if (h->cfg.system_kind == RX_SYSTEM_NONE) RX_FAIL(h, RX_ERR_INVALID, "engine has no particle system");
    if (!xyz) RX_FAIL(h, RX_ERR_INVALID, std::string(what) + ": null buffer");
    int lo, n, skip;
    int rc = local_range(h, first, count, &lo, &n, &skip);
    if (rc) return rc;
    return rxi_convert_out(h, src, lo, n, xyz + (size_t)skip * h->cfg.n_atoms * 3, wrap);
}

extern "C" int rx_set_positions(rx_engine *h, int32_t first, int32_t count, const double *xyz) {
    ENTER(h);
    return set_xyz(h, h->d_pos, first, count, xyz, "rx_set_positions");
}
extern "C" int rx_set_velocities(rx_engine *h, int32_t first, int32_t count, const double *xyz) {
    ENTER(h);
    return set_xyz(h, h->d_vel, first, count, xyz, "rx_set_velocities");
}
extern "C" int rx_get_positions(rx_engine *h, int32_t first, int32_t count, double *xyz) {
    ENTER(h);
    return get_xyz(h, h->d_pos, first, count, xyz, h->cfg.system_kind == RX_SYSTEM_LJ_ALCH, "rx_get_positions");
}
extern "C" int rx_get_velocities(rx_engine *h, int32_t first, int32_t count, double *xyz) {
    ENTER(h);
    return get_xyz(h, h->d_vel, first, count, xyz, false, "rx_get_velocities");
}

bool rxi_is_pinned(const rx_engine *h, const void *p, size_t bytes) {
    const char *c = (const char *)p;
    for (const auto &r : h->pinned)
        if (c >= r.first && c + bytes <= r.first + r.second) return true;
    return false;
}

/* Page-lock a caller buffer (cudaHostRegister) so that rx_set_* / rx_get_* copy straight between it and the device instead
 * of staging through the engine's own pinned buffer: the host-resident SamplerStates of MultiStateSampler live in one
 * such buffer.  The engine unregisters what is still registered when it is destroyed. */
extern "C" int rx_pin_host_memory(rx_engine *h, void *ptr, uint64_t bytes) {
    ENTER(h);
    if (!ptr || !bytes) RX_FAIL(h, RX_ERR_INVALID, "rx_pin_host_memory: null buffer");
    RX_CHECK_CUDA(h, cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterDefault));
    h->pinned.push_back(std::make_pair((const char *)ptr, (size_t)bytes));
    return RX_OK;
}
extern "C" int rx_unpin_host_memory(rx_engine *h, void *ptr) {
    ENTER(h);
    for (size_t q = 0; q < h->pinned.size(); q++)
        if (h->pinned[q].first == (const char *)ptr) {
            RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
            cudaHostUnregister(ptr);
            h->pinned.erase(h->pinned.begin() + q);
            return RX_OK;
        }
    RX_FAIL(h, RX_ERR_INVALID, "rx_unpin_host_memory: buffer was not registered");
}

extern "C" int rx_get_replica_energies(rx_engine *h, double *potential, double *kinetic) {
    ENTER(h);
    const int K = h->cfg.n_replicas;
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    if (potential) RX_CHECK_CUDA(h, cudaMemcpy(potential, h->d_pot, sizeof(double) * K, cudaMemcpyDeviceToHost));
    if (kinetic) RX_CHECK_CUDA(h, cudaMemcpy(kinetic, h->d_kin, sizeof(double) * K, cudaMemcpyDeviceToHost));
    return RX_OK;
}

extern "C" int rx_randomize_velocities(rx_engine *h, uint64_t seed, uint64_t stream) {
    ENTER(h);
    if (!h->have_particles || !h->have_states) RX_FAIL(h, RX_ERR_INVALID, "rx_randomize_velocities: set particles and states first");
    return rxi_randomize_velocities(h, seed, stream);
}

extern "C" int rx_minimize(rx_engine *h, double tolerance, int32_t max_iterations, double *rms_force, int32_t *iterations) {
    ENTER(h);
    if (!h->have_particles || !h->have_states) RX_FAIL(h, RX_ERR_INVALID, "rx_minimize: set particles and states first");
    if (!(tolerance > 0.0)) RX_FAIL(h, RX_ERR_INVALID, "rx_minimize: tolerance must be positive");
    if (max_iterations < 0) RX_FAIL(h, RX_ERR_INVALID, "rx_minimize: max_iterations must be >= 0");
    const int K = h->cfg.n_replicas;
    double *d_rms = nullptr;
    int *d_it = nullptr;
    RX_CHECK_CUDA(h, cudaMalloc(&d_rms, sizeof(double) * K));
    if (cudaMalloc(&d_it, sizeof(int) * K) != cudaSuccess) { cudaFree(d_rms); RX_FAIL(h, RX_ERR_CUDA, "rx_minimize: out of device memory"); }
    cudaMemsetAsync(d_rms, 0, sizeof(double) * K, h->stream);
    cudaMemsetAsync(d_it, 0, sizeof(int) * K, h->stream);
    int rc = rxi_minimize(h, tolerance, max_iterations == 0 ? 20000 : max_iterations, d_rms, d_it);
    if (rc == RX_OK && cudaStreamSynchronize(h->stream) != cudaSuccess) { h->err = "rx_minimize: kernel failed"; rc = RX_ERR_CUDA; }
    if (rc == RX_OK && rms_force) cudaMemcpy(rms_force, d_rms, sizeof(double) * K, cudaMemcpyDeviceToHost);
    if (rc == RX_OK && iterations) cudaMemcpy(iterations, d_it, sizeof(int) * K, cudaMemcpyDeviceToHost);
    cudaFree(d_rms); cudaFree(d_it);
    return rc;
}

extern "C" int rx_set_replica_states(rx_engine *h, const int64_t *states) {
    ENTER(h);
    const int K = h->cfg.n_replicas, M = h->cfg.n_states;
    std::vector<int> p(K);
    for (int k = 0; k < K; k++) {
        if (states[k] < 0 || states[k] >= M) RX_FAIL(h, RX_ERR_INVALID, "rx_set_replica_states: state index out of range");
        p[k] = (int)states[k];
    }
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    RX_CHECK_CUDA(h, cudaMemcpy(h->d_perm, p.data(), sizeof(int) * K, cudaMemcpyHostToDevice));
    return RX_OK;
}
extern "C" int rx_get_replica_states(rx_engine *h, int64_t *states) {
    ENTER(h);
    const int K = h->cfg.n_replicas;
    std::vector<int> p(K);
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    RX_CHECK_CUDA(h, cudaMemcpy(p.data(), h->d_perm, sizeof(int) * K, cudaMemcpyDeviceToHost));
    for (int k = 0; k < K; k++) states[k] = p[k];
    return RX_OK;
}

static int check_ready(rx_engine *h, const char *who) {
    if (h->cfg.system_kind == RX_SYSTEM_NONE) RX_FAIL(h, RX_ERR_INVALID, std::string(who) + ": engine has no particle system");
    if (!h->have_particles || !h->have_states) RX_FAIL(h, RX_ERR_INVALID, std::string(who) + ": rx_set_particles and rx_set_states must be called first");
    return RX_OK;
}

static int check_device_error(rx_engine *h) {
    int e = 0;
    RX_CHECK_CUDA(h, cudaMemcpy(&e, h->d_err, sizeof(int), cudaMemcpyDeviceToHost));
    if (e) {
        cudaMemset(h->d_err, 0, sizeof(int));
        RX_FAIL(h, e, e == RX_ERR_CAPACITY ? "lambda-controlled pair list overflowed its capacity" : "device-side error");
    }
    return RX_OK;
}

static int finish_propagate(rx_engine *h, PhaseTimer &T, int32_t *nan_flags, const char *who);

extern "C" int rx_propagate(rx_engine *h, uint64_t seed, uint64_t iteration, int32_t reassign, int32_t *nan_flags) {
    ENTER(h);
    int rc = check_ready(h, "rx_propagate");
    if (rc) return rc;
    if (!h->have_integrator) RX_FAIL(h, RX_ERR_INVALID, "rx_propagate: rx_set_integrator must be called first");
    PhaseTimer T(h, 1);
    int launches = 0;
    rc = rxi_snapshot_state(h);
    if (rc) return rc;
    rc = rxi_propagate(h, seed, iteration, reassign, &launches);
    if (rc) return rc;
    T.stop(launches);
    return finish_propagate(h, T, nan_flags, "rx_propagate");
}

/* Replaces the restart loop of BaseIntegratorMove.apply (openmmtools/mcmc.py:706-759): the replicas whose NaN flag is set
 * go back to the state they had when rx_propagate began and are propagated again (other noise: pass another seed); the
 * replicas that came through are left alone. */
extern "C" int rx_propagate_retry(rx_engine *h, uint64_t seed, uint64_t iteration, int32_t reassign, int32_t *nan_flags) {
    ENTER(h);
    int rc = check_ready(h, "rx_propagate_retry");
    if (rc) return rc;
    if (!h->have_integrator) RX_FAIL(h, RX_ERR_INVALID, "rx_propagate_retry: rx_set_integrator must be called first");
    PhaseTimer T(h, 1);
    int launches = 0;
    rc = rxi_restore_failed(h);
    if (rc) return rc;
    rc = rxi_propagate(h, seed, iteration, reassign, &launches, h->d_retry);
    if (rc) return rc;
    T.stop(launches + 1);
    return finish_propagate(h, T, nan_flags, "rx_propagate_retry");
}

// The NaN flags of the last propagation: *any tells whether an owned replica has one; nan_flags[K], when given, receives the
// owned replicas' flags and 0 for the others.
static int owned_nan_flags(rx_engine *h, int32_t *nan_flags, bool *any) {
    const int K = h->cfg.n_replicas;
    std::vector<int> f(K, 0);
    RX_CHECK_CUDA(h, cudaMemcpy(f.data(), h->d_nan, sizeof(int) * K, cudaMemcpyDeviceToHost));
    *any = false;
    for (int k = 0; k < K; k++) {
        const int v = (k >= h->k0 && k < h->k0 + h->kloc) ? f[k] : 0;
        if (nan_flags) nan_flags[k] = v;
        *any |= v != 0;
    }
    return RX_OK;
}

static int finish_propagate(rx_engine *h, PhaseTimer &T, int32_t *nan_flags, const char *who) {
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    T.accumulate();
    bool any = false;
    int rc = owned_nan_flags(h, nan_flags, &any);
    if (rc) return rc;
    if (any) RX_FAIL(h, RX_ERR_NAN, std::string(who) + ": NaN encountered in positions, velocities or potential energy");
    return RX_OK;
}

extern "C" int rx_compute_energies(rx_engine *h, double *u_out) {
    ENTER(h);
    int rc = check_ready(h, "rx_compute_energies");
    if (rc) return rc;
    PhaseTimer T(h, 2);
    int launches = 0;
    rc = rxi_compute_energy_rows(h, &launches);
    if (rc) return rc;
    rc = rxi_allgather_energies(h);
    if (rc) return rc;
    T.stop(launches);
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    T.accumulate();
    rc = check_device_error(h);
    if (rc) return rc;
    if (u_out) RX_CHECK_CUDA(h, cudaMemcpy(u_out, h->d_u, sizeof(double) * (size_t)h->cfg.n_replicas * h->cfg.n_states, cudaMemcpyDeviceToHost));
    return RX_OK;
}

extern "C" int rx_set_energies(rx_engine *h, const double *u) {
    ENTER(h);
    if (!u) RX_FAIL(h, RX_ERR_INVALID, "rx_set_energies: null");
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    RX_CHECK_CUDA(h, cudaMemcpy(h->d_u, u, sizeof(double) * (size_t)h->cfg.n_replicas * h->cfg.n_states, cudaMemcpyHostToDevice));
    return RX_OK;
}
extern "C" int rx_get_energies(rx_engine *h, double *u) {
    ENTER(h);
    if (!u) RX_FAIL(h, RX_ERR_INVALID, "rx_get_energies: null");
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    RX_CHECK_CUDA(h, cudaMemcpy(u, h->d_u, sizeof(double) * (size_t)h->cfg.n_replicas * h->cfg.n_states, cudaMemcpyDeviceToHost));
    return RX_OK;
}

extern "C" int rx_compute_energies_at(rx_engine *h, const rx_state_params *st, int32_t n, double *u_out) {
    ENTER(h);
    int rc = check_ready(h, "rx_compute_energies_at");
    if (rc) return rc;
    if (!st || !u_out || n < 1) RX_FAIL(h, RX_ERR_INVALID, "rx_compute_energies_at: bad arguments");
    std::vector<StateDev> hs;
    rc = convert_states(h, st, n, hs, "rx_compute_energies_at");
    if (rc) return rc;
    const int K = h->cfg.n_replicas;
    StateDev *d_st = nullptr;
    double *d_out = nullptr;
    RX_CHECK_CUDA(h, cudaMalloc(&d_st, sizeof(StateDev) * n));
    cudaError_t e = cudaMalloc(&d_out, sizeof(double) * (size_t)K * n);
    if (e != cudaSuccess) { cudaFree(d_st); RX_FAIL(h, RX_ERR_CUDA, std::string("cudaMalloc: ") + cudaGetErrorString(e)); }
    int launches = 0;
    cudaMemcpyAsync(d_st, hs.data(), sizeof(StateDev) * n, cudaMemcpyHostToDevice, h->stream);
    cudaMemsetAsync(d_out, 0, sizeof(double) * (size_t)K * n, h->stream);
    rc = rxi_compute_energy_rows_at(h, d_st, n, d_out, &launches);
    if (!rc) rc = rxi_allgather_rows(h, d_out, n);
    if (!rc) {
        e = cudaMemcpyAsync(u_out, d_out, sizeof(double) * (size_t)K * n, cudaMemcpyDeviceToHost, h->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
        if (e != cudaSuccess) { h->err = std::string("rx_compute_energies_at: ") + cudaGetErrorString(e); rc = RX_ERR_CUDA; }
    }
    cudaStreamSynchronize(h->stream);
    cudaFree(d_st);
    cudaFree(d_out);
    if (rc) return rc;
    h->phase_launches[2] += launches;
    return check_device_error(h);
}

extern "C" int rx_mix_seed(rx_engine *h, int32_t stream, uint32_t seed) {
    ENTER(h);
    return rxi_mix_seed(h, stream, seed);
}
extern "C" int rx_mix_skip(rx_engine *h, int32_t stream, uint64_t n_words) {
    ENTER(h);
    return rxi_mix_skip(h, stream, n_words);
}

static int fetch_mix_results(rx_engine *h, int64_t *states_out, int64_t *nacc, int64_t *nprop) {
    const size_t mm = (size_t)h->cfg.n_states * h->cfg.n_states;
    if (states_out) { int rc = rx_get_replica_states(h, states_out); if (rc) return rc; }
    if (nacc) RX_CHECK_CUDA(h, cudaMemcpy(nacc, h->d_nacc, sizeof(int64_t) * mm, cudaMemcpyDeviceToHost));
    if (nprop) RX_CHECK_CUDA(h, cudaMemcpy(nprop, h->d_nprop, sizeof(int64_t) * mm, cudaMemcpyDeviceToHost));
    return RX_OK;
}

extern "C" int rx_mix_swap_all(rx_engine *h, int64_t nswap, int64_t *states_out, int64_t *nacc, int64_t *nprop) {
    ENTER(h);
    if (nswap < 0) RX_FAIL(h, RX_ERR_INVALID, "rx_mix_swap_all: nswap_attempts must be >= 0");
    PhaseTimer T(h, 0);
    int launches = 0;
    int rc = rxi_mix_swap_all(h, nswap, &launches);
    if (rc) return rc;
    T.stop(launches);
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    T.accumulate();
    return fetch_mix_results(h, states_out, nacc, nprop);
}

extern "C" int rx_mix_swap_neighbors(rx_engine *h, int64_t *states_out, int64_t *nacc, int64_t *nprop) {
    ENTER(h);
    PhaseTimer T(h, 0);
    int launches = 0;
    int rc = rxi_mix_swap_neighbors(h, &launches);
    if (rc) return rc;
    T.stop(launches);
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    T.accumulate();
    return fetch_mix_results(h, states_out, nacc, nprop);
}

extern "C" int rx_get_mix_counts(rx_engine *h, int64_t *nacc, int64_t *nprop) {
    ENTER(h);
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    return fetch_mix_results(h, nullptr, nacc, nprop);
}

extern "C" int rx_mix_stream_position(rx_engine *h, int32_t stream, uint64_t *words) {
    ENTER(h);
    if (stream < 0 || stream > 1 || !words) RX_FAIL(h, RX_ERR_INVALID, "rx_mix_stream_position: bad arguments");
    *words = h->streams[stream].consumed;
    return RX_OK;
}

// The fused iteration loop of multistatesampler.py:776-782, n_iterations times: phase 0 on the previous iteration's energies
// (`step(iteration, &launches)`: a mixing step, a SAMS step or nothing) -> propagate -> energies.  Messages start with `who`.
template <class Step>
static int run_iterations(rx_engine *h, const char *who, int32_t n_iterations, uint64_t seed, uint64_t first_iteration,
                          int32_t reassign, Step &&step) {
    for (int it = 0; it < n_iterations; it++) {
        int lm = 0, lp = 0, le = 0;
        PhaseTimer Tm(h, 0);
        int rc = step(first_iteration + it, &lm);
        if (rc) return rc;
        Tm.stop(lm);
        PhaseTimer Tp(h, 1);
        rc = rxi_propagate(h, seed, first_iteration + it, reassign, &lp);
        if (rc) return rc;
        Tp.stop(lp);
        PhaseTimer Te(h, 2);
        rc = rxi_compute_energy_rows(h, &le);
        if (rc) return rc;
        rc = rxi_allgather_energies(h);
        if (rc) return rc;
        Te.stop(le);
        RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
        Tm.accumulate(); Tp.accumulate(); Te.accumulate();
    }
    int rc = check_device_error(h);
    if (rc) return rc;
    bool any = false;
    rc = owned_nan_flags(h, nullptr, &any);
    if (rc) return rc;
    if (any) RX_FAIL(h, RX_ERR_NAN, std::string(who) + ": NaN encountered in a replica");
    return RX_OK;
}

extern "C" int rx_run_iterations(rx_engine *h, int32_t n_iterations, int32_t mixing, uint64_t seed,
                                 uint64_t first_iteration, int32_t reassign) {
    ENTER(h);
    int rc = check_ready(h, "rx_run_iterations");
    if (rc) return rc;
    if (!h->have_integrator) RX_FAIL(h, RX_ERR_INVALID, "rx_run_iterations: rx_set_integrator must be called first");
    if (mixing < 0 || mixing > 2) RX_FAIL(h, RX_ERR_INVALID, "rx_run_iterations: mixing must be 0, 1 or 2");
    const long long K = h->cfg.n_replicas;
    return run_iterations(h, "rx_run_iterations", n_iterations, seed, first_iteration, reassign, [&](uint64_t, int *lm) {
        if (mixing == 1) return rxi_mix_swap_all(h, K * K * K, lm);
        if (mixing == 2) return rxi_mix_swap_neighbors(h, lm);
        return (int)RX_OK;
    });
}

// ---- SAMS (rx_sams.cuh) ------------------------------------------------------------------------------------------------------
extern "C" int rx_sams_set(rx_engine *h, const rx_sams_config *config, const double *log_target, const double *logZ,
                           const int64_t *histogram) {
    ENTER(h);
    if (!config || !log_target || !logZ) RX_FAIL(h, RX_ERR_INVALID, "rx_sams_set: null argument");
    return rxi_sams_set(h, config, log_target, logZ, histogram);
}

extern "C" int rx_sams_step(rx_engine *h, int64_t iteration, int32_t update_weights, const int64_t *histogram) {
    ENTER(h);
    int rc = check_ready(h, "rx_sams_step");
    if (rc) return rc;
    if (histogram && (rc = rxi_sams_set_histogram(h, histogram))) return rc;
    int lm = 0;
    PhaseTimer Tm(h, 0);
    rc = rxi_sams_step(h, iteration, update_weights, &lm);
    if (rc) return rc;
    Tm.stop(lm);
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    Tm.accumulate();
    return check_device_error(h);
}

extern "C" int rx_sams_get(rx_engine *h, double *logZ, double *log_weights, int64_t *histogram, int32_t *stage, int64_t *t0,
                           double *gamma, int64_t *states, int64_t *previous_states) {
    ENTER(h);
    return rxi_sams_get(h, logZ, log_weights, histogram, stage, t0, gamma, states, previous_states);
}

extern "C" int rx_sams_run_iterations(rx_engine *h, int32_t n_iterations, uint64_t seed, uint64_t first_iteration, int32_t reassign) {
    ENTER(h);
    int rc = check_ready(h, "rx_sams_run_iterations");
    if (rc) return rc;
    if (!h->have_integrator) RX_FAIL(h, RX_ERR_INVALID, "rx_sams_run_iterations: rx_set_integrator must be called first");
    // sams.py:395-437 as the mixing: jump + weight update
    return run_iterations(h, "rx_sams_run_iterations", n_iterations, seed, first_iteration, reassign, [&](uint64_t iteration, int *lm) {
        return rxi_sams_step(h, (long long)iteration, iteration > 0 ? 1 : 0, lm);
    });
}

extern "C" int rx_get_phase_times(rx_engine *h, double ms[4], int64_t counts[4], int32_t reset) {
    ENTER(h);
    for (int i = 0; i < 4; i++) {
        if (ms) ms[i] = h->phase_ms[i];
        if (counts) counts[i] = h->phase_launches[i];
        if (reset) { h->phase_ms[i] = 0; h->phase_launches[i] = 0; }
    }
    return RX_OK;
}

extern "C" int rx_timer_mark(rx_engine *h, int32_t which) {
    ENTER(h);
    if (which < 0 || which > 1) RX_FAIL(h, RX_ERR_INVALID, "rx_timer_mark: which must be 0 or 1");
    RX_CHECK_CUDA(h, cudaEventRecord(h->ev_user[which], h->stream));
    return RX_OK;
}
extern "C" int rx_timer_elapsed(rx_engine *h, double *ms) {
    ENTER(h);
    if (!ms) RX_FAIL(h, RX_ERR_INVALID, "rx_timer_elapsed: null");
    RX_CHECK_CUDA(h, cudaEventSynchronize(h->ev_user[1]));
    float f = 0;
    RX_CHECK_CUDA(h, cudaEventElapsedTime(&f, h->ev_user[0], h->ev_user[1]));
    *ms = f;
    return RX_OK;
}
extern "C" int rx_selftest_exp(rx_engine *h, const double *x, double *y, int32_t n) {
    if (!h) return RX_ERR_INVALID;
    if (n > 0 && (!x || !y)) RX_FAIL(h, RX_ERR_INVALID, "rx_selftest_exp: null array");
    RX_CHECK_CUDA(h, cudaSetDevice(h->cfg.device));
    return rxi_selftest_exp(h, x, y, n);
}

extern "C" int rx_get_mix_stats(rx_engine *h, int64_t out[6]) {
    ENTER(h);
    for (int i = 0; i < 6; i++) out[i] = h->mix_stats[i];
    return RX_OK;
}

// ---- NCCL through dlopen: the single-GPU path has no NCCL dependency -------------------------------
typedef struct { char internal[128]; } rx_nccl_id;
typedef int (*nccl_get_id_t)(rx_nccl_id *);
typedef int (*nccl_init_rank_t)(void **, int, rx_nccl_id, int);
typedef int (*nccl_allgather_t)(const void *, void *, size_t, int, void *, cudaStream_t);
typedef const char *(*nccl_errstr_t)(int);
#define RX_NCCL_FLOAT64 8 /* ncclFloat64 / ncclDouble in nccl.h's ncclDataType_t */

extern "C" int rx_comm_unique_id(const char *path, void *id_out) {
    if (!path || !id_out) { g_rx_create_error = "rx_comm_unique_id: null argument"; return RX_ERR_INVALID; }
    void *lib = dlopen(path, RTLD_NOW | RTLD_GLOBAL);
    if (!lib) { g_rx_create_error = std::string("dlopen failed: ") + dlerror(); return RX_ERR_COMM; }
    nccl_get_id_t f = (nccl_get_id_t)dlsym(lib, "ncclGetUniqueId");
    if (!f) { g_rx_create_error = "ncclGetUniqueId not found"; return RX_ERR_COMM; }
    rx_nccl_id id;
    int r = f(&id);
    if (r != 0) { g_rx_create_error = "ncclGetUniqueId failed"; return RX_ERR_COMM; }
    memcpy(id_out, &id, sizeof(id));
    return RX_OK;
}

extern "C" int rx_comm_init(rx_engine *h, const char *path, const void *unique_id) {
    ENTER(h);
    if (h->cfg.world_size == 1) return RX_OK;
    if (!path || !unique_id) RX_FAIL(h, RX_ERR_INVALID, "rx_comm_init: null argument");
    h->nccl_lib = dlopen(path, RTLD_NOW | RTLD_GLOBAL);
    if (!h->nccl_lib) RX_FAIL(h, RX_ERR_COMM, std::string("dlopen failed: ") + dlerror());
    nccl_init_rank_t f = (nccl_init_rank_t)dlsym(h->nccl_lib, "ncclCommInitRank");
    if (!f) RX_FAIL(h, RX_ERR_COMM, "ncclCommInitRank not found");
    rx_nccl_id id;
    memcpy(&id, unique_id, sizeof(id));
    int r = f(&h->nccl_comm, h->cfg.world_size, id, h->cfg.rank);
    if (r != 0) {
        nccl_errstr_t es = (nccl_errstr_t)dlsym(h->nccl_lib, "ncclGetErrorString");
        RX_FAIL(h, RX_ERR_COMM, std::string("ncclCommInitRank failed: ") + (es ? es(r) : "?"));
    }
    if ((h->cfg.n_replicas % h->cfg.world_size) != 0) RX_FAIL(h, RX_ERR_INVALID, "rx_comm_init: n_replicas must be divisible by world_size");
    return RX_OK;
}

int rxi_allgather_rows(rx_engine *h, double *d_matrix, int n_cols) {
    if (h->cfg.world_size == 1) return RX_OK;
    if (!h->nccl_comm) RX_FAIL(h, RX_ERR_COMM, "world_size > 1 but rx_comm_init has not been called");
    nccl_allgather_t f = (nccl_allgather_t)dlsym(h->nccl_lib, "ncclAllGather");
    if (!f) RX_FAIL(h, RX_ERR_COMM, "ncclAllGather not found");
    const size_t cnt = (size_t)h->kloc * n_cols;
    // in place: each rank's rows already sit at their final offset
    int r = f(d_matrix + (size_t)h->k0 * n_cols, d_matrix, cnt, RX_NCCL_FLOAT64, h->nccl_comm, h->stream);
    if (r != 0) RX_FAIL(h, RX_ERR_COMM, "ncclAllGather failed");
    return RX_OK;
}

int rxi_allgather_energies(rx_engine *h) { return rxi_allgather_rows(h, h->d_u, h->cfg.n_states); }
