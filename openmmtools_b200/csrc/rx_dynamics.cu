// rx_dynamics.cu -- propagation (Langevin splitting dynamics) and the reduced-potential matrix.
//
// k_propagate   replaces MultiStateSampler._propagate_replicas (multistatesampler.py:1287-1337) ->
//               BaseIntegratorMove.apply (mcmc.py:668-776) -> LangevinIntegrator V/R/O substeps
//               (integrators.py:1404-1460): one CTA per replica, the replica lives in shared memory and
//               registers for all n_steps, one force evaluation per step (CustomIntegrator's lazy `f`).
// k_energy_rows replaces MultiStateSampler._compute_replica_energies (multistatesampler.py:1458-1494) ->
//               ThermodynamicState.reduced_potential_at_states (states.py:911-992): like the reference it
//               evaluates the lambda-independent groups once per configuration and only the
//               lambda-controlled pairs once per state (states.py:3649-3691).  All double precision.
// Energy function: alchemy/alchemy.py:1379-1388 (soft-core sterics), :1723-1750 / :1903-1919 (which pairs go
// to which force), testsystems.py:1956-1997 (switched LJ, cutoff-periodic).
#include "rx_internal.cuh"
#include <cooperative_groups.h>
namespace cg = cooperative_groups;
#include <math.h>
#include <string.h>
#include <stdlib.h>
#include <type_traits>

// ---------------------------------------------------------------------------------------------------
// Philox4x32-10 counter-based generator: noise is a pure function of (seed, iteration, replica, atom, step)
// ---------------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ void philox_round(uint32_t &c0, uint32_t &c1, uint32_t &c2, uint32_t &c3,
                                                       uint32_t k0, uint32_t k1) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
}
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
    uint32_t c0 = ctr.x, c1 = ctr.y, c2 = ctr.z, c3 = ctr.w, k0 = key.x, k1 = key.y;
#pragma unroll
    for (int r = 0; r < 10; r++) {
        philox_round(c0, c1, c2, c3, k0, k1);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}
// three standard normals from one Philox block (Box-Muller on words 0,1 and 2,3); fast-math intrinsics: the
// absolute error (~1e-6) is far below the float32 resolution of the velocity update it feeds
__device__ __forceinline__ float3 philox_normal3(uint4 r) {
    const float u1 = ((float)(r.x >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u2 = ((float)(r.y >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u3 = ((float)(r.z >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u4 = ((float)(r.w >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float ra = sqrtf(-2.0f * __logf(u1)), rb = sqrtf(-2.0f * __logf(u3));
    float s1, c1;
    __sincosf(6.283185307179586f * u2, &s1, &c1);
    const float c2 = __cosf(6.283185307179586f * u4);
    return make_float3(ra * c1, ra * s1, rb * c2);
}

__device__ __forceinline__ float fast_rcp(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float fast_rsqrt(float x) { float y; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// ---------------------------------------------------------------------------------------------------
// A move as the kernels see it (move_dev()).  A launch carries its move in DynParams::mv; when the states carry different
// moves (multistatesampler.py:906-910: one MCMCMove per state) a table holds one per state, and a replica is propagated with
// the move of the state it is in.  (Field order: inside DynParams, dt and n_steps fall on 8-byte boundaries, so the
// kernels read dt, a and n_steps, n_prog in pairs.)
struct MoveDev {
    float dt, a, b;             // timestep, O-step coefficients exp(-gamma h), sqrt(1-exp(-2 gamma h))
    int reassign;
    double dt_d, a_d, b_d;      // the same in f64 (the molecule kernel)
    int n_steps, n_prog, nV, nR, nO;
    char prog[RX_MAX_PROGRAM];
};

struct DynParams {
    int N, kind;
    float Lx, Ly, Lz, iLx, iLy, iLz;
    float rc2, rs2, rs, inv_w;  // cutoff^2, switch^2, switch, 1/(rc-rs)
    int use_switch, annihilate, c_is_6;
    float sc_c;                 // softcore_c
    MoveDev mv;                 // the launch's move
    int maxnb;                  // Verlet-list capacity per atom (0: all-pairs only)
    int sort_atoms;             // re-deal atoms to threads by neighbour count at every list build
    float rl2, rin2;            // (cutoff + skin_out)^2, (cutoff + skin_in)^2
    float half_in2, half_out2;  // (skin_in/2)^2, ((skin_out - skin_in)/2)^2
};

struct PairLam { float la, ob; };

// Pair interaction in float: returns -dU/dr / r (so f_i += ret * (xi - xj)) and optionally the energy.
// One formula for every pair kind: plain LJ is the soft core with lambda^a = 1, alpha (1-lambda)^b = 0
// (x = (sigma/r)^6), so a warp never diverges on the pair kind.  Approximate reciprocals (1 ulp-class MUFU ops).
// C6: softcore_c == 6 (the reference default, alchemy.py:424); SW: the switching function is on.
template <bool C6, bool SW, bool ENERGY>
__device__ __forceinline__ float lj_pair_f(const DynParams &p, float r2, float sig, float eps, bool softcore,
                                           PairLam lam, float &energy) {
    const float la = softcore ? lam.la : 1.0f, ob = softcore ? lam.ob : 0.0f;
    const float inv_r2 = fast_rcp(r2);
    const float q = r2 * fast_rcp(sig * sig);
    float rsc, x, iD;
    if (C6) { rsc = q * q * q; iD = fast_rcp(ob + rsc); x = iD; }
    else { rsc = __powf(q, 0.5f * p.sc_c); const float D = ob + rsc; iD = fast_rcp(D); x = __powf(D, -6.0f / p.sc_c); }
    const float t4 = la * 4.0f * eps;
    const float tx = t4 * x;
    float e = tx * (x - 1.0f);
    // -dU/dr / r = t4 (2x-1) 6 x (r/sigma)^c / (D r^2)
    float fr = tx * (12.0f * x - 6.0f) * (rsc * iD) * inv_r2;
    if (SW && r2 > p.rs2) {
        const float rinv = fast_rsqrt(r2);
        const float r = r2 * rinv;
        const float t = (r - p.rs) * p.inv_w;
        const float t2 = t * t;
        const float S = 1.0f + t2 * t * (-10.0f + t * (15.0f - 6.0f * t));
        const float dS = t2 * (-30.0f + t * (60.0f - 30.0f * t)) * p.inv_w;
        fr = fr * S - e * dS * rinv;
        e *= S;
    }
    if (ENERGY) energy = e;
    return fr;
}

__device__ __forceinline__ double block_reduce_sum(double v, double *s_red) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (l == 0) s_red[w] = v;
    __syncthreads();
    double t = 0;
    if (threadIdx.x == 0) for (int q = 0; q < nw; q++) t += s_red[q];  // fixed order: deterministic
    return t;  // valid on thread 0
}

// Shared-memory accesses by 32-bit shared-space address: the generic-pointer path re-derives the CTA's shared window
// (S2R SR_CgaCtaId + LEA) inside the pair loop.
__device__ __forceinline__ float4 lds_f4(unsigned a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
    return v;
}
#define RX_MAX_ATOMS 1024
__device__ __forceinline__ float2 lds_f2(unsigned a) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ unsigned lds_u16(unsigned a) {
    unsigned short v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ void sts_u16(unsigned a, unsigned v) {
    asm volatile("st.shared.u16 [%0], %1;" :: "r"(a), "h"((unsigned short)v) : "memory");
}

// Minimum image without the XU pipe: round-to-nearest-even of d/L through the 1.5*2^23 magic constant
// (|d/L| < 2^22), two FMA-pipe operations instead of FMUL + FRND.
__device__ __forceinline__ float min_image_f(float d, float L, float iL) {
    const float n = __fadd_rn(__fmaf_rn(d, iL, 12582912.0f), -12582912.0f);
    return __fmaf_rn(-L, n, d);
}

// Everything the pair loop needs that does not change inside a launch, gathered in registers once.
struct PairCtx {
    float Lx, Ly, Lz, iLx, iLy, iLz, rc2;
    float x, y, z, sig_i, se_i;
    bool alch_i;
    PairLam lam;
};

// One candidate pair with atom j (position records at pos_base, parameter records par_off bytes further).
template <bool C6, bool SW, bool ENERGY>
__device__ __forceinline__ void pair_term(const DynParams &p, const PairCtx &c, unsigned pos_base, int par_off, unsigned j,
                                          float &ax, float &ay, float &az, float &en) {
    const unsigned aj = pos_base + 16u * j;
    const float4 pj = lds_f4(aj);
    const float dx = min_image_f(c.x - pj.x, c.Lx, c.iLx), dy = min_image_f(c.y - pj.y, c.Ly, c.iLy),
                dz = min_image_f(c.z - pj.z, c.Lz, c.iLz);
    const float r2 = dx * dx + dy * dy + dz * dz;
    if (r2 < c.rc2) {
        const float2 qj = lds_f2(aj + (unsigned)par_off);
        const bool alch_j = qj.y != 0.f;
        const bool soft = (c.alch_i != alch_j) || (c.alch_i && alch_j && p.annihilate);
        float e;
        const float fr = lj_pair_f<C6, SW, ENERGY>(p, r2, 0.5f * (c.sig_i + pj.w), c.se_i * qj.x, soft, c.lam, e);
        ax += fr * dx; ay += fr * dy; az += fr * dz;
        if (ENERGY) en += 0.5f * e;
    }
}

// Force on one atom from the inner part of its neighbour list or, in the fallback, from all other atoms.
template <bool C6, bool SW, bool ENERGY>
__device__ __forceinline__ void lj_forces(const DynParams &p, const PairCtx &c, unsigned pos_base, int par_off,
                                          unsigned nb_t, int N, int ncol, int a, bool use_list, int n_inner,
                                          float &fx, float &fy, float &fz, float &en) {
    float ax = 0.f, ay = 0.f, az = 0.f, e = 0.f;
    if (use_list) {
        const unsigned stride = 2u * (unsigned)ncol;
        unsigned q = nb_t;
        for (int n = 0; n < n_inner; n++, q += stride)
            pair_term<C6, SW, ENERGY>(p, c, pos_base, par_off, lds_u16(q), ax, ay, az, e);
    } else {
        for (int j = 0; j < N; j++)
            if (j != a) pair_term<C6, SW, ENERGY>(p, c, pos_base, par_off, (unsigned)j, ax, ay, az, e);
    }
    fx = ax; fy = ay; fz = az; en = e;
}

#define RX_SORT_BINS 128

// One CTA per owned replica, one atom per thread (N <= 1024).
//
// Neighbour search is a dual list held in shared memory, one column per thread:
//   outer list  every j with r < cutoff + skin_out when it was built (an all-pairs pass);
//   inner list  the leading n_inner entries of the column: the outer entries with r < cutoff + skin_in when the
//               column was last partitioned.  The force loop visits only these.
// The column is re-partitioned when some atom has moved more than skin_in/2 since the last partition, and the outer
// list is rebuilt when (checked at that moment) some atom has moved more than (skin_out - skin_in)/2 since the build,
// so that a pair missing from the outer list is still farther than cutoff + skin_in.
//
// Which atom a thread owns is re-decided at every outer build: atoms are dealt to threads in order of their inner
// neighbour count, so the lanes of a warp run pair loops of nearly equal length.  Per-atom results do not depend on
// the assignment (each atom sums its own list in list order, noise is keyed by atom id, the energy reductions run in
// atom order).
//
// Positions are double buffered: a force evaluation writes the moved positions into the buffer the previous
// evaluation did not read, and the displacement vote (__syncthreads_or) is the only barrier of the step.
// A replica may be split over a cluster of CL = 4 thread blocks (prop_plan() chooses it for a few large replicas, CL = 1
// otherwise): block q of the cluster owns the atoms [q Nq, (q+1) Nq), every block keeps ALL positions in its own shared
// memory -- a block writes the new positions of its atoms into every block's buffer through distributed shared memory -- and
// the step's only barrier becomes a cluster barrier.  The displacement votes are cluster wide, so the lists are rebuilt at the
// same steps and with the same contents as in one block: trajectories do not depend on CL (each atom sums its own list in list
// order, noise is keyed by atom id).
// PS: per-state moves (the move comes from `moves[state]` instead of `p.mv`).
template <bool C6, bool SW, int CL, bool PS>
__global__ void __launch_bounds__(1024) k_propagate(DynParams p, const float4 *__restrict__ atom,
                                                    const StateDev *__restrict__ states, const int *__restrict__ perm,
                                                    float4 *__restrict__ pos, float4 *__restrict__ vel, int k0,
                                                    uint2 key, uint32_t iteration,
                                                    double *__restrict__ pot, double *__restrict__ kin,
                                                    int *__restrict__ nan_flag, const int *__restrict__ only,
                                                    const MoveDev *__restrict__ moves) {
    static_assert(CL == 1 || CL == 4, "a replica runs in one block or in a cluster of four");
    extern __shared__ float4 s_dyn[];
    // (the whole cluster takes this exit together: `only` is indexed by replica)
    if (only && !only[k0 + blockIdx.x / CL]) return;   // a retry launch propagates the replicas that failed, nothing else
    float4 *s_par = s_dyn + RX_MAX_ATOMS;  // [RX_MAX_ATOMS] (sqrt_eps, alch, -, -); s_dyn[0..] / s_dyn[2*MAX..]: positions
    float4 *s_ref = s_dyn + 3 * RX_MAX_ATOMS;                  // [nthr] the thread's position at the last outer build
    unsigned short *s_nb = (unsigned short *)(s_ref + blockDim.x);  // [maxnb][nthr] lists, slot-major (conflict free)
    __shared__ double s_red[32];
    __shared__ int s_vote[2];            // cluster-wide votes (alternating words)
    __shared__ double s_part[3 * 4];     // per-block partial sums, gathered in block 0 of the cluster
    const int r = blockIdx.x / CL, q = blockIdx.x % CL, k = k0 + r, t = threadIdx.x, nthr = blockDim.x;
    const int Nq = (p.N + CL - 1) / CL, a_base = q * Nq;
    const int n_own = min(Nq, p.N - a_base);
    const bool active = t < n_own;   // threads beyond the block's atoms own none (they keep an id past the block's range)
    int a = a_base + t;              // the atom this thread owns
    unsigned vote_id = 0;
    if (t < 2) s_vote[t] = 0;
    // OR of `flag` over all threads of the cluster (of the block when CL == 1), doubling as the step's barrier
    auto cluster_or = [&](bool flag) -> bool {
        if (CL == 1) return __syncthreads_or(flag ? 1 : 0) != 0;
        vote_id++;
        int *word = &s_vote[vote_id & 1u];
        if (flag) {
            cg::cluster_group cl = cg::this_cluster();
#pragma unroll
            for (int c = 0; c < CL; c++) *cl.map_shared_rank(word, c) = (int)vote_id;   // every voter writes the same value
        }
        cg::this_cluster().sync();   // release / acquire: the positions and the votes written before it are visible
        return *(volatile int *)word == (int)vote_id;
    };
    const StateDev st = states[perm[k]];
    const PairLam lam = {(float)st.la, (float)st.ob};
    // the move: the launch's, or the one of this replica's state
    const MoveDev &mv = PS ? moves[perm[k]] : p.mv;
    // (read once: loaded from `moves` inside the step loop, they cost the per-state variants a register spill)
    const float m_a = mv.a, m_b = mv.b;
    const int m_steps = mv.n_steps, m_nprog = mv.n_prog;
    // (the program is interpreted: the compiler does not hoist these divisions out of the step loop; same values, same bits)
    const float h_V = mv.dt / (float)mv.nV, h_R = mv.dt / (float)mv.nR;
    float sig_i, se_i, inv_m, sigma_v;
    bool alch_i;
    auto load_atom = [&]() {
        const float4 a4 = active ? atom[a] : make_float4(1.f, 0.f, 1.f, 0.f);
        sig_i = a4.x; se_i = a4.y; inv_m = a4.z; alch_i = a4.w != 0.f;
        sigma_v = sqrtf((float)st.kT * inv_m);  // sqrt(kT/m), integrators.py:1314
    };
    load_atom();
    float4 x4 = active ? pos[(size_t)r * p.N + a] : make_float4(0, 0, 0, 0);
    float4 v4 = active ? vel[(size_t)r * p.N + a] : make_float4(0, 0, 0, 0);
    float x = x4.x, y = x4.y, z = x4.z, vx = v4.x, vy = v4.y, vz = v4.z;
    if (mv.reassign && active) {  // context.setVelocitiesToTemperature, mcmc.py:711
        const float3 g = philox_normal3(philox4x32_10(make_uint4(a, 0x80000000u, k, iteration), key));
        vx = sigma_v * g.x; vy = sigma_v * g.y; vz = sigma_v * g.z;
    }
    for (int j = t; j < p.N; j += nthr) {   // parameter records of ALL atoms (the pair loop reads those of its partners)
        const float4 a4 = atom[j];
        s_par[j] = make_float4(a4.y, a4.w != 0.f ? 1.f : 0.f, 0.f, 0.f);
    }
    if (CL > 1) cg::this_cluster().sync();   // every block of the cluster is resident and has cleared its vote words
    float fx = 0, fy = 0, fz = 0;
    bool f_valid = false;
    const float hx0 = (float)st.ho_x0[0], hx1 = (float)st.ho_x0[1], hx2 = (float)st.ho_x0[2], hK = (float)st.ho_K;
    const bool lj = p.kind != RX_SYSTEM_HARMONIC;

    bool use_list = lj && p.maxnb > 0;
    bool have_list = false;        // an outer list exists
    int n_all = 0, n_inner = 0;
    float xi = x, yi = y, zi = z;  // position at the last partition
    int cur = 1;                   // position buffer of the latest force evaluation (0: s_dyn, 1: s_dyn + 2*MAX)
    const unsigned dyn_base = (unsigned)__cvta_generic_to_shared(s_dyn);
    const unsigned nb_t = (unsigned)__cvta_generic_to_shared(s_nb + t);
    const unsigned stride = 2u * (unsigned)nthr;

    // Deal the atoms to the threads again, sorted by (inner neighbour count, atom's previous thread): a stable
    // counting sort through scratch space in the (dead) list area.
    auto reassign_atoms = [&](const float4 *s_pos) {
        const int nw = nthr >> 5, lane = t & 31, w = t >> 5;
        float4 *x_v = (float4 *)s_nb;                                // [nthr] velocities by atom id
        unsigned short *x_order = (unsigned short *)(x_v + nthr);    // [nthr] atom of each new thread
        unsigned short *x_cnt = x_order + nthr;                      // [nw][BINS] per-warp bin counts -> offsets
        unsigned short *x_base = x_cnt + nw * RX_SORT_BINS;          // [BINS] bin totals -> bases
        const int bin = active ? min(n_inner, RX_SORT_BINS - 2) : RX_SORT_BINS - 1;
        __syncthreads();  // every thread is done with its column (a partition may just have run)
        for (int q = t; q < nw * RX_SORT_BINS; q += nthr) x_cnt[q] = 0;
        x_v[a - a_base] = make_float4(vx, vy, vz, 0.f);
        __syncthreads();
        const unsigned m = __match_any_sync(0xffffffffu, bin);
        if (lane == __ffs(m) - 1) x_cnt[w * RX_SORT_BINS + bin] = (unsigned short)__popc(m);
        __syncthreads();
        for (int b = t; b < RX_SORT_BINS; b += nthr) {
            int run = 0;
            for (int q = 0; q < nw; q++) { const int c = x_cnt[q * RX_SORT_BINS + b]; x_cnt[q * RX_SORT_BINS + b] = (unsigned short)run; run += c; }
            x_base[b] = (unsigned short)run;
        }
        __syncthreads();
        if (t == 0) {
            int run = 0;
            for (int b = 0; b < RX_SORT_BINS; b++) { const int c = x_base[b]; x_base[b] = (unsigned short)run; run += c; }
        }
        __syncthreads();
        const int rank = x_base[bin] + x_cnt[w * RX_SORT_BINS + bin] + __popc(m & ((1u << lane) - 1u));
        x_order[rank] = (unsigned short)a;
        __syncthreads();
        a = x_order[t];
        const float4 vv = x_v[a - a_base];
        vx = vv.x; vy = vv.y; vz = vv.z;
        load_atom();
        if (active) { const float4 pa = s_pos[a]; x = pa.x; y = pa.y; z = pa.z; }
        __syncthreads();  // the scratch is dead: the list may be written
    };
    // Move the outer entries with r < cutoff + skin_in to the front of the column (every entry is tested once).
    auto partition = [&](const float4 *s_pos) {
        int lo = 0, hi = n_all - 1;
        if (active) {
            while (lo <= hi) {
                const unsigned ql = nb_t + (unsigned)lo * stride;
                const unsigned e = lds_u16(ql);
                const float4 pj = s_pos[e];
                const float dx = min_image_f(x - pj.x, p.Lx, p.iLx), dy = min_image_f(y - pj.y, p.Ly, p.iLy),
                            dz = min_image_f(z - pj.z, p.Lz, p.iLz);
                if (dx * dx + dy * dy + dz * dz < p.rin2) lo++;
                else {
                    const unsigned qh = nb_t + (unsigned)hi * stride;
                    sts_u16(ql, lds_u16(qh));
                    sts_u16(qh, e);
                    hi--;
                }
            }
        }
        n_inner = lo;
        xi = x; yi = y; zi = z;
    };
    auto build_outer = [&](const float4 *s_pos) {
        if (p.sort_atoms) reassign_atoms(s_pos);
        int cnt = 0;
        if (active) {
            for (int j = 0; j < p.N; j++) {
                const float4 pj = s_pos[j];
                const float dx = min_image_f(x - pj.x, p.Lx, p.iLx), dy = min_image_f(y - pj.y, p.Ly, p.iLy),
                            dz = min_image_f(z - pj.z, p.Lz, p.iLz);
                const float r2 = dx * dx + dy * dy + dz * dz;
                if (r2 < p.rl2 && j != a) {
                    if (cnt < p.maxnb) s_nb[cnt * nthr + t] = (unsigned short)j;
                    cnt++;
                }
            }
        }
        s_ref[t] = make_float4(x, y, z, 0.f);
        n_all = cnt;
        have_list = true;
        if (cluster_or(cnt > p.maxnb)) use_list = false;  // denser than the capacity: all-pairs from now on (the whole cluster)
    };
    // Make the list valid for the positions in buffer s_pos (all threads call this together).
    auto refresh_list = [&](const float4 *s_pos) {
        const float4 rf = s_ref[t];
        const float mx = x - rf.x, my = y - rf.y, mz = z - rf.z;
        const bool far = !have_list || (active && mx * mx + my * my + mz * mz > p.half_out2);
        if (cluster_or(far)) {
            const bool first = !have_list;
            build_outer(s_pos);
            if (use_list) partition(s_pos);
            if (first && p.sort_atoms && use_list) {  // the first build only counted neighbours for the sort
                build_outer(s_pos);
                if (use_list) partition(s_pos);
            }
        } else {
            partition(s_pos);
        }
    };

    PairCtx pc;
    pc.Lx = p.Lx; pc.Ly = p.Ly; pc.Lz = p.Lz; pc.iLx = p.iLx; pc.iLy = p.iLy; pc.iLz = p.iLz; pc.rc2 = p.rc2;
    pc.lam = lam;
    const int N = p.N;
    // Publish the current positions and make the neighbour list valid for them: one barrier unless a list is rebuilt.
    auto publish = [&]() {
        cur ^= 1;
        float4 *s_pos = s_dyn + (cur ? 2 * RX_MAX_ATOMS : 0);
        if (active) {
            const float4 me = make_float4(x, y, z, sig_i);
            if (CL == 1) s_pos[a] = me;
            else {
                cg::cluster_group cl = cg::this_cluster();
#pragma unroll
                for (int c = 0; c < CL; c++) cl.map_shared_rank(s_pos, c)[a] = me;
            }
        }
        const float mx = x - xi, my = y - yi, mz = z - zi;
        const bool moved = use_list && (!have_list || (active && mx * mx + my * my + mz * mz > p.half_in2));
        if (cluster_or(moved)) refresh_list(s_pos);
    };
    auto compute_forces = [&](bool want_energy, float &e_out) {
        if (!lj) {
            fx = -hK * (x - hx0); fy = -hK * (y - hx1); fz = -hK * (z - hx2);
            e_out = want_energy ? 0.5f * hK * ((x - hx0) * (x - hx0) + (y - hx1) * (y - hx1) + (z - hx2) * (z - hx2)) : 0.f;
            return;
        }
        if (!f_valid) publish();
        if (active) {
            pc.x = x; pc.y = y; pc.z = z; pc.sig_i = sig_i; pc.se_i = se_i; pc.alch_i = alch_i;
            const unsigned pos_base = dyn_base + (cur ? 2u * 16u * RX_MAX_ATOMS : 0u);
            const int par_off = cur ? -16 * RX_MAX_ATOMS : 16 * RX_MAX_ATOMS;
            if (want_energy) lj_forces<C6, SW, true>(p, pc, pos_base, par_off, nb_t, N, nthr, a, use_list, n_inner, fx, fy, fz, e_out);
            else lj_forces<C6, SW, false>(p, pc, pos_base, par_off, nb_t, N, nthr, a, use_list, n_inner, fx, fy, fz, e_out);
        } else {
            fx = fy = fz = 0.f; e_out = 0.f;
        }
    };

    uint32_t ocount = 0;
    float dummy;
    for (int s = 0; s < m_steps; s++) {
        for (int q = 0; q < m_nprog; q++) {
            const char op = mv.prog[q];
            if (op == 'V') {
                if (!f_valid) { compute_forces(false, dummy); f_valid = true; }
                const float h = h_V;
                vx += h * fx * inv_m; vy += h * fy * inv_m; vz += h * fz * inv_m;
            } else if (op == 'R') {
                const float h = h_R;
                x += h * vx; y += h * vy; z += h * vz;
                f_valid = false;
            } else {  // 'O'
                const float3 g = philox_normal3(philox4x32_10(make_uint4(a, ocount, k, iteration), key));
                ocount++;
                vx = m_a * vx + m_b * sigma_v * g.x;
                vy = m_a * vy + m_b * sigma_v * g.y;
                vz = m_a * vz + m_b * sigma_v * g.z;
            }
        }
    }
    // potential (in the replica's current state) and kinetic energy, SamplerState.potential_energy/kinetic_energy;
    // summed in atom order whatever the thread assignment is
    float e_i = 0;
    compute_forces(true, e_i);
    __syncthreads();  // the list is dead from here: its area carries the per-atom terms
    double2 *x_e = (double2 *)s_nb;
    x_e[a - a_base] = make_double2((double)e_i, active ? 0.5 * (double)(vx * vx + vy * vy + vz * vz) / (double)inv_m : 0.0);
    __syncthreads();
    const double2 et = x_e[t];
    double U = block_reduce_sum(t < n_own ? et.x : 0.0, s_red);
    double KE = block_reduce_sum(t < n_own ? et.y : 0.0, s_red);
    const bool bad = active && !(isfinite(x) && isfinite(y) && isfinite(z) && isfinite(vx) && isfinite(vy) && isfinite(vz));
    int any_bad = __syncthreads_or(bad ? 1 : 0);
    if (CL > 1) {   // block 0 of the cluster adds the partial sums in block order
        cg::cluster_group cl = cg::this_cluster();
        if (t == 0) {
            double *dst = cl.map_shared_rank(s_part, 0);
            dst[3 * q] = U; dst[3 * q + 1] = KE; dst[3 * q + 2] = any_bad ? 1.0 : 0.0;
        }
        cl.sync();
        if (q == 0 && t == 0) {
            U = 0; KE = 0; any_bad = 0;
            for (int c = 0; c < CL; c++) { U += s_part[3 * c]; KE += s_part[3 * c + 1]; any_bad |= s_part[3 * c + 2] != 0.0; }
        }
    }
    if (t == 0 && q == 0) {
        pot[k] = U + st.offset;
        kin[k] = KE;
        nan_flag[k] = (any_bad || !isfinite(U)) ? 1 : 0;
    }
    if (active) {
        if (lj) {  // getState(enforcePeriodicBox=True), mcmc.py:731
            x -= p.Lx * floorf(x * p.iLx); y -= p.Ly * floorf(y * p.iLy); z -= p.Lz * floorf(z * p.iLz);
        }
        pos[(size_t)r * p.N + a] = make_float4(x, y, z, 0.f);
        vel[(size_t)r * p.N + a] = make_float4(vx, vy, vz, 0.f);
    }
    if (CL > 1) cg::this_cluster().sync();   // no block leaves while another may still write into its shared memory
}

__global__ void k_randomize_velocities(int N, const float4 *__restrict__ atom, const StateDev *__restrict__ states,
                                       const int *__restrict__ perm, float4 *__restrict__ vel, int k0, uint2 key,
                                       uint32_t stream_id) {
    const int r = blockIdx.x, k = k0 + r;
    const StateDev st = states[perm[k]];
    for (int t = threadIdx.x; t < N; t += blockDim.x) {
        const float sv = sqrtf((float)st.kT * atom[t].z);
        const float3 g = philox_normal3(philox4x32_10(make_uint4(t, 0xC0000000u, k, stream_id), key));
        vel[(size_t)r * N + t] = make_float4(sv * g.x, sv * g.y, sv * g.z, 0.f);
    }
}

// ---------------------------------------------------------------------------------------------------
// Energy rows, double precision.
// ---------------------------------------------------------------------------------------------------
struct EnParams {
    int N, M, kind, n_alch;
    double Lx, Ly, Lz;
    double rc2, rs, rc, inv_w;
    int use_switch, annihilate, c_is_6;
    double sc_c;
    int pair_cap;
};

__device__ __forceinline__ double min_image_d(double d, double L) { return d - L * rint(d / L); }
__device__ __forceinline__ double switch_d(const EnParams &p, double r) {
    if (!p.use_switch || r <= p.rs) return 1.0;
    const double t = (r - p.rs) * p.inv_w;
    return 1.0 + t * t * t * (-10.0 + t * (15.0 - 6.0 * t));
}

__global__ void __launch_bounds__(512) k_energy_rows(EnParams p, const double4 *__restrict__ atom_d,
                                                     const int *__restrict__ alch_list,
                                                     const StateDev *__restrict__ states,
                                                     const float4 *__restrict__ pos, int k0, double2 *__restrict__ pairs,
                                                     double *__restrict__ u, int *__restrict__ err) {
    extern __shared__ double s_en[];
    double *sx = s_en, *sy = s_en + p.N, *sz = s_en + 2 * p.N;
    __shared__ double s_red[32];
    __shared__ int s_scan[32];
    __shared__ double s_U0;
    __shared__ int s_npairs;
    const int r = blockIdx.x, k = k0 + r, t = threadIdx.x, nt = blockDim.x;
    for (int q = t; q < p.N; q += nt) {
        const float4 x4 = pos[(size_t)r * p.N + q];
        sx[q] = (double)x4.x; sy[q] = (double)x4.y; sz[q] = (double)x4.z;
    }
    __syncthreads();
    double U0 = 0.0;
    if (p.kind == RX_SYSTEM_HARMONIC) {
        // u[k,l] = beta_l (sum_i K_l/2 |x_i - x0_l|^2 + offset_l)
        for (int l = t; l < p.M; l += nt) {
            const StateDev st = states[l];
            double U = 0;
            for (int i = 0; i < p.N; i++) {
                const double dx = sx[i] - st.ho_x0[0], dy = sy[i] - st.ho_x0[1], dz = sz[i] - st.ho_x0[2];
                U += 0.5 * st.ho_K * (dx * dx + dy * dy + dz * dz);
            }
            u[(size_t)k * p.M + l] = st.beta * (U + st.offset);
        }
        return;
    }
    // ---- phase 1: lambda-independent pairs (E-E, and A-A when not annihilating), half shell: i with i+1..i+N/2
    const int half = p.N / 2;
    for (int i = t; i < p.N; i += nt) {
        const double4 ai = atom_d[i];
        const bool alch_i = ai.w != 0.0;
        for (int d = 1; d <= half; d++) {
            if ((p.N % 2 == 0) && d == half && i >= half) break;  // the antipodal pair is counted once
            int j = i + d; if (j >= p.N) j -= p.N;
            const double4 aj = atom_d[j];
            const bool alch_j = aj.w != 0.0;
            const bool soft = (alch_i != alch_j) || (alch_i && alch_j && p.annihilate);
            if (soft) continue;
            const double dx = min_image_d(sx[i] - sx[j], p.Lx), dy = min_image_d(sy[i] - sy[j], p.Ly),
                         dz = min_image_d(sz[i] - sz[j], p.Lz);
            const double r2 = dx * dx + dy * dy + dz * dz;
            if (r2 >= p.rc2) continue;
            const double sig = 0.5 * (ai.x + aj.x), eps = sqrt(ai.y * aj.y);
            const double s2 = sig * sig / r2, s6 = s2 * s2 * s2;
            U0 += 4.0 * eps * (s6 * s6 - s6) * switch_d(p, sqrt(r2));
        }
    }
    const double U0_tot = block_reduce_sum(U0, s_red);
    if (t == 0) s_U0 = U0_tot;
    // ---- phase 2: lambda-controlled pairs (alchemical atom a) x (atom j), deterministic order by a stable scan
    double2 *my_pairs = pairs + (size_t)r * p.pair_cap;
    int total = 0;
    for (int pass = 0; pass < 2; pass++) {
        int cnt = 0, base = 0;
        if (pass == 1) {
            // exclusive scan of per-thread counts (warp shuffle + warp totals)
            const int lane = t & 31, w = t >> 5, nw = (nt + 31) >> 5;
            int incl = total;  // `total` holds this thread's count from pass 0
            for (int o = 1; o < 32; o <<= 1) { int n = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += n; }
            if (lane == 31) s_scan[w] = incl;
            __syncthreads();
            int woff = 0;
            for (int q = 0; q < w; q++) woff += s_scan[q];
            base = woff + incl - total;
            if (t == nt - 1) s_npairs = base + total;
            (void)nw;
        }
        for (int ai_ = 0; ai_ < p.n_alch; ai_++) {
            const int a = alch_list[ai_];
            const double4 pa = atom_d[a];
            for (int j = t; j < p.N; j += nt) {
                if (j == a) continue;
                const double4 pj = atom_d[j];
                const bool alch_j = pj.w != 0.0;
                if (alch_j && (!p.annihilate || j < a)) continue;  // A-A: only when annihilating, counted once
                const double dx = min_image_d(sx[a] - sx[j], p.Lx), dy = min_image_d(sy[a] - sy[j], p.Ly),
                             dz = min_image_d(sz[a] - sz[j], p.Lz);
                const double r2 = dx * dx + dy * dy + dz * dz;
                if (r2 >= p.rc2) continue;
                if (pass == 1) {
                    const int slot = base + cnt;
                    if (slot < p.pair_cap) {
                        const double sig = 0.5 * (pa.x + pj.x), eps = sqrt(pa.y * pj.y);
                        const double q = r2 / (sig * sig);
                        const double rsc = p.c_is_6 ? q * q * q : pow(q, 0.5 * p.sc_c);
                        my_pairs[slot] = make_double2(rsc, 4.0 * eps * switch_d(p, sqrt(r2)));
                    }
                }
                cnt++;
            }
        }
        if (pass == 0) total = cnt;
    }
    __syncthreads();
    int npairs = s_npairs;
    if (npairs > p.pair_cap) { if (t == 0) atomicExch(err, RX_ERR_CAPACITY); npairs = p.pair_cap; }
    // ---- phase 3: one state per thread, pairs summed in list order
    const double U0s = s_U0;
    for (int l = t; l < p.M; l += nt) {
        const StateDev st = states[l];
        double Ua = 0.0;
        for (int q = 0; q < npairs; q++) {
            const double2 pr = my_pairs[q];
            const double D = st.ob + pr.x;
            const double x = p.c_is_6 ? 1.0 / D : pow(D, -6.0 / p.sc_c);
            Ua += st.la * pr.y * x * (x - 1.0);
        }
        u[(size_t)k * p.M + l] = st.beta * (U0s + Ua + st.offset);
    }
}

// ---------------------------------------------------------------------------------------------------
// host <-> device conversions at the boundary (double xyz <-> float4)
// ---------------------------------------------------------------------------------------------------
__global__ void k_pack(const double *__restrict__ in, float4 *__restrict__ out, long long n) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n) out[i] = make_float4((float)in[3 * i], (float)in[3 * i + 1], (float)in[3 * i + 2], 0.f);
}
__global__ void k_unpack(const float4 *__restrict__ in, double *__restrict__ out, long long n, int wrap, double Lx,
                         double Ly, double Lz) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 v = in[i];
    double x = v.x, y = v.y, z = v.z;
    if (wrap) { x -= Lx * floor(x / Lx); y -= Ly * floor(y / Ly); z -= Lz * floor(z / Lz); }
    out[3 * i] = x; out[3 * i + 1] = y; out[3 * i + 2] = z;
}

int rxi_convert_in(rx_engine *h, float4 *dst, int first_local, int count, const double *host_xyz, bool) {
    const long long n = (long long)count * h->cfg.n_atoms;
    if (n == 0) return RX_OK;
    if (h->cfg.system_kind == RX_SYSTEM_MOLECULE) {   // the state of a molecule is kept in f64: a plain copy
        double *d = (double *)dst + (size_t)first_local * h->cfg.n_atoms * 3;
        RX_CHECK_CUDA(h, cudaMemcpyAsync(d, host_xyz, n * 3 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
        return RX_OK;
    }
    const double *src = host_xyz;
    if (!rxi_is_pinned(h, host_xyz, n * 3 * sizeof(double))) {   // pageable caller memory goes through the pinned staging buffer
        memcpy(h->h_io, host_xyz, n * 3 * sizeof(double));
        src = h->h_io;
    }
    RX_CHECK_CUDA(h, cudaMemcpyAsync(h->d_io, src, n * 3 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    k_pack<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(h->d_io, dst + (size_t)first_local * h->cfg.n_atoms, n);
    RX_CHECK_CUDA(h, cudaGetLastError());
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    return RX_OK;
}

int rxi_convert_out(rx_engine *h, const float4 *src, int first_local, int count, double *host_xyz, bool wrap) {
    const long long n = (long long)count * h->cfg.n_atoms;
    if (n == 0) return RX_OK;
    if (h->cfg.system_kind == RX_SYSTEM_MOLECULE) {
        const double *d = (const double *)src + (size_t)first_local * h->cfg.n_atoms * 3;
        RX_CHECK_CUDA(h, cudaMemcpyAsync(host_xyz, d, n * 3 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
        return RX_OK;
    }
    k_unpack<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(src + (size_t)first_local * h->cfg.n_atoms, h->d_io, n,
                                                                 wrap ? 1 : 0, h->cfg.box[0], h->cfg.box[1], h->cfg.box[2]);
    RX_CHECK_CUDA(h, cudaGetLastError());
    const bool direct = rxi_is_pinned(h, host_xyz, n * 3 * sizeof(double));
    RX_CHECK_CUDA(h, cudaMemcpyAsync(direct ? host_xyz : h->h_io, h->d_io, n * 3 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    if (!direct) memcpy(host_xyz, h->h_io, n * 3 * sizeof(double));
    return RX_OK;
}

#include "rx_molecule.cuh"

// ---------------------------------------------------------------------------------------------------
// The kernels' form of a move.
static MoveDev move_dev(const rx_state_move &m) {
    MoveDev d;
    memset(&d, 0, sizeof(d));
    for (const char *q = m.program; *q; q++) {
        if (*q == 'V') d.nV++; else if (*q == 'R') d.nR++; else d.nO++;
        d.prog[d.n_prog++] = *q;
    }
    d.dt = (float)m.dt; d.n_steps = m.n_steps; d.reassign = m.reassign;
    const double hO = m.dt / (d.nO > 0 ? d.nO : 1);   // integrators.py:1141-1146
    d.dt_d = m.dt; d.a_d = exp(-m.gamma * hO); d.b_d = sqrt(1.0 - exp(-2.0 * m.gamma * hO));
    d.a = (float)d.a_d; d.b = (float)d.b_d;
    return d;
}

static void fill_dyn(const rx_engine *h, DynParams &p) {
    const rx_config &c = h->cfg;
    memset(&p, 0, sizeof(p));
    p.N = c.n_atoms; p.kind = c.system_kind;
    p.Lx = (float)c.box[0]; p.Ly = (float)c.box[1]; p.Lz = (float)c.box[2];
    p.iLx = (float)(1.0 / c.box[0]); p.iLy = (float)(1.0 / c.box[1]); p.iLz = (float)(1.0 / c.box[2]);
    p.rc2 = (float)(c.r_cutoff * c.r_cutoff); p.rs2 = (float)(c.r_switch * c.r_switch); p.rs = (float)c.r_switch;
    p.inv_w = (float)(1.0 / (c.r_cutoff - c.r_switch));
    p.use_switch = c.use_switch; p.annihilate = c.annihilate_sterics;
    p.c_is_6 = (c.softcore_c == 6.0); p.sc_c = (float)c.softcore_c;
    p.mv = move_dev(h->move);
}

// The per-state move table (rx_set_state_integrator), uploaded when it changed.
int rxi_upload_state_moves(rx_engine *h) {
    if (!h->state_moves_dirty) return RX_OK;
    const int M = h->cfg.n_states;
    std::vector<MoveDev> tab((size_t)M);
    for (int l = 0; l < M; l++) tab[(size_t)l] = move_dev(h->state_moves[(size_t)l]);
    if (!h->d_moves) RX_CHECK_CUDA(h, cudaMalloc(&h->d_moves, sizeof(MoveDev) * (size_t)M));
    RX_CHECK_CUDA(h, cudaMemcpyAsync(h->d_moves, tab.data(), sizeof(MoveDev) * (size_t)M, cudaMemcpyHostToDevice, h->stream));
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));   // (tab is a stack object)
    h->state_moves_dirty = false;
    return RX_OK;
}

// How k_propagate runs for a particle system: the launch shape and the neighbour-list geometry of DynParams.
struct PropPlan {
    int cl;          // blocks per replica (one thread-block cluster): 1 or 4
    int threads;     // per block: one thread per atom of the block, whole warps
    size_t smem;     // dynamic shared memory per block
    int maxnb, sort_atoms;
    float rl2, rin2, half_in2, half_out2;
};

static PropPlan prop_plan(const rx_engine *h) {
    const rx_config &c = h->cfg;
    const int N = c.n_atoms;
    const bool lj = c.system_kind == RX_SYSTEM_LJ_ALCH;
    PropPlan pl = {};
    // Measured on the 512-atom fluid (500 steps, in the iteration loop, profiles/r2_cluster_propagate.txt): 32 replicas
    // 2.27-2.36 ms in one block, 2.20-2.29 in a cluster of four; 64 replicas 2.28-2.37 / 2.31-2.39.  A block of 128 threads
    // leaves ONE warp per scheduler, which runs the step's ~1100 dependent instructions no faster than four warps sharing a
    // scheduler do: the split only pays for the few replicas that would otherwise leave three quarters of the GPU idle, so
    // that is the only case it is chosen for.  Per-state moves have no cluster variant.
    pl.cl = (lj && N >= 256 && h->kloc * 4 <= h->n_sms && h->state_moves.empty()) ? 4 : 1;
    pl.threads = ((N + pl.cl - 1) / pl.cl + 31) / 32 * 32;
    pl.rl2 = pl.rin2 = (float)(c.r_cutoff * c.r_cutoff);
    // shared memory: two position buffers + the parameter records + per-thread reference positions + the list area
    const size_t atoms_bytes = (size_t)3 * RX_MAX_ATOMS * sizeof(float4) + (size_t)pl.threads * sizeof(float4);
    size_t area = (size_t)pl.threads * sizeof(double2);  // the list area doubles as scratch for the final reductions
    if (lj && N >= 64 && !getenv("RX_NO_VERLET")) {
        // Dual neighbour list: outer skin 0.40 nm (at 300 K and 10/ps friction the all-pairs build usually lasts a
        // whole 500-step launch), inner skin 0.05 nm (a re-partition of the column about every 25 steps; both tuned
        // on the 512-atom fluid, see profiles/prop_r1_v6.summary.txt).  Capacity from the
        // shared-memory budget (two CTAs per SM up to 512 atoms); denser systems fall back to all-pairs in the kernel.
        double skin_in = 0.05;
        double rl = c.r_cutoff + 0.40;
        for (int d = 0; d < 3; d++) if (rl > 0.5 * c.box[d]) rl = 0.5 * c.box[d];
        const double eff_out = rl - c.r_cutoff;
        if (skin_in > eff_out / 3.0) skin_in = eff_out / 3.0;
        if (eff_out > 0.03) {
            const size_t budget = (pl.threads > 512 ? 200 : 112) * 1024;
            int cap = (int)((budget - atoms_bytes) / ((size_t)pl.threads * sizeof(unsigned short)));
            if (cap > 128) cap = 128;
            if (cap >= 8) {
                pl.maxnb = cap;
                pl.rl2 = (float)(rl * rl);
                pl.rin2 = (float)((c.r_cutoff + skin_in) * (c.r_cutoff + skin_in));
                pl.half_in2 = (float)(0.25 * skin_in * skin_in);
                pl.half_out2 = (float)(0.25 * (eff_out - skin_in) * (eff_out - skin_in));
                const size_t list_bytes = (((size_t)cap * pl.threads * sizeof(unsigned short)) + 15) / 16 * 16;
                // scratch of the atom re-assignment: velocities, order, per-warp bin counts, bin bases
                const size_t sort_bytes = (size_t)pl.threads * (sizeof(float4) + 2) + (size_t)(pl.threads / 32 + 1) * RX_SORT_BINS * 2;
                pl.sort_atoms = list_bytes >= sort_bytes ? 1 : 0;
                if (list_bytes > area) area = list_bytes;
            }
        }
    }
    pl.smem = atoms_bytes + area;
    return pl;
}

// Calls f(C6, SW) -- std::integral_constant<bool, ...> arguments -- with the pair-function specialisation of the engine.
template <class F>
static int with_pair_kind(const DynParams &p, F &&f) {
    using T = std::true_type;
    using U = std::false_type;
    if (p.c_is_6) return p.use_switch ? f(T(), T()) : f(T(), U());
    return p.use_switch ? f(U(), T()) : f(U(), U());
}

template <bool C6, bool SW, int CL, bool PS>
static int launch_propagate(rx_engine *h, const PropPlan &pl, const DynParams &p, uint2 key, uint32_t iteration,
                            const int *d_only) {
    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3((unsigned)(h->kloc * CL));
    lc.blockDim = dim3((unsigned)pl.threads);
    lc.dynamicSmemBytes = pl.smem;
    lc.stream = h->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    lc.attrs = at;
    lc.numAttrs = 1;
    if (pl.smem > 48 * 1024)
        RX_CHECK_CUDA(h, cudaFuncSetAttribute(k_propagate<C6, SW, CL, PS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
    RX_CHECK_CUDA(h, cudaLaunchKernelEx(&lc, k_propagate<C6, SW, CL, PS>, p, (const float4 *)h->d_atom, (const StateDev *)h->d_states,
                                        (const int *)h->d_perm, h->d_pos, h->d_vel, h->k0, key, iteration, h->d_pot, h->d_kin,
                                        h->d_nan, d_only, (const MoveDev *)h->d_moves));
    return RX_OK;
}

int rxi_propagate(rx_engine *h, uint64_t seed, uint64_t iteration, int reassign, int *launches, const int *d_only) {
    if (h->kloc == 0) return RX_OK;
    DynParams p;
    fill_dyn(h, p);
    const int N = h->cfg.n_atoms;
    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32) ^ (uint32_t)(iteration >> 32));
    if (h->cfg.system_kind == RX_SYSTEM_MOLECULE) {
        if (!h->state_moves.empty()) RX_FAIL(h, RX_ERR_UNSUPPORTED, "rx_propagate: per-state moves are not provided for molecules");
        const MolDev *md = (const MolDev *)h->mol_dev;
        const bool no_star = getenv("RX_MOL_NO_STAR") != nullptr;   // cross-check: the general cluster path for every molecule
        auto kern = (md->max_cluster <= 3 && !no_star) ? k_propagate_mol<true> : k_propagate_mol<false>;
        kern<<<h->kloc, 32 * MOL_WARPS, md->dyn_shared_bytes, h->stream>>>(*md, p, (const StateDev *)h->d_states, (const int *)h->d_perm, (double *)h->d_pos,
                                                                           (double *)h->d_vel, h->k0, key, (uint32_t)iteration, reassign, h->d_pot,
                                                                           h->d_kin, h->d_nan, d_only);
        RX_CHECK_CUDA(h, cudaGetLastError());
        (*launches)++;
        return RX_OK;
    }
    if (N > 1024) RX_FAIL(h, RX_ERR_UNSUPPORTED, "rx_propagate: more than 1024 atoms per replica is not supported yet");
    const bool per_state = !h->state_moves.empty();
    int rc = per_state ? rxi_upload_state_moves(h) : RX_OK;
    if (rc) return rc;
    const PropPlan pl = prop_plan(h);
    p.maxnb = pl.maxnb; p.sort_atoms = pl.sort_atoms;
    p.rl2 = pl.rl2; p.rin2 = pl.rin2; p.half_in2 = pl.half_in2; p.half_out2 = pl.half_out2;
    p.mv.reassign = reassign;
    const uint32_t it32 = (uint32_t)iteration;
    rc = with_pair_kind(p, [&](auto c6, auto sw) -> int {
        constexpr bool C6 = decltype(c6)::value, SW = decltype(sw)::value;
        if (per_state) return launch_propagate<C6, SW, 1, true>(h, pl, p, key, it32, d_only);
        if (pl.cl == 4) return launch_propagate<C6, SW, 4, false>(h, pl, p, key, it32, d_only);
        return launch_propagate<C6, SW, 1, false>(h, pl, p, key, it32, d_only);
    });
    if (rc) return rc;
    RX_CHECK_CUDA(h, cudaGetLastError());
    (*launches)++;
    return RX_OK;
}

// Start-of-iteration snapshot of positions and velocities (the restart policy of mcmc.py:706-759 retries a failed replica
// from the state it had when the move began) and the restore of the replicas whose NaN flag is set.
int rxi_snapshot_state(rx_engine *h) {
    if (h->kloc == 0) return RX_OK;
    const size_t bytes = (h->cfg.system_kind == RX_SYSTEM_MOLECULE ? 3 * sizeof(double) : sizeof(float4)) * (size_t)h->kloc * h->cfg.n_atoms;
    if (!h->d_pos_snap) {
        RX_CHECK_CUDA(h, cudaMalloc(&h->d_pos_snap, bytes));
        RX_CHECK_CUDA(h, cudaMalloc(&h->d_vel_snap, bytes));
        RX_CHECK_CUDA(h, cudaMalloc(&h->d_retry, sizeof(int) * h->cfg.n_replicas));
    }
    RX_CHECK_CUDA(h, cudaMemcpyAsync(h->d_pos_snap, h->d_pos, bytes, cudaMemcpyDeviceToDevice, h->stream));
    RX_CHECK_CUDA(h, cudaMemcpyAsync(h->d_vel_snap, h->d_vel, bytes, cudaMemcpyDeviceToDevice, h->stream));
    h->have_snapshot = true;
    return RX_OK;
}

__global__ void k_restore_failed(const int *__restrict__ nan_flag, int *__restrict__ retry, int k0, int N,
                                 const float4 *__restrict__ pos_snap, const float4 *__restrict__ vel_snap,
                                 float4 *__restrict__ pos, float4 *__restrict__ vel) {
    const int r = blockIdx.x, k = k0 + r;
    const int failed = nan_flag[k];
    if (threadIdx.x == 0) retry[k] = failed;
    if (!failed) return;
    for (int t = threadIdx.x; t < N; t += blockDim.x) {
        pos[(size_t)r * N + t] = pos_snap[(size_t)r * N + t];
        vel[(size_t)r * N + t] = vel_snap[(size_t)r * N + t];
    }
}

int rxi_restore_failed(rx_engine *h) {
    if (h->kloc == 0) return RX_OK;
    if (!h->have_snapshot) RX_FAIL(h, RX_ERR_INVALID, "rx_propagate_retry: no start-of-iteration snapshot (call rx_propagate first)");
    if (h->cfg.system_kind == RX_SYSTEM_MOLECULE) {
        k_restore_failed_mol<<<h->kloc, 32, 0, h->stream>>>(h->d_nan, h->d_retry, h->k0, h->cfg.n_atoms, (const double *)h->d_pos_snap,
                                                           (const double *)h->d_vel_snap, (double *)h->d_pos, (double *)h->d_vel);
        RX_CHECK_CUDA(h, cudaGetLastError());
        return RX_OK;
    }
    k_restore_failed<<<h->kloc, 256, 0, h->stream>>>(h->d_nan, h->d_retry, h->k0, h->cfg.n_atoms, h->d_pos_snap, h->d_vel_snap,
                                                    h->d_pos, h->d_vel);
    RX_CHECK_CUDA(h, cudaGetLastError());
    return RX_OK;
}

// ---------------------------------------------------------------------------------------------------
// Energy minimisation of every owned replica in its current state: MultiStateSampler.minimize
// (multistatesampler.py:612-647) -> _minimize_replica (:1339-1402), which runs a FIRE descent first
// (integrators.py FIREMinimizationIntegrator).  FIRE as published (Bitzek et al., PRL 97, 170201 (2006)):
// semi-implicit Euler dynamics with the velocity steered towards the force, the time step grown while the power
// F.v stays positive and the motion stopped when it turns negative; plus a cap on the displacement per step so the
// overlapping starts of the reference's test systems cannot blow up.  One CTA per replica, one atom per thread,
// all-pairs forces (this is a set-up step, not the hot path).  Velocities are left untouched.
// ---------------------------------------------------------------------------------------------------
template <bool C6, bool SW>
__global__ void __launch_bounds__(1024) k_minimize(DynParams p, const float4 *__restrict__ atom,
                                                   const StateDev *__restrict__ states, const int *__restrict__ perm,
                                                   float4 *__restrict__ pos, int k0, float tol_rms, int max_iter,
                                                   double *__restrict__ rms_out, int *__restrict__ iters_out) {
    extern __shared__ float4 s_dyn[];
    float4 *s_pos = s_dyn, *s_par = s_dyn + RX_MAX_ATOMS;
    __shared__ float s_part[32][3];
    __shared__ float s_sum[3];
    const int r = blockIdx.x, k = k0 + r, t = threadIdx.x, nw = blockDim.x >> 5;
    const bool active = t < p.N;
    const StateDev st = states[perm[k]];
    const float4 a4 = active ? atom[t] : make_float4(1.f, 0.f, 1.f, 0.f);
    const float sig_i = a4.x, se_i = a4.y, inv_m = a4.z;
    const bool alch_i = a4.w != 0.f;
    const float4 x4 = active ? pos[(size_t)r * p.N + t] : make_float4(0, 0, 0, 0);
    float x = x4.x, y = x4.y, z = x4.z, vx = 0.f, vy = 0.f, vz = 0.f;
    if (active) { s_pos[t] = make_float4(x, y, z, sig_i); s_par[t] = make_float4(se_i, alch_i ? 1.f : 0.f, 0.f, 0.f); }
    __syncthreads();
    PairCtx pc;
    pc.Lx = p.Lx; pc.Ly = p.Ly; pc.Lz = p.Lz; pc.iLx = p.iLx; pc.iLy = p.iLy; pc.iLz = p.iLz; pc.rc2 = p.rc2;
    pc.sig_i = sig_i; pc.se_i = se_i; pc.alch_i = alch_i; pc.lam = {(float)st.la, (float)st.ob};
    const unsigned pos_base = (unsigned)__cvta_generic_to_shared(s_dyn);
    const float hx0 = (float)st.ho_x0[0], hx1 = (float)st.ho_x0[1], hx2 = (float)st.ho_x0[2], hK = (float)st.ho_K;
    const float dt0 = 0.001f, dt_max = 0.010f, alpha0 = 0.1f, max_move = 0.01f;  // ps, ps, -, nm per step
    float dt = dt0, alpha = alpha0;
    int n_pos = 0, it = 0;
    float rms = 0.f;
    for (;;) {
        float fx = 0.f, fy = 0.f, fz = 0.f, e = 0.f;
        if (p.kind == RX_SYSTEM_HARMONIC) { fx = -hK * (x - hx0); fy = -hK * (y - hx1); fz = -hK * (z - hx2); }
        else if (active) {
            pc.x = x; pc.y = y; pc.z = z;
            lj_forces<C6, SW, false>(p, pc, pos_base, 16 * RX_MAX_ATOMS, 0u, p.N, p.N, t, false, 0, fx, fy, fz, e);
        }
        if (!active) { fx = fy = fz = 0.f; }
        // block sums of F.F, F.v, v.v (fixed order: deterministic)
        float q0 = fx * fx + fy * fy + fz * fz, q1 = fx * vx + fy * vy + fz * vz, q2 = vx * vx + vy * vy + vz * vz;
        for (int o = 16; o > 0; o >>= 1) {
            q0 += __shfl_down_sync(0xffffffffu, q0, o); q1 += __shfl_down_sync(0xffffffffu, q1, o); q2 += __shfl_down_sync(0xffffffffu, q2, o);
        }
        if ((t & 31) == 0) { s_part[t >> 5][0] = q0; s_part[t >> 5][1] = q1; s_part[t >> 5][2] = q2; }
        __syncthreads();  // also: every thread has finished reading the positions
        if (t < 3) { float s = 0.f; for (int w = 0; w < nw; w++) s += s_part[w][t]; s_sum[t] = s; }
        __syncthreads();
        const float FF = s_sum[0], P = s_sum[1], VV = s_sum[2];
        rms = sqrtf(FF / (3.0f * (float)p.N));
        if (!(rms > tol_rms) || it >= max_iter) break;  // converged, out of iterations, or NaN
        it++;
        if (P > 0.f) {
            const float mix = alpha * sqrtf(VV / fmaxf(FF, 1e-30f));
            vx = (1.f - alpha) * vx + mix * fx; vy = (1.f - alpha) * vy + mix * fy; vz = (1.f - alpha) * vz + mix * fz;
            if (++n_pos > 5) { dt = fminf(dt * 1.1f, dt_max); alpha *= 0.99f; }
        } else {
            vx = vy = vz = 0.f; dt *= 0.5f; alpha = alpha0; n_pos = 0;
        }
        vx += dt * fx * inv_m; vy += dt * fy * inv_m; vz += dt * fz * inv_m;
        float mx = dt * vx, my = dt * vy, mz = dt * vz;
        const float m2 = mx * mx + my * my + mz * mz;
        if (m2 > max_move * max_move) {  // displacement cap: rescale this atom's velocity
            const float sc = max_move * rsqrtf(m2);
            vx *= sc; vy *= sc; vz *= sc; mx *= sc; my *= sc; mz *= sc;
        }
        x += mx; y += my; z += mz;
        if (active) s_pos[t] = make_float4(x, y, z, sig_i);
        __syncthreads();
    }
    if (t == 0) { rms_out[k] = (double)rms; iters_out[k] = it; }
    if (active) {
        if (p.kind != RX_SYSTEM_HARMONIC) { x -= p.Lx * floorf(x * p.iLx); y -= p.Ly * floorf(y * p.iLy); z -= p.Lz * floorf(z * p.iLz); }
        pos[(size_t)r * p.N + t] = make_float4(x, y, z, 0.f);
    }
}

int rxi_minimize(rx_engine *h, double tolerance, int max_iterations, double *d_rms, int *d_iters) {
    if (h->kloc == 0) return RX_OK;
    if (h->cfg.system_kind == RX_SYSTEM_MOLECULE) {
        const MolDev *m = (const MolDev *)h->mol_dev;
        k_minimize_mol<<<h->kloc, 32, m->shared_bytes, h->stream>>>(*m, (double *)h->d_pos, h->k0, tolerance,
                                                                   max_iterations > 0 ? max_iterations : 100000, d_rms, d_iters);
        RX_CHECK_CUDA(h, cudaGetLastError());
        return RX_OK;
    }
    DynParams p;
    fill_dyn(h, p);
    const int N = h->cfg.n_atoms;
    if (N > 1024) RX_FAIL(h, RX_ERR_UNSUPPORTED, "rx_minimize: more than 1024 atoms per replica is not supported yet");
    const int threads = ((N + 31) / 32) * 32;
    const size_t smem = (size_t)2 * RX_MAX_ATOMS * sizeof(float4);
    return with_pair_kind(p, [&](auto c6, auto sw) -> int {
        k_minimize<decltype(c6)::value, decltype(sw)::value><<<h->kloc, threads, smem, h->stream>>>(
            p, h->d_atom, h->d_states, h->d_perm, h->d_pos, h->k0, (float)tolerance, max_iterations, d_rms, d_iters);
        RX_CHECK_CUDA(h, cudaGetLastError());
        return RX_OK;
    });
}

int rxi_randomize_velocities(rx_engine *h, uint64_t seed, uint64_t stream_id) {
    if (h->kloc == 0) return RX_OK;
    const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
    if (h->cfg.system_kind == RX_SYSTEM_MOLECULE) {   // (k_propagate_mol projects incoming velocities onto the constraints)
        k_randomize_velocities_mol<<<h->kloc, 32, 0, h->stream>>>(*(const MolDev *)h->mol_dev, (const StateDev *)h->d_states,
                                                                 (const int *)h->d_perm, (double *)h->d_vel, h->k0, key, (uint32_t)stream_id);
        RX_CHECK_CUDA(h, cudaGetLastError());
        RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
        return RX_OK;
    }
    k_randomize_velocities<<<h->kloc, 256, 0, h->stream>>>(h->cfg.n_atoms, h->d_atom, h->d_states, h->d_perm, h->d_vel, h->k0,
                                                           key, (uint32_t)stream_id);
    RX_CHECK_CUDA(h, cudaGetLastError());
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    return RX_OK;
}

// Energy rows of the owned replicas at `n_states` states described by the device table `d_states`, written to
// d_out[K][n_states] (rows [k0, k0+kloc)).  The resident table/matrix are the default.
int rxi_compute_energy_rows_at(rx_engine *h, const StateDev *d_states, int n_states, double *d_out, int *launches) {
    if (h->kloc == 0) return RX_OK;
    const rx_config &c = h->cfg;
    if (c.system_kind == RX_SYSTEM_MOLECULE) {
        k_energy_mol<<<h->kloc, 32, ((const MolDev *)h->mol_dev)->shared_bytes, h->stream>>>(*(const MolDev *)h->mol_dev, d_states, n_states, (const double *)h->d_pos, h->k0, d_out);
        RX_CHECK_CUDA(h, cudaGetLastError());
        (*launches)++;
        return RX_OK;
    }
    EnParams p;
    memset(&p, 0, sizeof(p));
    p.N = c.n_atoms; p.M = n_states; p.kind = c.system_kind; p.n_alch = h->n_alch;
    p.Lx = c.box[0]; p.Ly = c.box[1]; p.Lz = c.box[2];
    p.rc2 = c.r_cutoff * c.r_cutoff; p.rs = c.r_switch; p.rc = c.r_cutoff;
    p.inv_w = 1.0 / (c.r_cutoff - c.r_switch);
    p.use_switch = c.use_switch; p.annihilate = c.annihilate_sterics;
    p.c_is_6 = (c.softcore_c == 6.0); p.sc_c = c.softcore_c;
    p.pair_cap = h->pair_cap;
    const size_t smem = (size_t)3 * c.n_atoms * sizeof(double);
    if (smem > 48 * 1024) RX_CHECK_CUDA(h, cudaFuncSetAttribute(k_energy_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_energy_rows<<<h->kloc, 512, smem, h->stream>>>(p, h->d_atom_d, h->d_alch_list, d_states, h->d_pos, h->k0,
                                                    (double2 *)h->d_pairs, d_out, h->d_err);
    RX_CHECK_CUDA(h, cudaGetLastError());
    (*launches)++;
    return RX_OK;
}

int rxi_compute_energy_rows(rx_engine *h, int *launches) {
    return rxi_compute_energy_rows_at(h, h->d_states, h->cfg.n_states, h->d_u, launches);
}


// ---------------------------------------------------------------------------------------------------
// Molecule tables (rx_set_molecule): per-atom term lists, the pair mask, constraint clusters.
// ---------------------------------------------------------------------------------------------------
template <typename T>
static int mol_upload(rx_engine *h, const std::vector<T> &v, const T **out) {
    void *d = nullptr;
    // (+16: the kernels stage these tables into shared memory in 8-byte pieces and may read up to the next multiple of 8)
    const size_t bytes = sizeof(T) * (v.empty() ? 1 : v.size()) + 16;
    RX_CHECK_CUDA(h, cudaMalloc(&d, bytes));
    RX_CHECK_CUDA(h, cudaMemset(d, 0, bytes));
    if (!v.empty()) RX_CHECK_CUDA(h, cudaMemcpy(d, v.data(), sizeof(T) * v.size(), cudaMemcpyHostToDevice));
    h->mol_allocs.push_back(d);
    *out = (const T *)d;
    return RX_OK;
}

int rxi_set_molecule(rx_engine *h, const rx_molecule *mol) {
    const int n = h->cfg.n_atoms;
    if (n > MOL_MAX_ATOMS) RX_FAIL(h, RX_ERR_UNSUPPORTED, "rx_set_molecule: more than 32 atoms per molecule is not provided");
    if (!mol->mass || !mol->charge || !mol->sigma || !mol->epsilon) RX_FAIL(h, RX_ERR_INVALID, "rx_set_molecule: null per-atom arrays");
    auto atom_ok = [&](double v) { return v >= 0 && v < n && v == floor(v); };
    for (void *d : h->mol_allocs) cudaFree(d);
    h->mol_allocs.clear();
    std::vector<double> mass(mol->mass, mol->mass + n), charge(mol->charge, mol->charge + n), sigma(mol->sigma, mol->sigma + n),
        eps(mol->epsilon, mol->epsilon + n);
    for (int i = 0; i < n; i++)
        if (!(mass[i] > 0) || !(sigma[i] > 0) || eps[i] < 0) RX_FAIL(h, RX_ERR_INVALID, "rx_set_molecule: need mass > 0, sigma > 0, epsilon >= 0");
    std::vector<std::vector<MolBond>> ba(n);
    std::vector<std::vector<MolAngle>> aa(n);
    std::vector<std::vector<MolTorsion>> ta(n);
    std::vector<std::vector<MolExc>> xa(n);
    std::vector<unsigned> mask(n);
    for (int i = 0; i < n; i++) mask[i] = (n == 32 ? 0xffffffffu : ((1u << n) - 1u)) & ~(1u << i);
    for (int b = 0; b < mol->n_bonds; b++) {
        const double *q = mol->bonds + 4 * b;
        if (!atom_ok(q[0]) || !atom_ok(q[1]) || q[0] == q[1]) RX_FAIL(h, RX_ERR_INVALID, "rx_set_molecule: bad bond");
        const int i = (int)q[0], j = (int)q[1];
        ba[i].push_back(MolBond{j, 0, q[2], q[3]});
        ba[j].push_back(MolBond{i, 0, q[2], q[3]});
    }
    for (int a = 0; a < mol->n_angles; a++) {
        const double *q = mol->angles + 5 * a;
        if (!atom_ok(q[0]) || !atom_ok(q[1]) || !atom_ok(q[2])) RX_FAIL(h, RX_ERR_INVALID, "rx_set_molecule: bad angle");
        const int id[3] = {(int)q[0], (int)q[1], (int)q[2]};
        for (int role = 0; role < 3; role++) aa[id[role]].push_back(MolAngle{id[0], id[1], id[2], role, q[3], q[4]});
    }
    for (int t = 0; t < mol->n_torsions; t++) {
        const double *q = mol->torsions + 7 * t;
        if (!atom_ok(q[0]) || !atom_ok(q[1]) || !atom_ok(q[2]) || !atom_ok(q[3])) RX_FAIL(h, RX_ERR_INVALID, "rx_set_molecule: bad torsion");
        const int id[4] = {(int)q[0], (int)q[1], (int)q[2], (int)q[3]};
        for (int role = 0; role < 4; role++) ta[id[role]].push_back(MolTorsion{id[0], id[1], id[2], id[3], (int)q[4], role, q[5], q[6]});
    }
    for (int e = 0; e < mol->n_exclusions; e++) {
        const int64_t i = mol->exclusions[2 * e], j = mol->exclusions[2 * e + 1];
        if (i < 0 || i >= n || j < 0 || j >= n || i == j) RX_FAIL(h, RX_ERR_INVALID, "rx_set_molecule: bad exclusion");
        mask[i] &= ~(1u << j); mask[j] &= ~(1u << i);
    }
    for (int e = 0; e < mol->n_exceptions; e++) {
        const double *q = mol->exceptions + 5 * e;
        if (!atom_ok(q[0]) || !atom_ok(q[1]) || q[0] == q[1]) RX_FAIL(h, RX_ERR_INVALID, "rx_set_molecule: bad exception");
        const int i = (int)q[0], j = (int)q[1];
        mask[i] &= ~(1u << j); mask[j] &= ~(1u << i);
        xa[i].push_back(MolExc{j, 0, q[2], q[3], q[4]});
        xa[j].push_back(MolExc{i, 0, q[2], q[3], q[4]});
    }
    // constraint clusters: connected components, constraints kept in list order inside a cluster
    std::vector<int> comp(n);
    for (int i = 0; i < n; i++) comp[i] = i;
    auto find = [&](int x) { while (comp[x] != x) x = comp[x] = comp[comp[x]]; return x; };
    for (int c = 0; c < mol->n_constraints; c++) {
        const double *q = mol->constraints + 3 * c;
        if (!atom_ok(q[0]) || !atom_ok(q[1]) || q[0] == q[1] || !(q[2] > 0)) RX_FAIL(h, RX_ERR_INVALID, "rx_set_molecule: bad constraint");
        comp[find((int)q[0])] = find((int)q[1]);
    }
    std::vector<int> cluster_of(n, -1), c_off(1, 0);
    std::vector<std::vector<MolCons>> cl;
    for (int c = 0; c < mol->n_constraints; c++) {
        const double *q = mol->constraints + 3 * c;
        const int root = find((int)q[0]);
        if (cluster_of[root] < 0) { cluster_of[root] = (int)cl.size(); cl.emplace_back(); }
        cl[cluster_of[root]].push_back(MolCons{(int)q[0], (int)q[1], q[2]});
    }
    if ((int)cl.size() > 32) RX_FAIL(h, RX_ERR_UNSUPPORTED, "rx_set_molecule: more than 32 constraint clusters");
    std::vector<MolCons> cons;
    for (auto &c : cl) { cons.insert(cons.end(), c.begin(), c.end()); c_off.push_back((int)cons.size()); }
    auto flatten = [&](auto &per_atom, auto &flat, std::vector<int> &off) {
        off.assign(1, 0);
        for (int i = 0; i < n; i++) { flat.insert(flat.end(), per_atom[i].begin(), per_atom[i].end()); off.push_back((int)flat.size()); }
    };
    std::vector<MolBond> bonds; std::vector<MolAngle> angles; std::vector<MolTorsion> tors; std::vector<MolExc> exc;
    std::vector<int> b_off, a_off, t_off, x_off;
    flatten(ba, bonds, b_off); flatten(aa, angles, a_off); flatten(ta, tors, t_off); flatten(xa, exc, x_off);
    std::vector<double> seps(n);
    for (int i = 0; i < n; i++) seps[i] = sqrt(eps[i]);
    // (padding so that the 8-byte staging copies never read past an allocation)
    b_off.push_back(0); a_off.push_back(0); t_off.push_back(0); x_off.push_back(0); mask.push_back(0);
    MolDev *m = (MolDev *)h->mol_dev;
    if (!m) { m = new MolDev(); h->mol_dev = m; }
    memset(m, 0, sizeof(*m));
    for (int i = 0; i <= n; i++) { m->b_off_h[i] = b_off[i]; m->a_off_h[i] = a_off[i]; m->t_off_h[i] = t_off[i]; m->x_off_h[i] = x_off[i]; }
    {
        auto up = [](size_t b) { return (b + 15) & ~(size_t)15; };
        m->shared_bytes = (int)(up(sizeof(MolBond) * bonds.size()) + up(sizeof(MolAngle) * angles.size()) + up(sizeof(MolTorsion) * tors.size()) +
                                up(sizeof(MolExc) * exc.size()) + 4 * up(sizeof(int) * (n + 2)) + 3 * up(sizeof(double) * n) + up(sizeof(unsigned) * (n + 1)) + 64);
    }
    m->n = n; m->n_clusters = (int)cl.size(); m->remove_cm = mol->remove_cm_motion ? 1 : 0;
    for (auto &c : cl) m->max_cluster = std::max(m->max_cluster, (int)c.size());
    m->tol = mol->constraint_tolerance > 0 ? mol->constraint_tolerance : 1e-8;   // integrators.py constraint_tolerance default
    // ---- term tables of the dynamics (each term once) and the slots of their force contributions: atom by atom, in the
    // order bonds, angles, torsions, pairs, each in list order
    {
        struct Contrib { int kind, term, role; };
        std::vector<std::vector<Contrib>> per_atom(n);
        std::vector<TBond> tb((size_t)mol->n_bonds);
        std::vector<TAngle> tang((size_t)mol->n_angles);
        std::vector<TTors> tt((size_t)mol->n_torsions);
        std::vector<TPair> tp;
        for (int b = 0; b < mol->n_bonds; b++) {
            const double *q = mol->bonds + 4 * b;
            tb[b] = TBond{(short)q[0], (short)q[1], 0, 0, (float)q[2], (float)q[3]};
            per_atom[(int)q[0]].push_back({0, b, 0}); per_atom[(int)q[1]].push_back({0, b, 1});
        }
        for (int a = 0; a < mol->n_angles; a++) {
            const double *q = mol->angles + 5 * a;
            tang[a] = TAngle{(short)q[0], (short)q[1], (short)q[2], 0, 0, 0, (float)q[3], (float)q[4]};
            for (int r = 0; r < 3; r++) per_atom[(int)q[r]].push_back({1, a, r});
        }
        for (int t = 0; t < mol->n_torsions; t++) {
            const double *q = mol->torsions + 7 * t;
            tt[t] = TTors{(short)q[0], (short)q[1], (short)q[2], (short)q[3], 0, 0, 0, 0, (float)q[4], (float)q[5], (float)q[6]};
            for (int r = 0; r < 4; r++) per_atom[(int)q[r]].push_back({2, t, r});
        }
        for (int i = 0; i < n; i++)
            for (int j = i + 1; j < n; j++)
                if ((mask[i] >> j) & 1u) {
                    tp.push_back(TPair{(short)i, (short)j, 0, 0, (float)(MOL_ONE_4PI_EPS0 * charge[i] * charge[j]),
                                       (float)(0.5 * (sigma[i] + sigma[j])), (float)sqrt(eps[i] * eps[j])});
                    per_atom[i].push_back({3, (int)tp.size() - 1, 0}); per_atom[j].push_back({3, (int)tp.size() - 1, 1});
                }
        for (int e = 0; e < mol->n_exceptions; e++) {
            const double *q = mol->exceptions + 5 * e;
            tp.push_back(TPair{(short)q[0], (short)q[1], 0, 0, (float)(MOL_ONE_4PI_EPS0 * q[2]), (float)q[3], (float)q[4]});
            per_atom[(int)q[0]].push_back({3, (int)tp.size() - 1, 0}); per_atom[(int)q[1]].push_back({3, (int)tp.size() - 1, 1});
        }
        std::vector<int> goff(1, 0);
        int slot = 0;
        for (int i = 0; i < n; i++) {
            for (const Contrib &c : per_atom[i]) {
                short *dst = nullptr;
                if (c.kind == 0) dst = c.role == 0 ? &tb[c.term].si : &tb[c.term].sj;
                else if (c.kind == 1) dst = c.role == 0 ? &tang[c.term].si : (c.role == 1 ? &tang[c.term].sj : &tang[c.term].sk);
                else if (c.kind == 2) dst = c.role == 0 ? &tt[c.term].si : (c.role == 1 ? &tt[c.term].sj : (c.role == 2 ? &tt[c.term].sk : &tt[c.term].sl));
                else dst = c.role == 0 ? &tp[c.term].si : &tp[c.term].sj;
                *dst = (short)slot++;
            }
            goff.push_back(slot);
        }
        goff.push_back(slot);   // (padding to an even count)
        auto up = [](size_t b) { return (b + 15) & ~(size_t)15; };
        MolTerms hd;
        memset(&hd, 0, sizeof(hd));
        size_t off = up(sizeof(MolTerms));
        hd.o_bond = (int)off; off += up(sizeof(TBond) * tb.size());
        hd.o_angle = (int)off; off += up(sizeof(TAngle) * tang.size());
        hd.o_tors = (int)off; off += up(sizeof(TTors) * tt.size());
        hd.o_pair = (int)off; off += up(sizeof(TPair) * tp.size());
        hd.o_goff = (int)off; off += up(sizeof(int) * goff.size());
        std::vector<unsigned char> blob(off, 0);
        memcpy(blob.data(), &hd, sizeof(hd));
        if (!tb.empty()) memcpy(blob.data() + hd.o_bond, tb.data(), sizeof(TBond) * tb.size());
        if (!tang.empty()) memcpy(blob.data() + hd.o_angle, tang.data(), sizeof(TAngle) * tang.size());
        if (!tt.empty()) memcpy(blob.data() + hd.o_tors, tt.data(), sizeof(TTors) * tt.size());
        if (!tp.empty()) memcpy(blob.data() + hd.o_pair, tp.data(), sizeof(TPair) * tp.size());
        memcpy(blob.data() + hd.o_goff, goff.data(), sizeof(int) * goff.size());
        const unsigned char *d_blob = nullptr;
        int rcb = mol_upload(h, blob, &d_blob);
        if (rcb) return rcb;
        m->terms = (const MolTerms *)d_blob;
        m->terms_bytes = (int)off;
        m->n_tb = (int)tb.size(); m->n_ta = (int)tang.size(); m->n_tt = (int)tt.size(); m->n_tp = (int)tp.size(); m->n_slots = slot;
        m->dyn_shared_bytes = m->shared_bytes + (int)up(off) + (int)up(sizeof(float) * 3 * (size_t)(slot > 0 ? slot : 1));
    }
    int rc = 0;
    if ((rc = mol_upload(h, mass, &m->mass)) || (rc = mol_upload(h, charge, &m->charge)) || (rc = mol_upload(h, sigma, &m->sigma)) ||
        (rc = mol_upload(h, eps, &m->eps)) || (rc = mol_upload(h, seps, &m->seps)) || (rc = mol_upload(h, b_off, &m->b_off)) || (rc = mol_upload(h, a_off, &m->a_off)) ||
        (rc = mol_upload(h, t_off, &m->t_off)) || (rc = mol_upload(h, x_off, &m->x_off)) || (rc = mol_upload(h, c_off, &m->c_off)) ||
        (rc = mol_upload(h, bonds, &m->bonds)) || (rc = mol_upload(h, angles, &m->angles)) || (rc = mol_upload(h, tors, &m->torsions)) ||
        (rc = mol_upload(h, exc, &m->exc)) || (rc = mol_upload(h, cons, &m->cons)) || (rc = mol_upload(h, mask, &m->nb_mask)))
        return rc;
    h->have_particles = true;
    return RX_OK;
}

void rxi_free_molecule(rx_engine *h) {
    for (void *d : h->mol_allocs) cudaFree(d);
    h->mol_allocs.clear();
    delete (MolDev *)h->mol_dev;
    h->mol_dev = nullptr;
}
