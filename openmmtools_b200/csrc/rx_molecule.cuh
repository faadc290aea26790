// rx_molecule.cuh -- a small molecule in vacuum per replica (included at the end of rx_dynamics.cu).
//
// The system testsystems.AlanineDipeptideVacuum builds (/root/reference/openmmtools/testsystems.py:3352-3388:
// AmberPrmtopFile.createSystem(implicitSolvent=None, constraints=HBonds, nonbondedCutoff=None)) propagated by the constrained
// Langevin splitting of /root/reference/openmmtools/integrators.py:1404-1460:
//   R  x1 = x + (dt/nR) v;  x = constrain(x1);  v += (x - x1) / (dt/nR);  constrain velocities      (:1404-1422)
//   V  v += (dt/nV) f / m;  constrain velocities                                                    (:1424-1447)
//   O  v = a v + b sqrt(kT/m) xi;  constrain velocities                                             (:1449-1460)
// with the centre-of-mass velocity removed at the start of every step (CMMotionRemover through addUpdateContextState).
//
// k_propagate_mol: one block of four warps per replica, the state (x, v in f64) on chip for all steps.  Warp 0 integrates --
// one lane per atom (N <= 32), one lane per constraint cluster -- and all 128 threads evaluate the force terms in f32 on the
// f64 positions: every bond / angle / torsion / pair ONCE, by whichever thread its index falls to, into fixed shared-memory
// slots that each atom then adds up in slot order (no atomics: the same bits every run, whatever the thread count).
// Constraints are solved cluster by cluster (connected components of the constraint graph, e.g. a CH3 group) by the lane that
// owns the cluster.  Clusters of <= 3 constraints (every H-bond cluster) take the MolStar path: register copies of the
// cluster's <= 4 atoms, the RATTLE matrix inverted once per position update in closed form, SHAKE as chord iterations on that
// inverse (k_propagate_mol<true>); larger clusters a Newton M-SHAKE (<= 4 constraints) or Gauss-Seidel sweeps
// (k_propagate_mol<false>).  All of them reach the constrained point of oracle/rx_oracle_mol.c's sweeps to the tolerance.
// The energy kernel (k_energy_mol, f64) and the minimiser (k_minimize_mol) use one warp per replica and the per-atom term
// lists (a lane computes the terms that contain its atom).
#pragma once

#define MOL_MAX_ATOMS 32
#define MOL_ONE_4PI_EPS0 138.935456

struct MolBond { int j, pad; double K, r0; };
struct MolAngle { int i, j, k, role; double K, t0; };
struct MolTorsion { int i, j, k, l, n, role; double phase, kk; };
struct MolExc { int j, pad; double qq, sig, eps; };
struct MolCons { int i, j; double d; };

// Term tables of the dynamics' force evaluation: every bond / angle / torsion / interacting pair is evaluated ONCE, by
// whichever lane its index falls to (t = lane, lane + 32, ...), in f32; its contributions go to fixed slots of a shared-memory
// array and every atom then adds up ITS slots in slot order -- no atomics, the same bits every run.  (The per-atom
// evaluation of mol_atom() runs each angle three and each torsion four times, with loops of unequal length per lane.)
struct TBond { short i, j, si, sj; float K, r0; };
struct TAngle { short i, j, k, si, sj, sk; float K, t0; };
struct TTors { short i, j, k, l, si, sj, sk, sl; float n, phase, kk; };
struct TPair { short i, j, si, sj; float qq, sig, eps; };   // qq = 138.935456 q_i q_j (exceptions: their own values)
struct MolTerms {      // one contiguous blob: header, then the arrays (offsets in bytes from the blob's start)
    int o_bond, o_angle, o_tors, o_pair, o_goff, pad[3];
};

struct MolDev {
    int n, n_clusters, remove_cm, max_cluster;   // max_cluster: constraints in the largest cluster
    double tol;
    const double *mass, *charge, *sigma, *eps, *seps;
    const int *b_off, *a_off, *t_off, *x_off, *c_off;
    int b_off_h[MOL_MAX_ATOMS + 1], a_off_h[MOL_MAX_ATOMS + 1], t_off_h[MOL_MAX_ATOMS + 1], x_off_h[MOL_MAX_ATOMS + 1];   // (host copies: counts)
    int shared_bytes;
    const MolBond *bonds;
    const MolAngle *angles;
    const MolTorsion *torsions;
    const MolExc *exc;
    const MolCons *cons;
    const unsigned *nb_mask;     // bit b of nb_mask[a]: the pair (a, b) has the plain Coulomb + LJ interaction
    // term-parallel force evaluation of the dynamics (one entry per TERM, see mol_forces_terms)
    const struct MolTerms *terms;
    int terms_bytes, n_tb, n_ta, n_tt, n_tp, n_slots, dyn_shared_bytes;
};

__device__ __forceinline__ void mol_cross(const double *a, const double *b, double *c) {
    c[0] = a[1] * b[2] - a[2] * b[1]; c[1] = a[2] * b[0] - a[0] * b[2]; c[2] = a[0] * b[1] - a[1] * b[0];
}
__device__ __forceinline__ double mol_dot(const double *a, const double *b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }

template <typename R> __device__ __forceinline__ R mol_sqrt(R x);
template <> __device__ __forceinline__ float mol_sqrt<float>(float x) { return sqrtf(x); }
template <> __device__ __forceinline__ double mol_sqrt<double>(double x) { return sqrt(x); }
template <typename R> __device__ __forceinline__ R mol_acos(R x);
template <> __device__ __forceinline__ float mol_acos<float>(float x) { return acosf(x); }
template <> __device__ __forceinline__ double mol_acos<double>(double x) { return acos(x); }
template <typename R> __device__ __forceinline__ R mol_atan2(R y, R x);
template <> __device__ __forceinline__ float mol_atan2<float>(float y, float x) { return atan2f(y, x); }
template <> __device__ __forceinline__ double mol_atan2<double>(double y, double x) { return atan2(y, x); }
template <typename R> __device__ __forceinline__ void mol_sincos(R x, R *s, R *c);
template <> __device__ __forceinline__ void mol_sincos<float>(float x, float *s, float *c) { sincosf(x, s, c); }
template <> __device__ __forceinline__ void mol_sincos<double>(double x, double *s, double *c) { sincos(x, s, c); }

// The term tables of one molecule in shared memory (a few KB: read every step by every lane).
struct MolShared {
    const MolBond *bonds; const MolAngle *angles; const MolTorsion *torsions; const MolExc *exc;
    const int *b_off, *a_off, *t_off, *x_off;
    const double *charge, *sigma, *seps;   // seps = sqrt(epsilon)
    const unsigned *nb_mask;
    int n;
};

// Force on atom a (ENERGY: instead the energy of the terms this atom owns: bonds/exceptions/pairs with the larger partner
// index, angles and torsions in which it has role 0).  X: positions of all atoms in shared memory.  R: the arithmetic type --
// float for the forces of the dynamics (as in k_propagate: f32 forces on f64-stored positions, differences taken in f64),
// double for energies.
template <bool ENERGY, typename R>
__device__ double mol_atom(const MolShared &m, const double (*X)[3], int a, double *f) {
    double e = 0.0;
    R fx = 0, fy = 0, fz = 0;
    const double xa[3] = {X[a][0], X[a][1], X[a][2]};
    for (int q = m.b_off[a]; q < m.b_off[a + 1]; q++) {
        const MolBond b = m.bonds[q];
        const R d[3] = {(R)(xa[0] - X[b.j][0]), (R)(xa[1] - X[b.j][1]), (R)(xa[2] - X[b.j][2])};
        const R r = mol_sqrt<R>(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]), dr = r - (R)b.r0;
        if (ENERGY) { if (b.j > a) e += 0.5 * b.K * (double)dr * (double)dr; }
        else { const R c = -(R)b.K * dr / r; fx += c * d[0]; fy += c * d[1]; fz += c * d[2]; }
    }
    for (int q = m.a_off[a]; q < m.a_off[a + 1]; q++) {
        const MolAngle g = m.angles[q];
        R u[3], v[3];
        for (int c = 0; c < 3; c++) { u[c] = (R)(X[g.i][c] - X[g.j][c]); v[c] = (R)(X[g.k][c] - X[g.j][c]); }
        const R ru2 = u[0] * u[0] + u[1] * u[1] + u[2] * u[2], rv2 = v[0] * v[0] + v[1] * v[1] + v[2] * v[2];
        const R iruv = (R)1 / mol_sqrt<R>(ru2 * rv2);
        R cs = (u[0] * v[0] + u[1] * v[1] + u[2] * v[2]) * iruv;
        cs = cs > (R)1 ? (R)1 : (cs < (R)-1 ? (R)-1 : cs);
        const R dt = mol_acos<R>(cs) - (R)g.t0;
        if (ENERGY) { if (g.role == 0) e += 0.5 * g.K * (double)dt * (double)dt; }
        else {
            const R sn = mol_sqrt<R>((R)1 - cs * cs);
            const R gg = (sn > (R)1e-6) ? (R)g.K * dt / sn : (R)0;
            R o[3];
            for (int c = 0; c < 3; c++) {
                const R fi = gg * (v[c] * iruv - cs * u[c] / ru2);
                const R fk = gg * (u[c] * iruv - cs * v[c] / rv2);
                o[c] = g.role == 0 ? fi : (g.role == 2 ? fk : -(fi + fk));
            }
            fx += o[0]; fy += o[1]; fz += o[2];
        }
    }
    for (int q = m.t_off[a]; q < m.t_off[a + 1]; q++) {
        const MolTorsion t = m.torsions[q];
        R rij[3], rkj[3], rkl[3], mm[3], nn[3];
        for (int c = 0; c < 3; c++) { rij[c] = (R)(X[t.i][c] - X[t.j][c]); rkj[c] = (R)(X[t.k][c] - X[t.j][c]); rkl[c] = (R)(X[t.k][c] - X[t.l][c]); }
        mm[0] = rij[1] * rkj[2] - rij[2] * rkj[1]; mm[1] = rij[2] * rkj[0] - rij[0] * rkj[2]; mm[2] = rij[0] * rkj[1] - rij[1] * rkj[0];
        nn[0] = rkj[1] * rkl[2] - rkj[2] * rkl[1]; nn[1] = rkj[2] * rkl[0] - rkj[0] * rkl[2]; nn[2] = rkj[0] * rkl[1] - rkj[1] * rkl[0];
        const R rkj2 = rkj[0] * rkj[0] + rkj[1] * rkj[1] + rkj[2] * rkj[2], nrkj = mol_sqrt<R>(rkj2);
        const R phi = mol_atan2<R>(nrkj * (rij[0] * nn[0] + rij[1] * nn[1] + rij[2] * nn[2]), mm[0] * nn[0] + mm[1] * nn[1] + mm[2] * nn[2]);
        R sn, cs;
        mol_sincos<R>((R)t.n * phi - (R)t.phase, &sn, &cs);
        if (ENERGY) { if (t.role == 0) e += t.kk * (1.0 + (double)cs); }
        else {
            const R dU = -(R)t.kk * (R)t.n * sn;
            const R m2 = mm[0] * mm[0] + mm[1] * mm[1] + mm[2] * mm[2], n2 = nn[0] * nn[0] + nn[1] * nn[1] + nn[2] * nn[2];
            const R pp = (rij[0] * rkj[0] + rij[1] * rkj[1] + rij[2] * rkj[2]) / rkj2, qq = (rkl[0] * rkj[0] + rkl[1] * rkj[1] + rkl[2] * rkj[2]) / rkj2;
            const R ci = -dU * nrkj / m2, cl = dU * nrkj / n2;
            R o[3];
            for (int c = 0; c < 3; c++) {
                const R fi = ci * mm[c], fl = cl * nn[c];
                const R sv = pp * fi - qq * fl;
                o[c] = t.role == 0 ? fi : (t.role == 1 ? sv - fi : (t.role == 2 ? -sv - fl : fl));
            }
            fx += o[0]; fy += o[1]; fz += o[2];
        }
    }
    const unsigned mask = m.nb_mask[a];
    const R qa = (R)(MOL_ONE_4PI_EPS0 * m.charge[a]), sa = (R)m.sigma[a], ea = (R)m.seps[a];
    for (int b = 0; b < m.n; b++) {
        if (!((mask >> b) & 1u)) continue;
        if (ENERGY && b < a) continue;
        const R d[3] = {(R)(xa[0] - X[b][0]), (R)(xa[1] - X[b][1]), (R)(xa[2] - X[b][2])};
        const R ir2 = (R)1 / (d[0] * d[0] + d[1] * d[1] + d[2] * d[2]), ir = mol_sqrt<R>(ir2);
        const R qq = qa * (R)m.charge[b], s = (R)0.5 * (sa + (R)m.sigma[b]), ee = ea * (R)m.seps[b];
        const R s2 = s * s * ir2, s6 = s2 * s2 * s2;
        if (ENERGY) e += (double)(qq * ir + (R)4 * ee * (s6 * s6 - s6));
        else { const R c = (qq * ir + (R)24 * ee * ((R)2 * s6 * s6 - s6)) * ir2; fx += c * d[0]; fy += c * d[1]; fz += c * d[2]; }
    }
    for (int q = m.x_off[a]; q < m.x_off[a + 1]; q++) {
        const MolExc x = m.exc[q];
        if (ENERGY && x.j < a) continue;
        const R d[3] = {(R)(xa[0] - X[x.j][0]), (R)(xa[1] - X[x.j][1]), (R)(xa[2] - X[x.j][2])};
        const R ir2 = (R)1 / (d[0] * d[0] + d[1] * d[1] + d[2] * d[2]), ir = mol_sqrt<R>(ir2);
        const R qq = (R)(MOL_ONE_4PI_EPS0 * x.qq);
        const R s2 = (R)(x.sig * x.sig) * ir2, s6 = s2 * s2 * s2;
        if (ENERGY) e += (double)(qq * ir + (R)4 * (R)x.eps * (s6 * s6 - s6));
        else { const R c = (qq * ir + (R)24 * (R)x.eps * ((R)2 * s6 * s6 - s6)) * ir2; fx += c * d[0]; fy += c * d[1]; fz += c * d[2]; }
    }
    if (!ENERGY) { f[0] = (double)fx; f[1] = (double)fy; f[2] = (double)fz; }
    return e;
}

// All terms, each once (see MolTerms).  FS: float[n_slots][3] in shared memory.
__device__ __forceinline__ void mol_forces_terms(const MolDev &m, const unsigned char *tb, const double (*X)[3], float (*FS)[3]) {
    const MolTerms *h = (const MolTerms *)tb;
    const int lane = threadIdx.x, nth = blockDim.x;   // (k_propagate_mol: all warps of the block; the other kernels: one warp)
    const TBond *B = (const TBond *)(tb + h->o_bond);
    // (which thread evaluates a term does not matter for the result -- fixed slots; the four kinds start at different threads so
    // that no thread gets a torsion AND an angle AND two pairs: the evaluation is as long as its busiest thread)
    for (int t = (lane + nth / 2) % nth; t < m.n_tb; t += nth) {
        const TBond b = B[t];
        const float d[3] = {(float)(X[b.i][0] - X[b.j][0]), (float)(X[b.i][1] - X[b.j][1]), (float)(X[b.i][2] - X[b.j][2])};
        const float r = sqrtf(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
        const float c = -b.K * (r - b.r0) / r;
        for (int q = 0; q < 3; q++) { FS[b.si][q] = c * d[q]; FS[b.sj][q] = -c * d[q]; }
    }
    const TAngle *A = (const TAngle *)(tb + h->o_angle);
    for (int t = nth - 1 - lane; t < m.n_ta; t += nth) {
        const TAngle g = A[t];
        float u[3], v[3];
        for (int c = 0; c < 3; c++) { u[c] = (float)(X[g.i][c] - X[g.j][c]); v[c] = (float)(X[g.k][c] - X[g.j][c]); }
        const float ru2 = u[0] * u[0] + u[1] * u[1] + u[2] * u[2], rv2 = v[0] * v[0] + v[1] * v[1] + v[2] * v[2];
        const float iruv = rsqrtf(ru2 * rv2);
        float cs = (u[0] * v[0] + u[1] * v[1] + u[2] * v[2]) * iruv;
        cs = fminf(1.f, fmaxf(-1.f, cs));
        const float dt = acosf(cs) - g.t0, sn = sqrtf(1.f - cs * cs);
        const float gg = (sn > 1e-6f) ? g.K * dt / sn : 0.f;
        for (int c = 0; c < 3; c++) {
            const float fi = gg * (v[c] * iruv - cs * u[c] / ru2), fk = gg * (u[c] * iruv - cs * v[c] / rv2);
            FS[g.si][c] = fi; FS[g.sk][c] = fk; FS[g.sj][c] = -(fi + fk);
        }
    }
    const TTors *T = (const TTors *)(tb + h->o_tors);
    for (int t = lane; t < m.n_tt; t += nth) {
        const TTors w = T[t];
        float rij[3], rkj[3], rkl[3], mm[3], nn[3];
        for (int c = 0; c < 3; c++) { rij[c] = (float)(X[w.i][c] - X[w.j][c]); rkj[c] = (float)(X[w.k][c] - X[w.j][c]); rkl[c] = (float)(X[w.k][c] - X[w.l][c]); }
        mm[0] = rij[1] * rkj[2] - rij[2] * rkj[1]; mm[1] = rij[2] * rkj[0] - rij[0] * rkj[2]; mm[2] = rij[0] * rkj[1] - rij[1] * rkj[0];
        nn[0] = rkj[1] * rkl[2] - rkj[2] * rkl[1]; nn[1] = rkj[2] * rkl[0] - rkj[0] * rkl[2]; nn[2] = rkj[0] * rkl[1] - rkj[1] * rkl[0];
        const float rkj2 = rkj[0] * rkj[0] + rkj[1] * rkj[1] + rkj[2] * rkj[2], nrkj = sqrtf(rkj2);
        const float phi = atan2f(nrkj * (rij[0] * nn[0] + rij[1] * nn[1] + rij[2] * nn[2]), mm[0] * nn[0] + mm[1] * nn[1] + mm[2] * nn[2]);
        float sn, cs;
        sincosf(w.n * phi - w.phase, &sn, &cs);
        const float dU = -w.kk * w.n * sn;
        const float m2 = mm[0] * mm[0] + mm[1] * mm[1] + mm[2] * mm[2], n2 = nn[0] * nn[0] + nn[1] * nn[1] + nn[2] * nn[2];
        const float pp = (rij[0] * rkj[0] + rij[1] * rkj[1] + rij[2] * rkj[2]) / rkj2, qq = (rkl[0] * rkj[0] + rkl[1] * rkj[1] + rkl[2] * rkj[2]) / rkj2;
        const float ci = -dU * nrkj / m2, cl = dU * nrkj / n2;
        for (int c = 0; c < 3; c++) {
            const float fi = ci * mm[c], fl = cl * nn[c], sv = pp * fi - qq * fl;
            FS[w.si][c] = fi; FS[w.sj][c] = sv - fi; FS[w.sk][c] = -sv - fl; FS[w.sl][c] = fl;
        }
    }
    const TPair *P = (const TPair *)(tb + h->o_pair);
    for (int t = ((lane - m.n_tt) % nth + nth) % nth; t < m.n_tp; t += nth) {
        const TPair p = P[t];
        const float d[3] = {(float)(X[p.i][0] - X[p.j][0]), (float)(X[p.i][1] - X[p.j][1]), (float)(X[p.i][2] - X[p.j][2])};
        const float ir2 = 1.f / (d[0] * d[0] + d[1] * d[1] + d[2] * d[2]), ir = sqrtf(ir2);
        const float s2 = p.sig * p.sig * ir2, s6 = s2 * s2 * s2;
        const float c = (p.qq * ir + 24.f * p.eps * (2.f * s6 * s6 - s6)) * ir2;
        for (int q = 0; q < 3; q++) { FS[p.si][q] = c * d[q]; FS[p.sj][q] = -c * d[q]; }
    }
}

// Copy the term tables into shared memory (all lanes of the warp; `buf` has room for mol_shared_bytes(m)).
__device__ void mol_stage(const MolDev &m, unsigned char *buf, MolShared &s) {
    const int n = m.n, lane = threadIdx.x;
    const size_t stride = (size_t)blockDim.x * 8;
    auto put = [&](const void *src, size_t bytes) {
        unsigned char *dst = buf;
        for (size_t q = lane * 8; q < bytes; q += stride) *(unsigned long long *)(dst + q) = *(const unsigned long long *)((const unsigned char *)src + q);
        buf += (bytes + 15) & ~(size_t)15;
        return dst;
    };
    s.n = n;
    const int nb = m.b_off_h[n], na = m.a_off_h[n], nt = m.t_off_h[n], nx = m.x_off_h[n];
    s.bonds = (const MolBond *)put(m.bonds, sizeof(MolBond) * nb);
    s.angles = (const MolAngle *)put(m.angles, sizeof(MolAngle) * na);
    s.torsions = (const MolTorsion *)put(m.torsions, sizeof(MolTorsion) * nt);
    s.exc = (const MolExc *)put(m.exc, sizeof(MolExc) * nx);
    s.b_off = (const int *)put(m.b_off, sizeof(int) * (n + 2)); s.a_off = (const int *)put(m.a_off, sizeof(int) * (n + 2));
    s.t_off = (const int *)put(m.t_off, sizeof(int) * (n + 2)); s.x_off = (const int *)put(m.x_off, sizeof(int) * (n + 2));
    s.charge = (const double *)put(m.charge, sizeof(double) * n); s.sigma = (const double *)put(m.sigma, sizeof(double) * n);
    s.seps = (const double *)put(m.seps, sizeof(double) * n);
    s.nb_mask = (const unsigned *)put(m.nb_mask, sizeof(unsigned) * (n + 1));
    if (blockDim.x > 32) __syncthreads(); else __syncwarp();
}

// Constraints are solved per cluster (connected component of the constraint graph) by ONE lane.  Clusters of up to
// MOL_MAXC constraints (a CH3 group has three) are solved as a whole: the velocity conditions are a linear system in the
// multipliers (one solve), the position conditions are solved by Newton iterations on the same coupled system
// (M-SHAKE: converges quadratically, 2-3 iterations where Gauss-Seidel sweeps need ~10).  Larger clusters fall back to
// Gauss-Seidel sweeps.  Both reach the same constrained point to the tolerance (the oracle uses sweeps).
#define MOL_MAXC 4

struct MolCluster {       // one lane's cluster, in registers / local memory for the whole kernel
    int nc;
    int i[MOL_MAXC], j[MOL_MAXC];
    double d2[MOL_MAXC], wi[MOL_MAXC], wj[MOL_MAXC];
    double coup[MOL_MAXC][MOL_MAXC];   // mass coupling of constraints c and d (see mol_load_cluster)
};

__device__ __forceinline__ void mol_load_cluster(const MolDev &m, int c, MolCluster &k) {
    const int q0 = m.c_off[c];
    k.nc = m.c_off[c + 1] - q0;
    // (static indices only, so that the whole record lives in registers)
#pragma unroll
    for (int a = 0; a < MOL_MAXC; a++) {
        const bool on = a < k.nc && k.nc <= MOL_MAXC;
        const MolCons s = on ? m.cons[q0 + a] : MolCons{0, 0, 1.0};
        k.i[a] = s.i; k.j[a] = s.j; k.d2[a] = s.d * s.d;
        k.wi[a] = on ? 1.0 / m.mass[s.i] : 0.0; k.wj[a] = on ? 1.0 / m.mass[s.j] : 0.0;
    }
    // a unit multiplier on constraint d moves x_i(d) by +w r_d and x_j(d) by -w r_d: its effect on the bond vector of c
#pragma unroll
    for (int a = 0; a < MOL_MAXC; a++)
#pragma unroll
        for (int b = 0; b < MOL_MAXC; b++) {
            double v = 0.0;
            if (k.i[a] == k.i[b]) v += k.wi[a];
            if (k.i[a] == k.j[b]) v -= k.wi[a];
            if (k.j[a] == k.i[b]) v -= k.wj[a];
            if (k.j[a] == k.j[b]) v += k.wj[a];
            k.coup[a][b] = v;
        }
}

// solve A g = b in place (A: NC x NC, diagonally dominant here), result in b; fully unrolled: everything stays in registers
template <int NC>
__device__ __forceinline__ void mol_solve(double (*A)[MOL_MAXC], double *b) {
#pragma unroll
    for (int p = 0; p < NC; p++) {
        const double ip = 1.0 / A[p][p];
#pragma unroll
        for (int r = p + 1; r < NC; r++) {
            const double f = A[r][p] * ip;
#pragma unroll
            for (int c = p; c < NC; c++) A[r][c] -= f * A[p][c];
            b[r] -= f * b[p];
        }
    }
#pragma unroll
    for (int p = NC - 1; p >= 0; p--) {
        double v = b[p];
#pragma unroll
        for (int c = p + 1; c < NC; c++) v -= A[p][c] * b[c];
        b[p] = v / A[p][p];
    }
}

// SHAKE on a cluster of NC constraints: Newton iterations on the coupled system (M-SHAKE).
template <int NC>
__device__ __forceinline__ void mol_shake_n(const MolDev &m, const MolCluster &k, const double (*XO)[3], double (*X)[3]) {
    double r0[MOL_MAXC][3];
#pragma unroll
    for (int a = 0; a < NC; a++)
#pragma unroll
        for (int q = 0; q < 3; q++) r0[a][q] = XO[k.i[a]][q] - XO[k.j[a]][q];
    for (int it = 0; it < 50; it++) {
        double A[MOL_MAXC][MOL_MAXC], g[MOL_MAXC], r[MOL_MAXC][3];
        bool done = true;
#pragma unroll
        for (int a = 0; a < NC; a++) {
#pragma unroll
            for (int q = 0; q < 3; q++) r[a][q] = X[k.i[a]][q] - X[k.j[a]][q];
            g[a] = k.d2[a] - mol_dot(r[a], r[a]);
            if (fabs(g[a]) > m.tol * k.d2[a]) done = false;
        }
        if (done) break;
#pragma unroll
        for (int a = 0; a < NC; a++)
#pragma unroll
            for (int b = 0; b < NC; b++) A[a][b] = 2.0 * k.coup[a][b] * mol_dot(r[a], r0[b]);
        mol_solve<NC>(A, g);
#pragma unroll
        for (int b = 0; b < NC; b++)
#pragma unroll
            for (int q = 0; q < 3; q++) { X[k.i[b]][q] += g[b] * k.wi[b] * r0[b][q]; X[k.j[b]][q] -= g[b] * k.wj[b] * r0[b][q]; }
    }
}

// RATTLE on a cluster of NC constraints: one linear solve.
template <int NC>
__device__ __forceinline__ void mol_rattle_n(const MolCluster &k, const double (*X)[3], double (*V)[3]) {
    double A[MOL_MAXC][MOL_MAXC], g[MOL_MAXC], r[MOL_MAXC][3];
#pragma unroll
    for (int a = 0; a < NC; a++) {
        double dv[3];
#pragma unroll
        for (int q = 0; q < 3; q++) { r[a][q] = X[k.i[a]][q] - X[k.j[a]][q]; dv[q] = V[k.i[a]][q] - V[k.j[a]][q]; }
        g[a] = mol_dot(r[a], dv);
    }
#pragma unroll
    for (int a = 0; a < NC; a++)
#pragma unroll
        for (int b = 0; b < NC; b++) A[a][b] = k.coup[a][b] * mol_dot(r[a], r[b]);
    mol_solve<NC>(A, g);
#pragma unroll
    for (int b = 0; b < NC; b++)
#pragma unroll
        for (int q = 0; q < 3; q++) { V[k.i[b]][q] -= g[b] * k.wi[b] * r[b][q]; V[k.j[b]][q] += g[b] * k.wj[b] * r[b][q]; }
}

// SHAKE on one cluster: positions X moved so that its constraints have their lengths, along the bond vectors of XO.
__device__ __forceinline__ void mol_shake_cluster(const MolDev &m, int c, const MolCluster &k, const double (*XO)[3], double (*X)[3]) {
    switch (k.nc) {
        case 1: mol_shake_n<1>(m, k, XO, X); return;
        case 2: mol_shake_n<2>(m, k, XO, X); return;
        case 3: mol_shake_n<3>(m, k, XO, X); return;
        case 4: mol_shake_n<4>(m, k, XO, X); return;
        default: break;
    }
    for (int it = 0; it < 500; it++) {
        bool done = true;
        for (int q = m.c_off[c]; q < m.c_off[c + 1]; q++) {
            const MolCons s = m.cons[q];
            const double d2 = s.d * s.d;
            double r[3], r0[3];
            for (int a = 0; a < 3; a++) { r[a] = X[s.i][a] - X[s.j][a]; r0[a] = XO[s.i][a] - XO[s.j][a]; }
            const double diff = d2 - mol_dot(r, r);
            if (fabs(diff) > m.tol * d2) {
                done = false;
                const double wi = 1.0 / m.mass[s.i], wj = 1.0 / m.mass[s.j];
                const double g = diff / (2.0 * (wi + wj) * mol_dot(r, r0));
                for (int a = 0; a < 3; a++) { X[s.i][a] += g * wi * r0[a]; X[s.j][a] -= g * wj * r0[a]; }
            }
        }
        if (done) break;
    }
}

// RATTLE on one cluster: the velocity components along its constraints are removed.
__device__ __forceinline__ void mol_rattle_cluster(const MolDev &m, int c, const MolCluster &k, const double (*X)[3], double (*V)[3]) {
    switch (k.nc) {
        case 1: mol_rattle_n<1>(k, X, V); return;
        case 2: mol_rattle_n<2>(k, X, V); return;
        case 3: mol_rattle_n<3>(k, X, V); return;
        case 4: mol_rattle_n<4>(k, X, V); return;
        default: break;
    }
    for (int it = 0; it < 500; it++) {
        bool done = true;
        for (int q = m.c_off[c]; q < m.c_off[c + 1]; q++) {
            const MolCons s = m.cons[q];
            double r[3], dv[3];
            for (int a = 0; a < 3; a++) { r[a] = X[s.i][a] - X[s.j][a]; dv[a] = V[s.i][a] - V[s.j][a]; }
            const double rv = mol_dot(r, dv), r2 = mol_dot(r, r);
            if (fabs(rv) > m.tol * r2) {
                done = false;
                const double wi = 1.0 / m.mass[s.i], wj = 1.0 / m.mass[s.j];
                const double g = rv / ((wi + wj) * r2);
                for (int a = 0; a < 3; a++) { V[s.i][a] -= g * wi * r[a]; V[s.j][a] += g * wj * r[a]; }
            }
        }
        if (done) break;
    }
}

// --- k_propagate_mol's constraint path for clusters of up to three constraints (every H-bond cluster: XH, XH2, XH3; a rigid
// water) ------------------------------------------------------------------------------------------------------------------
// A connected cluster of nc <= 3 constraints has at most 4 atoms: the lane that owns the cluster works on register copies of
// those atoms -- one load and one store per atom and call, nothing read back from shared memory in between (the coupled
// updates of the shared heavy atom were three dependent read-modify-writes per component before).  The geometry is two small
// coefficient tables: E[b][n] (+1, -1, 0: bond vector of constraint b = sum_n E x_n) and S[n][b] (+1/m_i, -1/m_j, 0: a unit
// multiplier on constraint b moves atom n by S r_b).
// The RATTLE matrix A = coup o (r r^T), coup = E S, depends on the positions only, and positions change in the R operations
// only: its inverse is formed ONCE per position update (closed form, one reciprocal) and serves the two to three velocity
// projections that follow as a matrix-vector product -- no pivoting, no division on the step's critical path.  SHAKE iterates
// with the same inverse (the Jacobian at the previous constrained positions is 2 A: a chord iteration; the bond vectors turn
// by about 1e-2 per R operation, so every iteration gains 1.5-2 digits), entirely in registers: 3 dot products and a 3x3
// product per iteration instead of a Newton solve.  Clusters with fewer constraints / atoms are padded (zero coefficients,
// unit diagonal): one instruction stream for all lanes.  Same constrained point as mol_shake_n / the oracle's sweeps to the
// tolerance.
struct MolStar {
    int nc, na;
    int idx[4];          // the cluster's atoms (padded with its first atom: read, never written)
    double S[4][3];
    float E[3][4];
    double d2[3];
    double coup[3][3];
    double r[3][3];      // bond vectors at the last constrained positions
    double Ai[3][3];     // inverse of coup o (r r^T)
};

__device__ __forceinline__ void mol_star_load(const MolDev &m, int c, MolStar &k) {
    const int q0 = m.c_off[c];
    k.nc = m.c_off[c + 1] - q0;
    int ci[3], cj[3], at[4] = {-1, -1, -1, -1}, na = 0;
    double wi[3], wj[3];
    // (static indices only, so that the whole record lives in registers)
#pragma unroll
    for (int a = 0; a < 3; a++) {
        const bool on = a < k.nc;
        const MolCons s = on ? m.cons[q0 + a] : MolCons{-1, -1, 1.0};
        ci[a] = s.i; cj[a] = s.j; k.d2[a] = s.d * s.d;
        wi[a] = on ? 1.0 / m.mass[s.i] : 0.0; wj[a] = on ? 1.0 / m.mass[s.j] : 0.0;
    }
#pragma unroll
    for (int a = 0; a < 3; a++)
#pragma unroll
        for (int e = 0; e < 2; e++) {
            const int atom = e ? cj[a] : ci[a];
            bool found = atom < 0;
#pragma unroll
            for (int n = 0; n < 4; n++) found |= at[n] == atom;
            if (!found) {
#pragma unroll
                for (int n = 0; n < 4; n++) if (n == na) at[n] = atom;
                na++;
            }
        }
    k.na = na;
#pragma unroll
    for (int n = 0; n < 4; n++) {
        k.idx[n] = n < na ? at[n] : at[0];
#pragma unroll
        for (int b = 0; b < 3; b++) {
            const bool is_i = at[n] >= 0 && at[n] == ci[b], is_j = at[n] >= 0 && at[n] == cj[b];
            k.S[n][b] = (is_i ? wi[b] : 0.0) - (is_j ? wj[b] : 0.0);
            k.E[b][n] = (float)((int)is_i - (int)is_j);
        }
    }
#pragma unroll
    for (int a = 0; a < 3; a++)
#pragma unroll
        for (int b = 0; b < 3; b++) {
            double v = 0.0;
#pragma unroll
            for (int n = 0; n < 4; n++) v += (double)k.E[a][n] * k.S[n][b];
            k.coup[a][b] = v;
        }
}

__device__ __forceinline__ void mol_star_invert(MolStar &k) {
    double A[3][3];
#pragma unroll
    for (int a = 0; a < 3; a++)
#pragma unroll
        for (int b = 0; b < 3; b++) A[a][b] = (a == b && a >= k.nc) ? 1.0 : k.coup[a][b] * mol_dot(k.r[a], k.r[b]);
    const double c00 = A[1][1] * A[2][2] - A[1][2] * A[2][1], c01 = A[1][0] * A[2][2] - A[1][2] * A[2][0],
                 c02 = A[1][0] * A[2][1] - A[1][1] * A[2][0];
    const double id = 1.0 / (A[0][0] * c00 - A[0][1] * c01 + A[0][2] * c02);
    k.Ai[0][0] = c00 * id;
    k.Ai[0][1] = (A[0][2] * A[2][1] - A[0][1] * A[2][2]) * id;
    k.Ai[0][2] = (A[0][1] * A[1][2] - A[0][2] * A[1][1]) * id;
    k.Ai[1][0] = -c01 * id;
    k.Ai[1][1] = (A[0][0] * A[2][2] - A[0][2] * A[2][0]) * id;
    k.Ai[1][2] = (A[0][2] * A[1][0] - A[0][0] * A[1][2]) * id;
    k.Ai[2][0] = c02 * id;
    k.Ai[2][1] = (A[0][1] * A[2][0] - A[0][0] * A[2][1]) * id;
    k.Ai[2][2] = (A[0][0] * A[1][1] - A[0][1] * A[1][0]) * id;
}

// bond vectors of the cluster's constraints from register copies of its atoms
__device__ __forceinline__ void mol_star_bonds(const MolStar &k, const double (*x)[3], double (*rb)[3]) {
#pragma unroll
    for (int a = 0; a < 3; a++)
#pragma unroll
        for (int q = 0; q < 3; q++) {
            double v = 0.0;
#pragma unroll
            for (int n = 0; n < 4; n++) v += (double)k.E[a][n] * x[n][q];
            rb[a][q] = v;
        }
}

__device__ __forceinline__ void mol_star_init(MolStar &k, const double (*X)[3]) {
    double x[4][3];
#pragma unroll
    for (int n = 0; n < 4; n++)
#pragma unroll
        for (int q = 0; q < 3; q++) x[n][q] = X[k.idx[n]][q];
    mol_star_bonds(k, x, k.r);
    mol_star_invert(k);
}

__device__ __forceinline__ void mol_star_rattle(const MolStar &k, double (*V)[3]) {
    double v[4][3], dv[3][3], g[3], lam[3];
#pragma unroll
    for (int n = 0; n < 4; n++)
#pragma unroll
        for (int q = 0; q < 3; q++) v[n][q] = V[k.idx[n]][q];
    mol_star_bonds(k, v, dv);
#pragma unroll
    for (int a = 0; a < 3; a++) g[a] = mol_dot(k.r[a], dv[a]);
#pragma unroll
    for (int b = 0; b < 3; b++) lam[b] = k.Ai[b][0] * g[0] + k.Ai[b][1] * g[1] + k.Ai[b][2] * g[2];
#pragma unroll
    for (int n = 0; n < 4; n++)
        if (n < k.na) {
#pragma unroll
            for (int q = 0; q < 3; q++)
                V[k.idx[n]][q] = v[n][q] - (k.S[n][0] * lam[0] * k.r[0][q] + k.S[n][1] * lam[1] * k.r[1][q] + k.S[n][2] * lam[2] * k.r[2][q]);
        }
}

// positions X (moved from the constrained positions the cache was built at) back onto the constraints, along the cached bond
// vectors; the cache is rebuilt at the result.
__device__ __forceinline__ void mol_star_shake(const MolDev &m, MolStar &k, double (*X)[3]) {
    double x[4][3], rc[3][3];
#pragma unroll
    for (int n = 0; n < 4; n++)
#pragma unroll
        for (int q = 0; q < 3; q++) x[n][q] = X[k.idx[n]][q];
    for (int it = 0; it < 60; it++) {
        double g[3], lam[3];
        bool done = true;
        mol_star_bonds(k, x, rc);
#pragma unroll
        for (int a = 0; a < 3; a++) {
            g[a] = a < k.nc ? k.d2[a] - mol_dot(rc[a], rc[a]) : 0.0;
            if (fabs(g[a]) > m.tol * k.d2[a]) done = false;
        }
        if (done) break;
#pragma unroll
        for (int b = 0; b < 3; b++) lam[b] = 0.5 * (k.Ai[b][0] * g[0] + k.Ai[b][1] * g[1] + k.Ai[b][2] * g[2]);
#pragma unroll
        for (int n = 0; n < 4; n++)
#pragma unroll
            for (int q = 0; q < 3; q++)
                x[n][q] += k.S[n][0] * lam[0] * k.r[0][q] + k.S[n][1] * lam[1] * k.r[1][q] + k.S[n][2] * lam[2] * k.r[2][q];
    }
#pragma unroll
    for (int n = 0; n < 4; n++)
        if (n < k.na) {
#pragma unroll
            for (int q = 0; q < 3; q++) X[k.idx[n]][q] = x[n][q];
        }
#pragma unroll
    for (int a = 0; a < 3; a++)
#pragma unroll
        for (int q = 0; q < 3; q++) k.r[a][q] = rc[a][q];
    mol_star_invert(k);
}

__device__ __forceinline__ double mol_warp_sum(double v) {   // fixed tree: bit-reproducible
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// One block of MOL_WARPS warps per owned replica.  Warp 0 integrates (one lane per atom, one lane per constraint cluster);
// all warps evaluate the force terms (each term once, by whichever thread its index falls to, into its fixed slots: the
// per-atom sums in slot order do not depend on the number of threads -- the same bits as with one warp), between two block
// barriers per force evaluation.  Every warp runs the same control flow (steps, program, lazy force flag); warps 1.. only take
// part in the force evaluations.  pos / vel: double[kloc][n][3].
#define MOL_WARPS 4
template <bool STAR>   // STAR: every constraint cluster has at most three constraints (MolDev::max_cluster): the MolStar path
__global__ void __launch_bounds__(32 * MOL_WARPS) k_propagate_mol(MolDev m, DynParams p, const StateDev *__restrict__ states,
                                                      const int *__restrict__ perm, double *__restrict__ pos,
                                                      double *__restrict__ vel, int k0, uint2 key, uint32_t iteration,
                                                      int reassign, double *__restrict__ pot, double *__restrict__ kin,
                                                      int *__restrict__ nan_flag, const int *__restrict__ only) {
    __shared__ double X[MOL_MAX_ATOMS][3], XO[MOL_MAX_ATOMS][3], V[MOL_MAX_ATOMS][3];
    extern __shared__ unsigned long long mol_tab[];
    const int r = blockIdx.x, k = k0 + r, a = threadIdx.x, n = m.n;
    if (only && !only[k]) return;
    MolShared ms;
    mol_stage(m, (unsigned char *)mol_tab, ms);
    // the dynamics' term tables and the slots of their force contributions, behind the other tables
    unsigned char *tb = (unsigned char *)mol_tab + m.shared_bytes;
    for (int q = threadIdx.x * 8; q < m.terms_bytes; q += 32 * MOL_WARPS * 8) *(unsigned long long *)(tb + q) = *(const unsigned long long *)((const unsigned char *)m.terms + q);
    float (*FS)[3] = (float (*)[3])(tb + ((m.terms_bytes + 15) & ~15));
    __syncthreads();
    const int *g_off = (const int *)(tb + ((const MolTerms *)tb)->o_goff);
    const bool active = a < n;
    const StateDev st = states[perm[k]];
    const double mass = active ? m.mass[a] : 1.0, sg = sqrt(st.kT / mass);
    const double inv_mt = 1.0 / mol_warp_sum(active ? mass : 0.0);
    if (active) {
        for (int c = 0; c < 3; c++) { X[a][c] = pos[((size_t)r * n + a) * 3 + c]; V[a][c] = vel[((size_t)r * n + a) * 3 + c]; }
        if (reassign) {   // context.setVelocitiesToTemperature, mcmc.py:711
            const float3 g = philox_normal3(philox4x32_10(make_uint4(a, 0x80000000u, k, iteration), key));
            V[a][0] = sg * g.x; V[a][1] = sg * g.y; V[a][2] = sg * g.z;
        }
    }
    MolCluster kc;
    MolStar ks;
    kc.nc = 0;
    const bool has_c = a < m.n_clusters;
    if (has_c) { if (STAR) mol_star_load(m, a, ks); else mol_load_cluster(m, a, kc); }
    __syncwarp();
    // incoming velocities obey the constraints
    if (has_c) { if (STAR) { mol_star_init(ks, X); mol_star_rattle(ks, V); } else mol_rattle_cluster(m, a, kc, X, V); }
    __syncwarp();
    const double inv_mass = 1.0 / mass;
    // (the program is interpreted, so the compiler does not hoist these out of the step loop: two f64 divisions per R)
    const double hm = (double)p.mv.dt_d / p.mv.nV * inv_mass, h = (double)p.mv.dt_d / p.mv.nR, inv_h = 1.0 / h;
    double f[3] = {0, 0, 0};
    bool f_valid = false;
    uint32_t ocount = 0;
    for (int s = 0; s < p.mv.n_steps; s++) {
        if (m.remove_cm) {
            double px = mol_warp_sum(active ? mass * V[a][0] : 0.0), py = mol_warp_sum(active ? mass * V[a][1] : 0.0),
                   pz = mol_warp_sum(active ? mass * V[a][2] : 0.0);
            if (active) { V[a][0] -= px * inv_mt; V[a][1] -= py * inv_mt; V[a][2] -= pz * inv_mt; }
            __syncwarp();
        }
        for (int q = 0; q < p.mv.n_prog; q++) {
            const char op = p.mv.prog[q];
            if (op == 'V') {
                if (!f_valid) {
                    __syncthreads();   // warp 0's positions are in shared memory
                    mol_forces_terms(m, tb, X, FS);
                    __syncthreads();   // every term's contributions are in their slots
                    if (active) {   // this atom's slots, in slot order
                        float fx = 0.f, fy = 0.f, fz = 0.f;
                        for (int q = g_off[a]; q < g_off[a + 1]; q++) { fx += FS[q][0]; fy += FS[q][1]; fz += FS[q][2]; }
                        f[0] = fx; f[1] = fy; f[2] = fz;
                    }
                    __syncwarp();
                    f_valid = true;
                }
                if (active) for (int c = 0; c < 3; c++) V[a][c] += hm * f[c];
                __syncwarp();
                if (has_c) { if (STAR) mol_star_rattle(ks, V); else mol_rattle_cluster(m, a, kc, X, V); }
                __syncwarp();
            } else if (op == 'R') {
                double xu[3] = {0, 0, 0};
                if (active) for (int c = 0; c < 3; c++) { XO[a][c] = X[a][c]; X[a][c] += h * V[a][c]; xu[c] = X[a][c]; }
                __syncwarp();
                if (m.n_clusters) {
                    if (has_c) { if (STAR) mol_star_shake(m, ks, X); else mol_shake_cluster(m, a, kc, XO, X); }
                    __syncwarp();
                    if (active) for (int c = 0; c < 3; c++) V[a][c] += (X[a][c] - xu[c]) * inv_h;
                    __syncwarp();
                    if (has_c) { if (STAR) mol_star_rattle(ks, V); else mol_rattle_cluster(m, a, kc, X, V); }
                    __syncwarp();
                }
                f_valid = false;
            } else {   // 'O'
                if (active) {
                    const float3 g = philox_normal3(philox4x32_10(make_uint4(a, ocount, k, iteration), key));
                    V[a][0] = p.mv.a_d * V[a][0] + p.mv.b_d * sg * (double)g.x;
                    V[a][1] = p.mv.a_d * V[a][1] + p.mv.b_d * sg * (double)g.y;
                    V[a][2] = p.mv.a_d * V[a][2] + p.mv.b_d * sg * (double)g.z;
                }
                ocount++;
                __syncwarp();
                if (has_c) { if (STAR) mol_star_rattle(ks, V); else mol_rattle_cluster(m, a, kc, X, V); }
                __syncwarp();
            }
        }
    }
    const double U = mol_warp_sum(active ? mol_atom<true, double>(ms, X, a, nullptr) : 0.0);
    const double KE = mol_warp_sum(active ? 0.5 * mass * (V[a][0] * V[a][0] + V[a][1] * V[a][1] + V[a][2] * V[a][2]) : 0.0);
    const bool bad = active && !(isfinite(X[a][0]) && isfinite(X[a][1]) && isfinite(X[a][2]) && isfinite(V[a][0]) &&
                                 isfinite(V[a][1]) && isfinite(V[a][2]));
    const unsigned any_bad = __ballot_sync(0xffffffffu, bad);
    if (a == 0) { pot[k] = U + st.offset; kin[k] = KE; nan_flag[k] = (any_bad || !isfinite(U)) ? 1 : 0; }
    if (active)
        for (int c = 0; c < 3; c++) { pos[((size_t)r * n + a) * 3 + c] = X[a][c]; vel[((size_t)r * n + a) * 3 + c] = V[a][c]; }
}

// MultiStateSampler.minimize (multistatesampler.py:611-647) for a molecule: FIRE descent on the constraint manifold.  The
// force is projected onto the manifold (components along the constrained bonds removed: the RATTLE solve with unit
// weights), the move is followed by SHAKE, the FIRE velocity is kept tangent.  Converged when the RMS of the projected force
// falls below tol_rms (kJ/mol/nm); f64 throughout.  (OpenMM's L-BFGS is not reproduced, as for the other systems.)
__global__ void __launch_bounds__(32) k_minimize_mol(MolDev m, double *__restrict__ pos, int k0, double tol_rms, int max_iter,
                                                     double *__restrict__ rms_out, int *__restrict__ iters_out) {
    __shared__ double X[MOL_MAX_ATOMS][3], XO[MOL_MAX_ATOMS][3], V[MOL_MAX_ATOMS][3], F[MOL_MAX_ATOMS][3];
    extern __shared__ unsigned long long mol_tab[];
    const int r = blockIdx.x, k = k0 + r, a = threadIdx.x, n = m.n;
    const bool active = a < n;
    MolShared ms;
    mol_stage(m, (unsigned char *)mol_tab, ms);
    MolCluster kc, ku;   // the cluster with its masses (SHAKE) and with unit weights (projections)
    kc.nc = ku.nc = 0;
    if (a < m.n_clusters) {
        mol_load_cluster(m, a, kc);
        ku = kc;
#pragma unroll
        for (int c = 0; c < MOL_MAXC; c++) { const bool on = c < ku.nc; ku.wi[c] = on ? 1.0 : 0.0; ku.wj[c] = on ? 1.0 : 0.0; }
#pragma unroll
        for (int c = 0; c < MOL_MAXC; c++)
#pragma unroll
            for (int d = 0; d < MOL_MAXC; d++) {
                double v = 0.0;
                if (ku.i[c] == ku.i[d]) v += ku.wi[c];
                if (ku.i[c] == ku.j[d]) v -= ku.wi[c];
                if (ku.j[c] == ku.i[d]) v -= ku.wj[c];
                if (ku.j[c] == ku.j[d]) v += ku.wj[c];
                ku.coup[c][d] = v;
            }
    }
    if (active) for (int c = 0; c < 3; c++) { X[a][c] = pos[((size_t)r * n + a) * 3 + c]; V[a][c] = 0.0; }
    __syncwarp();
    const double dt0 = 0.001, dt_max = 0.010, alpha0 = 0.1, max_move = 0.01;   // (as k_minimize)
    double dt = dt0, alpha = alpha0, rms = 0.0;
    int n_pos = 0, it = 0;
    for (;; it++) {
        double f[3] = {0, 0, 0};
        if (active) mol_atom<false, double>(ms, X, a, f);
        if (active) for (int c = 0; c < 3; c++) F[a][c] = f[c];
        __syncwarp();
        if (a < m.n_clusters && ku.nc <= MOL_MAXC) mol_rattle_cluster(m, a, ku, X, F);   // projected force
        __syncwarp();
        if (active) for (int c = 0; c < 3; c++) f[c] = F[a][c];
        const double FF = mol_warp_sum(active ? f[0] * f[0] + f[1] * f[1] + f[2] * f[2] : 0.0);
        rms = sqrt(FF / (3.0 * n));
        if (!(rms > tol_rms) || it >= max_iter) break;   // converged, out of iterations, or NaN
        double v[3] = {active ? V[a][0] : 0.0, active ? V[a][1] : 0.0, active ? V[a][2] : 0.0};
        const double P = mol_warp_sum(f[0] * v[0] + f[1] * v[1] + f[2] * v[2]);
        const double VV = mol_warp_sum(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
        if (P > 0.0) {
            const double mix = alpha * sqrt(VV / fmax(FF, 1e-300));
            for (int c = 0; c < 3; c++) v[c] = (1.0 - alpha) * v[c] + mix * f[c];
            if (++n_pos > 5) { dt = fmin(dt * 1.1, dt_max); alpha *= 0.99; }
        } else {
            v[0] = v[1] = v[2] = 0.0; dt *= 0.5; alpha = alpha0; n_pos = 0;
        }
        const double inv_m = active ? 1.0 / m.mass[a] : 0.0;
        for (int c = 0; c < 3; c++) v[c] += dt * f[c] * inv_m;
        double mv[3] = {dt * v[0], dt * v[1], dt * v[2]};
        const double m2 = mv[0] * mv[0] + mv[1] * mv[1] + mv[2] * mv[2];
        if (m2 > max_move * max_move) {   // displacement cap: rescale this atom's velocity
            const double sc = max_move / sqrt(m2);
            for (int c = 0; c < 3; c++) { v[c] *= sc; mv[c] *= sc; }
        }
        if (active) for (int c = 0; c < 3; c++) { XO[a][c] = X[a][c]; X[a][c] += mv[c]; V[a][c] = v[c]; }
        __syncwarp();
        if (a < m.n_clusters) mol_shake_cluster(m, a, kc, XO, X);
        __syncwarp();
        if (a < m.n_clusters && ku.nc <= MOL_MAXC) mol_rattle_cluster(m, a, ku, X, V);   // velocity stays tangent
        __syncwarp();
    }
    if (a == 0) { rms_out[k] = rms; iters_out[k] = it; }
    if (active) for (int c = 0; c < 3; c++) pos[((size_t)r * n + a) * 3 + c] = X[a][c];
}

// u[k][l] = beta_l (U(x_k) + offset_l): the states of a molecule differ in temperature only (parallel tempering,
// paralleltempering.py:175-237: one potential evaluation per replica, scaled by beta_l).
__global__ void __launch_bounds__(32) k_energy_mol(MolDev m, const StateDev *__restrict__ states, int n_states,
                                                   const double *__restrict__ pos, int k0, double *__restrict__ u_out) {
    __shared__ double X[MOL_MAX_ATOMS][3];
    extern __shared__ unsigned long long mol_tab[];
    const int r = blockIdx.x, k = k0 + r, a = threadIdx.x, n = m.n;
    const bool active = a < n;
    MolShared ms;
    mol_stage(m, (unsigned char *)mol_tab, ms);
    if (active) for (int c = 0; c < 3; c++) X[a][c] = pos[((size_t)r * n + a) * 3 + c];
    __syncwarp();
    const double U = mol_warp_sum(active ? mol_atom<true, double>(ms, X, a, nullptr) : 0.0);
    for (int l = a; l < n_states; l += 32) u_out[(size_t)k * n_states + l] = states[l].beta * (U + states[l].offset);
}

__global__ void k_randomize_velocities_mol(MolDev m, const StateDev *__restrict__ states, const int *__restrict__ perm,
                                           double *__restrict__ vel, int k0, uint2 key, uint32_t stream_id) {
    const int r = blockIdx.x, k = k0 + r, a = threadIdx.x;
    if (a >= m.n) return;
    const StateDev st = states[perm[k]];
    const double sv = sqrt(st.kT / m.mass[a]);
    const float3 g = philox_normal3(philox4x32_10(make_uint4(a, 0xC0000000u, k, stream_id), key));
    vel[((size_t)r * m.n + a) * 3 + 0] = sv * g.x;
    vel[((size_t)r * m.n + a) * 3 + 1] = sv * g.y;
    vel[((size_t)r * m.n + a) * 3 + 2] = sv * g.z;
}

__global__ void k_restore_failed_mol(const int *__restrict__ nan_flag, int *__restrict__ retry, int k0, int N,
                                     const double *__restrict__ pos_snap, const double *__restrict__ vel_snap,
                                     double *__restrict__ pos, double *__restrict__ vel) {
    const int r = blockIdx.x, k = k0 + r;
    const int failed = nan_flag[k];
    if (threadIdx.x == 0) retry[k] = failed;
    if (!failed) return;
    for (int q = threadIdx.x; q < 3 * N; q += blockDim.x) {
        pos[(size_t)r * N * 3 + q] = pos_snap[(size_t)r * N * 3 + q];
        vel[(size_t)r * N * 3 + q] = vel_snap[(size_t)r * N * 3 + q];
    }
}

