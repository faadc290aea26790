// rx_walk2.cuh -- second-generation swap-all walker for power-of-two K <= 256 (included by rx_mix.cu).
//
// Same algorithm and the same results as k_mix_walk_pow2<true> (replicaexchange.py:321-349 bit for bit); what
// changes is the length of the dependent chain of one speculation round:
//   * lane <-> slot mapping is FIXED (lane = slot mod 32) and the window [h, h+32) rotates over the lanes, so a lane
//     keeps its slot record in registers until the slot leaves the window and the record of its next slot (s + 32)
//     is prefetched a whole window ahead: no shared-memory ring access on the chain (v1: LDS ring -> LDS perm -> LDS
//     image; here: LDS perm -> LDS image).  Ballots are rotated into window order with one funnel shift;
//   * records are 16 bytes {i|j<<16, back-mask, f32 log-uniform of the NEXT slot, alternatives}; the f64 log-uniform the
//     exact path needs is recomputed from the two words of the stream (same log() as the pre-pass, same value);
//   * the commit's bookkeeping (log entry, counters, promotion of the lanes that left the window) is issued after the
//     next round's permutation loads, in their latency shadow;
//   * a second warp turns the records into ready-to-use slot contexts in a shared-memory ring (release/acquire fence
//     patterns on its two control words): the walker's round is bound by its instruction count, not by latency.
// The kernel runs the bulk of a pass; the last < 600 slots / < 130 attempts of a pass are left to
// k_mix_walk_pow2<true>, which reads the same records.
#pragma once

struct SlotRec2 {        // 16 bytes, one 2-word slot of the stream, state independent
    uint32_t ij;         // i | j << 16
    uint32_t backmask;   // bit 31-b: slot s-1-b shares a replica index with slot s (b = 0..30)
    uint32_t lu_next;    // float bits: log of the uniform the two words of slot s+1 would produce, rounded to f32
    uint32_t alts;       // a1_i | a1_j << 8: partner of i (of j) in the most recent earlier slot that touches it (else itself)
};

#define W2_LOOKBACK 48

// f64 log-uniform of slot s, exactly as k_slots_build / k_slots_build2 compute it
__device__ __forceinline__ double slot_logU(const uint32_t *__restrict__ words, unsigned s) {
    const double U = mt_double(words[2 * (size_t)s], words[2 * (size_t)s + 1]);
    return (U == 0.0) ? LOGU_ZERO : log(U);
}

__global__ void __launch_bounds__(256) k_slots_build2(const uint32_t *__restrict__ words, long long nslots, uint32_t mask,
                                                      SlotRec2 *__restrict__ rec) {
    __shared__ uint32_t s_ij[256 + W2_LOOKBACK];
    const long long s0 = (long long)blockIdx.x * 256;
    const int t = threadIdx.x;
    for (int q = t; q < 256 + W2_LOOKBACK; q += 256) {   // tile: slots s0-48 .. s0+255
        const long long s = s0 - W2_LOOKBACK + q;
        uint32_t ij = 0xffffffffu;
        if (s >= 0 && s < nslots) ij = (words[2 * s] & mask) | ((words[2 * s + 1] & mask) << 16);
        s_ij[q] = ij;
    }
    __syncthreads();
    const long long s = s0 + t;
    if (s >= nslots) return;
    const uint32_t ij = s_ij[t + W2_LOOKBACK];
    const uint32_t i = ij & 0xffffu, j = ij >> 16;
    uint32_t bm = 0, a1i = i, a1j = j;
    bool fi = false, fj = false;
#pragma unroll 4
    for (int b = 0; b < W2_LOOKBACK - 1; b++) {
        const uint32_t o = s_ij[t + W2_LOOKBACK - 1 - b];
        const uint32_t oi = o & 0xffffu, oj = o >> 16;
        const bool valid = (o != 0xffffffffu);
        if (b < 31) {
            const bool hit = valid && (oi == i || oi == j || oj == i || oj == j);
            bm |= (hit ? 1u : 0u) << (31 - b);
        }
        if (valid && oi != oj) {   // a slot with i == j never changes the permutation
            if (!fi && (oi == i || oj == i)) { a1i = (oi == i) ? oj : oi; fi = true; }
            if (!fj && (oi == j || oj == j)) { a1j = (oi == j) ? oj : oi; fj = true; }
        }
    }
    SlotRec2 r;
    r.ij = ij;
    r.backmask = bm;
    float lu = 0.f;
    if (s + 1 < nslots) lu = (float)slot_logU(words, (unsigned)(s + 1));
    r.lu_next = __float_as_uint(lu);
    r.alts = (a1i & 0xffu) | ((a1j & 0xffu) << 8);
    rec[s] = r;
}

// The filter's decision for one (i, j, si, sj): image values d_x = image of u[x, s_x] - rowmin_x (the maintained diagonal)
// and f_xy = image of u[x, s_y] - rowmin_x.  Same rigorous bound as k_mix_walk_pow2<true> (see its derivation there;
// the factor 3.2e-5 leaves 5 % over the 2^-15 + 2^-23 the roundings need, far more than the re-association below costs):
//   e0  = 3.2e-5 (|d_i| + |d_j|) + eps0        as soon as the states are known (before the image loads return),
//   eps = 3.2e-5 (|f_ij| + |f_ji|) + e0,       lp = (d_i - f_ij) + (d_j - f_ji),
//   log_p >= 0 is certain iff lp > eps; it is certainly < 0 iff lp < -eps; the comparison with the uniform is certain
//   iff |lp - lu| > mar = 1.3e-7 (|lp| + |lu|) + eps.
// eps0 = rowabs[i] + rowabs[j] + 1e-9, or -1e30 for a slot with i == j: the reference's log_p is then exactly 0 for finite
// energies (accepted without a draw) and lp is exactly 0 > eps; non-finite energies give lp = NaN (undecided: exact path).
__device__ __forceinline__ void w2_filter(float d_i, float f_ij, float d_j, float f_ji, float e0, float lu,
                                          bool &ge0, bool &acc, bool &undecided) {
    const float lp = (d_i - f_ij) + (d_j - f_ji);
    const float eps = fmaf(fabsf(f_ij) + fabsf(f_ji), 3.2e-5f, e0);
    ge0 = lp > eps;
    const float d = lp - lu;
    const float mar = fmaf(fabsf(lp) + fabsf(lu), 1.3e-7f, eps);
    const bool dec_lp = fabsf(lp) > eps;
    acc = ge0 || (dec_lp && d > mar);
    undecided = !(ge0 || (dec_lp && fabsf(d) > mar));
}

// One entry per replica k: the walker's view of the permutation.  `diag` is the image value of u[k, state] - rowmin_k, so
// a round reads the two diagonal terms of log_p together with the states (one dependent shared-memory level less) and
// only the two off-diagonal image values afterwards.  8 bytes: two wavefronts per warp-wide access at best.
struct __align__(8) W2Replica {
    int state;
    float diag;
};

__device__ __forceinline__ float w2_image(const unsigned short *__restrict__ s_qhi, const unsigned char *__restrict__ s_qlo, unsigned a) {
    return __uint_as_float(__byte_perm((unsigned)s_qhi[a], (unsigned)s_qlo[a], 0x1045));   // (hi << 16) | (lo << 8)
}

// Shared-memory accesses of the round loop by explicit 32-bit shared addresses.  (With generic pointers the compiler
// re-derives the shared window base from SR_CgaCtaId inside the loop -- an S2UR of a few hundred cycles on the chain.)
__device__ __forceinline__ uint2 w2_lds64(unsigned a) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ float w2_lds_f32(unsigned a) {   // (read-only table)
    float v;
    asm("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint4 w2_lds128(unsigned a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ uint4 w2_lds128_ctx(unsigned a) {   // ring contexts inside the round loop: published before the loop
    uint4 v;                                                    // was (re-)entered, not written again while they are in use
    asm("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ void w2_sts64(unsigned a, unsigned x, unsigned y) {
    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(a), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ unsigned w2_lds32(unsigned a) {
    unsigned v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
    return v;
}
__device__ __forceinline__ float w2_image_at(unsigned a_hi, unsigned a_lo) {   // the image is read-only while the walker runs
    unsigned hi, lo;
    asm("ld.shared.u16 %0, [%1];" : "=r"(hi) : "r"(a_hi));
    asm("ld.shared.u8 %0, [%1];" : "=r"(lo) : "r"(a_lo));
    return __uint_as_float(__byte_perm(hi, lo, 0x1045));
}

// The walker's record ring: 16 entries per lane (= per slot class mod 32), filled by the lane itself with asynchronous
// global->shared copies 15 windows ahead of use (no register, no scoreboard wait; DRAM latency is far below that);
// completion is tracked by the hardware (cp.async.wait_group): no flags, no fences, no second warp in the loop.
// (A producer warp that prepared ready-to-use contexts was tried: 106 instead of 125 instructions per round for the
// walker, but its shared-memory traffic and the acquire/release pairs made the walker's own loads wait twice as long --
// 210-260 ns per round against 177 ns for this organisation.)
#define W2_RING 512
__device__ __forceinline__ void w2_cp_async16(unsigned dst, const void *src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void w2_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void w2_cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// The exact decision for the attempt of slot s under the states (si, sj): bit 0 = log_p >= 0, bit 1 = accepted.  f64
// energies from L2, the reference's own arithmetic; the uniform is compared in the log domain outside a 1e-9 band and as
// U < exp(log_p) inside it.
__device__ __noinline__ unsigned w2_exact_decision(const SlotRec2 *__restrict__ rec, const uint32_t *__restrict__ words,
                                                   const double *__restrict__ u, unsigned s, unsigned si, unsigned sj, int logK) {
    const unsigned ij = rec[s].ij;
    const unsigned rowi = (ij & 0xffffu) << logK, rowj = (ij >> 16) << logK;
    const double logp = swap_logp(u[rowi | sj], u[rowj | si], u[rowi | si], u[rowj | sj]);
    if (logp >= 0.0) return 3u;
    const unsigned s1 = s + 1;
    const double dd = logp - slot_logU(words, s1);
    bool acc;
    if (dd > 1e-9) acc = true;
    else if (dd < -1e-9) acc = false;
    else acc = mt_double(words[2 * (size_t)s1], words[2 * (size_t)s1 + 1]) < rx_exp_cr(logp);
    return acc ? 2u : 0u;
}

// The image is re-laid out row by row in shared memory -- u16 plane of the row (2K bytes), then its u8 plane (K bytes) --
// so that one address per row serves both planes.
#define W2_THREADS 128   // warps 1.. only help with the prologue
__global__ void __launch_bounds__(W2_THREADS) k_mix_walk2(const SlotRec2 *__restrict__ rec, const uint32_t *__restrict__ words,
                                                  unsigned nslots, const double *__restrict__ u, int K, int logK,
                                                  int *__restrict__ perm_g, uint32_t *__restrict__ slot_log,
                                                  const unsigned char *__restrict__ filt,
                                                  const double *__restrict__ filt_rowabs, MixCtl *ctl) {
    extern __shared__ uint4 s_w2[];
    __shared__ unsigned long long s_ptrs[2];               // global base pointers of the round loop (see there)
    uint4 *s_ring = s_w2;                                  // [W2_RING] slot records
    W2Replica *s_rep = (W2Replica *)(s_ring + W2_RING);    // [K]
    unsigned char *s_q = (unsigned char *)(s_rep + K);     // image rows, 3K bytes each
    // (the warp index through a shuffle: the compiler then knows that it is the same in all lanes, and neither guards the
    // walker's ballots against divergence nor builds its loop with divergence-capable -- slowly resolved -- branches)
    const int tid = threadIdx.x, lane = tid & 31, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    {
        const unsigned short *ghi = (const unsigned short *)filt;
        const unsigned char *glo = filt + 2 * (size_t)K * K;
        if (K >= 16) {   // 16-byte pieces: 8 values of the u16 plane, 16 of the u8 plane, never across a row
            const uint4 *ghi4 = (const uint4 *)ghi, *glo4 = (const uint4 *)glo;   // (cudaMalloc alignment, 2 K^2 % 16 == 0)
            for (int q = tid; q < (K * K) / 8; q += W2_THREADS) {
                const int e = q * 8, row = e >> logK, col = e & (K - 1);
                *(uint4 *)(s_q + (size_t)3 * K * row + 2 * col) = ghi4[q];
            }
            for (int q = tid; q < (K * K) / 16; q += W2_THREADS) {
                const int e = q * 16, row = e >> logK, col = e & (K - 1);
                *(uint4 *)(s_q + (size_t)3 * K * row + 2 * K + col) = glo4[q];
            }
        } else {
            for (int q = tid; q < K * K; q += W2_THREADS) {
                const int row = q >> logK, col = q & (K - 1);
                unsigned char *rowp = s_q + (size_t)3 * K * row;
                ((unsigned short *)rowp)[col] = ghi[q];
                rowp[2 * K + col] = glo[q];
            }
        }
    }
    if (tid == 0) { s_ptrs[0] = (unsigned long long)__cvta_generic_to_global(slot_log); s_ptrs[1] = (unsigned long long)rec; }
    __syncthreads();
    float rowabs_max = 0.f;
    for (int q = tid; q < K; q += W2_THREADS) {
        W2Replica e;
        e.state = perm_g[q];
        const unsigned char *rowp = s_q + (size_t)3 * K * q;
        e.diag = __uint_as_float(__byte_perm((unsigned)((const unsigned short *)rowp)[e.state], (unsigned)rowp[2 * K + e.state], 0x1045));
        s_rep[q] = e;
    }
    // the rows' share of the filter's rounding bound, the largest of all rows (rounded up; K values, read by every warp)
    for (int q = lane; q < K; q += 32)
        rowabs_max = fmaxf(rowabs_max, __fmul_ru(1.6e-14f, __fadd_ru(__double2float_ru(fabs(filt_rowabs[q])), 0.5f)));
    for (int o = 16; o; o >>= 1) rowabs_max = fmaxf(rowabs_max, __shfl_xor_sync(0xffffffffu, rowabs_max, o));
    const float eps_rows = __fadd_ru(__fadd_ru(rowabs_max, rowabs_max), 1e-9f);
    __syncthreads();
    if (warp != 0) return;
    const uint4 *__restrict__ recs = (const uint4 *)rec;

    const unsigned head0 = (unsigned)ctl->head;
    unsigned h = head0;
    const long long remaining0 = ctl->remaining;
    unsigned rem = remaining0 > 0x7fffffffLL ? 0x7fffffffu : (unsigned)remaining0;
    const unsigned rem0 = rem;
    unsigned rounds = 0, slow = 0;
    // a round may start while h + 99 <= h_end: its lanes copy the records of slots up to h + 31 + 32 + 480 into the ring
    const unsigned h_end = nslots >= 1200u ? nslots - 560u : 0u;
    if (rem >= 130 && nslots >= 1200u && h + 99u <= h_end) {
        // 32-bit shared addresses (through a shuffle, so that they live in registers instead of being re-derived)
        const unsigned ring_base = __shfl_sync(0xffffffffu, (unsigned)__cvta_generic_to_shared((const void *)s_ring), 0);
        const unsigned rep_base = __shfl_sync(0xffffffffu, (unsigned)__cvta_generic_to_shared((const void *)s_rep), 0);
        const unsigned img_base = __shfl_sync(0xffffffffu, (unsigned)__cvta_generic_to_shared((const void *)s_q), 0);
        const unsigned row_bytes = 3u * (unsigned)K, lo_off = 2u * (unsigned)K;
        unsigned r = h & 31u;                           // lane of window position 0
        unsigned w = ((unsigned)lane - h) & 31u;        // this lane's window position
        unsigned sA = h + w;                            // this lane's slot
        // (the two global base pointers of the loop as opaque register values: taken from the constant bank where they are
        // used, each use would wait for an LDC)
        // (read back from shared memory by a volatile load: nothing the compiler can re-derive)
        const uint2 pl = w2_lds64((unsigned)__cvta_generic_to_shared((const void *)&s_ptrs[0]));
        const uint2 pr = w2_lds64((unsigned)__cvta_generic_to_shared((const void *)&s_ptrs[1]));
        const unsigned long long slot_log_r = ((unsigned long long)pl.y << 32) | pl.x;
        const uint4 *recs_r = (const uint4 *)(((unsigned long long)pr.y << 32) | pr.x);
        // slot contexts: A = the lane's slot, B = its next slot, one window later (its raw record is loaded a round ahead):
        // back-mask, f32 log-uniform of the following slot, the filter bound's constant term (-1e30 when i == j),
        // all-ones if i != j, shared addresses of the image rows and of the replica entries of i and j
        unsigned bmA, neqA, rowiA, rowjA, repiA, repjA;
        float luA, epsA;
        // of the next slot only what the commit needs at once is prepared a round ahead: its indices and the addresses of
        // its replica entries; the rest of its context is derived when (and only in the lanes where) the slot is entered
        unsigned iB, jB, repiB, repjB;
        auto ahead = [&](const uint4 q) {
            iB = q.x & 0xffffu; jB = q.x >> 16;
            repiB = rep_base + (iB << 3); repjB = rep_base + (jB << 3);
        };
        auto derive = [&](const uint4 q, unsigned &bm, float &lu, float &eps, unsigned &neq, unsigned &rowi, unsigned &rowj,
                          unsigned &repi, unsigned &repj) {
            const unsigned i = q.x & 0xffffu, j = q.x >> 16;
            bm = q.y; lu = __uint_as_float(q.z);
            neq = i != j ? 0xffffffffu : 0u;
            eps = i != j ? eps_rows : -1e30f;
            rowi = img_base + i * row_bytes; rowj = img_base + j * row_bytes;
            repi = rep_base + (i << 3); repj = rep_base + (j << 3);
        };
        // ring entry of slot s: s mod W2_RING; this lane owns the entries of its class (s mod 32)
        for (unsigned k = 0; k < 16u; k++) w2_cp_async16(ring_base + (((sA + 32u * k) & (W2_RING - 1)) << 4), recs + (sA + 32u * k));
        w2_cp_async_commit();
        w2_cp_async_wait<0>();
        __syncwarp();
        derive(w2_lds128(ring_base + ((sA & (W2_RING - 1)) << 4)), bmA, luA, epsA, neqA, rowiA, rowjA, repiA, repjA);
        unsigned ridxB = (sA + 32u) & (W2_RING - 1);   // ring entry of the next slot
        uint4 qB = w2_lds128(ring_base + (ridxB << 4));
        ahead(qB);
        uint2 ei = w2_lds64(repiA), ej = w2_lds64(repjA);   // {state, diag} of both replicas
        // what the round resolved last leaves to the next block: the committed window positions, the positions that leave
        // the window, all-ones if this lane's attempt changes the permutation, its log entry
        unsigned p_cm = 0, p_below = 0, p_chg = 0, p_entry = 0;
        float f_ij = 0.f, f_ji = 0.f;
        // Commit the round described by the p_* values, slide the window and fetch the states of the next round:
        // permutation stores, at once the next round's loads, then the lane state.
        auto commit = [&]() {
            // the window advances by the number of positions that leave it (computed here rather than where `below` appears,
            // at the end of the previous block: a population count is a long-latency operation whose scoreboard slot would
            // otherwise be waited for at the loop's back edge)
            const unsigned p_advance = (unsigned)__popc(p_below);
            const unsigned bit = 1u << w;
            const bool p_mine = (p_cm & bit) != 0u;
            const bool p_swaps = (p_cm & bit & p_chg) != 0u;
            const bool p_promoted = (p_below & bit) != 0u;
            if (p_swaps) {   // replica i takes state sj: its new diagonal value is the off-diagonal one just read
                w2_sts64(repiA, ej.x, __float_as_uint(f_ij));
                w2_sts64(repjA, ei.x, __float_as_uint(f_ji));
            }
            __syncwarp();
            // the states of the next round: of the next slot for the lanes that leave the window
            const uint2 ein = w2_lds64(p_promoted ? repiB : repiA), ejn = w2_lds64(p_promoted ? repjB : repjA);
            if (p_mine)   // sparse commit log, indexed by slot (zero = no attempt)
                asm volatile("st.global.u32 [%0], %1;" ::"l"(slot_log_r + 4ull * sA), "r"(p_entry) : "memory");
            if (p_promoted) {
                bmA = qB.y; luA = __uint_as_float(qB.z);
                neqA = iB != jB ? 0xffffffffu : 0u;
                epsA = iB != jB ? eps_rows : -1e30f;
                rowiA = img_base + iB * row_bytes; rowjA = img_base + jB * row_bytes;
                repiA = repiB; repjA = repjB;
                sA += 32u;
                w2_cp_async16(ring_base + (((ridxB - 32u) & (W2_RING - 1)) << 4), recs_r + (sA + 480u));   // over the entry of the slot just left
                ridxB = (ridxB + 32u) & (W2_RING - 1);
            }
            w2_cp_async_commit();
            // the record of the (possibly new) next slot: the lanes that stay re-read the one they hold
            qB = w2_lds128(ring_base + (ridxB << 4));
            h += p_advance;
            r = (r + p_advance) & 31u;
            rem -= __popc(p_cm);
            ei = ein;
            ej = ejn;
            w = (w - p_advance) & 31u;
        };
        unsigned Cw = 0;
        // Exact decisions injected into ONE fast round (see the rare path below): `bias` joins the lane's log_p, `luA` is
        // replaced, so that the filter reproduces the exact answer; both are restored when that round has been resolved.
        float bias = 0.f, lu_saved = 0.f;
        bool injected = false;
        for (;;) {
            // ---------------- the budget and the end of the pass, every 64 rounds at most: a round commits at most 32
            // attempts and advances at most 32 slots (the round resolved last stays pending across this step)
            if (rem < 130u || h + 99u > h_end) break;
            unsigned quota = min(min((rem - 97u) >> 5, (h_end - h - 66u) >> 5), injected ? 1u : 64u);
            // ---------------- fast rounds.  The loop is rotated: an iteration COMMITS the round resolved by the previous
            // one and then evaluates and resolves the next, so that the block begins with the dependent chain (stores ->
            // state loads -> image loads -> filter -> ballots); no data-dependent branch besides the loop's.
            do {
                commit();
                rounds++;
                const unsigned si = ei.x, sj = ej.x;
                f_ij = w2_image_at(rowiA + 2u * sj, rowiA + lo_off + sj);
                f_ji = w2_image_at(rowjA + 2u * si, rowjA + lo_off + si);
                const float e0 = fmaf(fabsf(__uint_as_float(ei.y)) + fabsf(__uint_as_float(ej.y)), 3.2e-5f, epsA);
                w2_cp_async_wait<8>();   // a copy is used 15 of the lane's promotions (at least 15 rounds) after it was issued
                ahead(qB);
                bool ge0, acc, undecided;
                w2_filter(__uint_as_float(ei.y), f_ij, __uint_as_float(ej.y) + bias, f_ji, e0, luA, ge0, acc, undecided);
                const unsigned und = undecided ? 1u : 0u;
                const bool changes = acc && neqA != 0u;
                const unsigned G = __ballot_sync(0xffffffffu, ge0);
                const unsigned A = __ballot_sync(0xffffffffu, changes);
                const unsigned Gw = __funnelshift_r(G, G, r), Aw = __funnelshift_r(A, A, r);   // window order
                // visited chain (see k_mix_walk_pow2): skip[s+1] = NG[s] & ~skip[s]
                const unsigned X = ~Gw;
                const unsigned starts = X & ~(X << 1);
                const unsigned SE = starts & 0x55555555u, SO = starts & 0xAAAAAAAAu;
                const unsigned sumE = X + SE, sumO = X + SO;
                const unsigned skip = (((sumE ^ X) & ~SE) & 0xAAAAAAAAu) | (((sumO ^ X) & ~SO) & 0x55555555u);
                const unsigned V = ~skip;
                const unsigned VA = V & Aw;
                unsigned earlier;   // bit 31-b: window position w-1-b is a visited state-changing swap
                asm("shl.b32 %0, %1, %2;" : "=r"(earlier) : "r"(VA), "r"(32u - w));
                // A round ends before the first visited lane that is stale -- or that the filter could not decide -- and
                // before the last window position when its attempt draws a uniform (log_p < 0): that uniform's slot lies
                // beyond the window, and committing it here would make the window advance by 33 (the lane of the skipped
                // slot would have to move on by two windows at once); the attempt simply opens the next round instead.
                const unsigned C = __ballot_sync(0xffffffffu, ((earlier & bmA) | und) != 0u);
                Cw = (__funnelshift_r(C, C, r) | (X & 0x80000000u)) & V;
                const unsigned low = Cw & (0u - Cw);
                const unsigned below = low - 1u;       // low == 0 -> all lanes
                p_cm = V & below; p_below = below; p_chg = changes ? 0xffffffffu : 0u;
                p_entry = (sj * (1u << LOG_STATE_BITS) + si) | (acc ? (1u << 31) | (1u << LOG_ACC_BIT) : (1u << 31));
                // (position 0 is always visited: nothing commits iff it is itself the lane that ends the round)
            } while (--quota != 0u && (Cw & 1u) == 0u);
            // (a no-op unless the round just resolved ran alone, with injected decisions: see below)
            const bool was_injected = injected;
            luA = was_injected ? lu_saved : luA;
            bias = 0.f;
            injected = false;
            if ((Cw & 1u) == 0u) continue;
            commit();   // (nothing to commit: positions the lanes on the round that could not start)
            w2_cp_async_wait<8>();
            ahead(qB);
            // ---------------- rare: the filter could not decide the window's first lane (nothing was committed: the states
            // are those the round was evaluated with).  Every undecided lane takes the exact decision for its slot and
            // injects it into the next fast round -- a bias of +-1e20..1e30 on its log_p and a matching log-uniform make
            // the filter reproduce it -- which is run alone (quota 1) and then resolves and commits like any other round.
            // (One exact attempt per rare event would cost 0.4 us per attempt on a degenerate matrix: at iteration 0 all
            // replicas are in the same configuration and every log_p is a rounding error around 0.)
            if (!was_injected) {
                const unsigned si = ei.x, sj = ej.x;
                const float f1 = w2_image_at(rowiA + 2u * sj, rowiA + lo_off + sj);
                const float f2 = w2_image_at(rowjA + 2u * si, rowjA + lo_off + si);
                const float e0 = fmaf(fabsf(__uint_as_float(ei.y)) + fabsf(__uint_as_float(ej.y)), 3.2e-5f, epsA);
                bool ge0, acc, undecided;
                w2_filter(__uint_as_float(ei.y), f1, __uint_as_float(ej.y), f2, e0, luA, ge0, acc, undecided);
                lu_saved = luA;
                if (undecided) {
                    const unsigned d = w2_exact_decision(rec, words, u, sA, si, sj, logK);
                    bias = (d & 1u) ? 1e30f : -1e20f;
                    if (!(d & 1u)) luA = (d & 2u) ? -1e30f : 0.f;
                    slow++;
                }
                __syncwarp();
                injected = true;
                continue;
            }
            // ---------------- rarer still: undecided WITH the exact decision injected (non-finite energies make log_p a NaN
            // whatever the bias): one exact attempt, exactly what the reference does (window position 0 commits; positions
            // 0 .. advance-1 leave the window; log_p < 0: the next slot is this attempt's uniform)
            {
                rounds++;
                bool ge0 = false, acc = false;
                const unsigned si = ei.x, sj = ej.x;
                f_ij = w2_image_at(rowiA + 2u * sj, rowiA + lo_off + sj);
                f_ji = w2_image_at(rowjA + 2u * si, rowjA + lo_off + si);
                if (w == 0u) {
                    const unsigned ij = rec[sA].ij;
                    const unsigned rowi = (ij & 0xffffu) << logK, rowj = (ij >> 16) << logK;
                    const double logp = swap_logp(u[rowi | sj], u[rowj | si], u[rowi | si], u[rowj | sj]);
                    ge0 = logp >= 0.0;
                    acc = ge0;
                    if (!ge0) {
                        const unsigned s1 = sA + 1;
                        const double dd = logp - slot_logU(words, s1);
                        if (dd > 1e-9) acc = true;
                        else if (dd < -1e-9) acc = false;
                        else acc = mt_double(words[2 * (size_t)s1], words[2 * (size_t)s1 + 1]) < rx_exp_cr(logp);
                    }
                    slow++;
                }
                __syncwarp();
                const bool first_ge0 = __ballot_sync(0xffffffffu, ge0) != 0u;
                p_cm = 1u;
                p_below = first_ge0 ? 1u : 3u;
                p_chg = (acc && neqA != 0u) ? 0xffffffffu : 0u;
                p_entry = (sj * (1u << LOG_STATE_BITS) + si) | (acc ? (1u << 31) | (1u << LOG_ACC_BIT) : (1u << 31));
                commit();
                w2_cp_async_wait<8>();
                ahead(qB);
                p_cm = p_below = 0;
            }
        }
        commit();   // the round resolved last, if one is pending
        w2_cp_async_wait<0>();
        __syncwarp();
        for (int q = lane; q < K; q += 32) perm_g[q] = s_rep[q].state;
    }
    slow = __reduce_add_sync(0xffffffffu, slow);
    if (lane == 0) {
        const long long remaining = remaining0 - (long long)(rem0 - rem);
        ctl->head = h;
        ctl->remaining = remaining;
        ctl->status = remaining > 0 ? 1 : 0;
        ctl->rounds += (int)rounds;
        ctl->slow_exp += slow;
    }
}

// Count matrices from the sparse commit log of k_mix_walk2 (one word per slot, bit 31 = an attempt started there).
__global__ void k_mix_count_slots(const uint32_t *__restrict__ slot_log, long long s0, long long s1, int M,
                                  unsigned long long *__restrict__ nacc, unsigned long long *__restrict__ nprop) {
    long long t = s0 + blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; t < s1; t += stride) {
        const uint32_t e = slot_log[t];
        if (!(e >> 31)) continue;
        const uint32_t si = e & ((1u << LOG_STATE_BITS) - 1u), sj = (e >> LOG_STATE_BITS) & ((1u << LOG_STATE_BITS) - 1u);
        atomicAdd(&nprop[(size_t)si * M + sj], 1ull);
        atomicAdd(&nprop[(size_t)sj * M + si], 1ull);
        if ((e >> LOG_ACC_BIT) & 1u) {
            atomicAdd(&nacc[(size_t)si * M + sj], 1ull);
            atomicAdd(&nacc[(size_t)sj * M + si], 1ull);
        }
    }
}
