// rx_walk_any.cuh -- speculative swap-all walker for ANY K <= 4095 (included by rx_mix.cu).
//
// For K that is not a power of two numba's randint rejects words (numba/_random.c: low bit_length(K-1) bits of one word,
// retried while >= K), so an attempt has no fixed length and no slot grid exists.  What stays true is that the words an
// attempt STARTING at word position p would consume for its two indices depend on the stream alone: a parallel pre-pass
// turns every position into a record {i, j, len, back-mask, log of the uniform at p + len}.  One warp then evaluates the
// 32 consecutive positions [h, h + 32) as if an attempt started at each of them, and follows the chain
//     next(p) = p + len(p) + (log_p(p) < 0 ? 2 : 0)
// from position h through the window by pointer jumping over the lanes (four doublings: a hop is at least two words, so
// at most 16 positions of a window are visited).  Staleness and the commit of the valid prefix are those of
// k_mix_walk_pow2.  Results are bit-identical to replicaexchange.py:321-349.
// The last < 80 words of a pass and the (astronomically rare) attempt whose indices need more than ANY_SCAN words are
// left to k_mix_walk_serial.
#pragma once

#define ANY_SCAN 40       // words scanned for the two indices of an attempt; P(more) < (1/2)^38 per attempt
#define ANY_MAX_K 4095    // 12-bit indices in the record

struct WordRec {          // 16 bytes, one per WORD position p: the attempt that would start there
    uint32_t ijl;         // i | j << 12 | len << 24; len = words that hold the two indices (0: unknown, see ANY_SCAN)
    uint32_t backmask;    // bit 31-b: the attempt at p-1-b shares a replica index with this one (or is unknown)
    double logU;          // log of the uniform made of words p+len, p+len+1: this attempt's draw if log_p < 0
};

__global__ void __launch_bounds__(256) k_words_build(const uint32_t *__restrict__ words, long long nwords, int K, uint32_t mask,
                                                     WordRec *__restrict__ rec) {
    __shared__ uint32_t s_w[256 + 31 + ANY_SCAN + 2];   // words of positions p0-31 .. p0+255+ANY_SCAN+1
    __shared__ uint32_t s_ijl[256 + 31];                 // records' first word for positions p0-31 .. p0+255
    const long long p0 = (long long)blockIdx.x * 256;
    const int t = threadIdx.x;
    for (int q = t; q < 256 + 31 + ANY_SCAN + 2; q += 256) {
        const long long p = p0 - 31 + q;
        s_w[q] = (p >= 0 && p < nwords) ? words[p] : 0u;
    }
    __syncthreads();
    for (int q = t; q < 256 + 31; q += 256) {
        const long long p = p0 - 31 + q;
        uint32_t ijl = 0;
        if (p >= 0 && p < nwords) {
            int found = 0;
            uint32_t i = 0;
            for (int k = 0; k < ANY_SCAN && p + k < nwords; k++) {
                const uint32_t r = s_w[q + k] & mask;
                if (r < (uint32_t)K) {
                    if (found == 0) { i = r; found = 1; }
                    else { ijl = i | (r << 12) | ((uint32_t)(k + 1) << 24); break; }
                }
            }
        }
        s_ijl[q] = ijl;
    }
    __syncthreads();
    const long long p = p0 + t;
    if (p >= nwords) return;
    const int q = t + 31;
    const uint32_t ijl = s_ijl[q];
    const uint32_t i = ijl & 0xfffu, j = (ijl >> 12) & 0xfffu, len = ijl >> 24;
    uint32_t bm = 0;
#pragma unroll 4
    for (int b = 0; b < 31; b++) {
        const uint32_t o = s_ijl[q - 1 - b];
        const uint32_t oi = o & 0xfffu, oj = (o >> 12) & 0xfffu;
        const bool hit = (o >> 24) == 0u || oi == i || oi == j || oj == i || oj == j;
        bm |= (hit ? 1u : 0u) << (31 - b);
    }
    WordRec r;
    r.ijl = ijl;
    r.backmask = bm;
    double lu = 0.0;
    if (len != 0u && p + len + 1 < nwords) {
        const double U = mt_double(s_w[q + len], s_w[q + len + 1]);
        lu = (U == 0.0) ? LOGU_ZERO : log(U);
    }
    r.logU = lu;
    rec[p] = r;
}

struct WalkShared {     // control words shared by the two warps
    volatile unsigned prod;   // records [0, prod) of this pass are in the ring (modulo RING)
    volatile unsigned head;   // walker position
    volatile unsigned done;
};

// CTA = 2 warps, organised like k_mix_walk_pow2: warp 1 streams the records into a shared-memory ring, warp 0 walks.
// head counts WORDS.  The energies are read from L2.
__global__ void __launch_bounds__(64) k_mix_walk_any(const WordRec *__restrict__ rec, const uint32_t *__restrict__ words,
                                                     unsigned nwords, const double *__restrict__ u, int K,
                                                     int *__restrict__ perm_g, uint32_t *__restrict__ commit_log, MixCtl *ctl) {
    extern __shared__ double s_mix[];
    __shared__ WalkShared sh;
    // layout: ring_lu[RING] f64 | diag[K] f64 | ring_ijl[RING] u32 | ring_bm[RING] u32 | perm[K] i32
    double *ring_lu = s_mix;
    double *s_diag = ring_lu + RING;
    uint32_t *ring_ijl = (uint32_t *)(s_diag + K);
    uint32_t *ring_bm = ring_ijl + RING;
    int *s_perm = (int *)(ring_bm + RING);
    // (the warp index through a shuffle: warp-uniform for the compiler, see k_mix_walk2)
    const int tid = threadIdx.x, lane = tid & 31, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    for (int q = tid; q < K; q += 64) {
        const int st = perm_g[q];
        s_perm[q] = st;
        s_diag[q] = u[(size_t)q * K + st];
    }
    const unsigned head0 = (unsigned)ctl->head;
    if (tid == 0) { sh.prod = head0; sh.head = head0; sh.done = 0; }
    __syncthreads();

    if (warp == 1) {
        // ---------------- producer: keep the ring filled up to head + RING - 64
        unsigned prod = head0;
        while (!sh.done) {
            const unsigned head = sh.head;
            unsigned limit = head + RING - 64;   // `head` only ever lags the walker (safe)
            if (limit > nwords) limit = nwords;
            if (prod < limit) {
                __threadfence_block();   // acquire: the walker is done with the entries below `head`
                WordRec r[4];
                unsigned cnt = limit - prod;
                if (cnt > 128) cnt = 128;
#pragma unroll
                for (int b = 0; b < 4; b++) {
                    const unsigned o = b * 32 + lane;
                    if (o < cnt) r[b] = rec[prod + o];
                }
#pragma unroll
                for (int b = 0; b < 4; b++) {
                    const unsigned o = b * 32 + lane;
                    if (o < cnt) {
                        const unsigned w = (prod + o) & (RING - 1);
                        ring_ijl[w] = r[b].ijl; ring_bm[w] = r[b].backmask; ring_lu[w] = r[b].logU;
                    }
                }
                prod += cnt;
                __threadfence_block();
                __syncwarp();
                if (lane == 0) sh.prod = prod;
            } else {
                __nanosleep(40);
            }
        }
        return;
    }

    // ---------------- walker (warp 0)
    unsigned h = head0;
    const long long remaining0 = ctl->remaining;
    unsigned rem = remaining0 > 0x7fffffffLL ? 0x7fffffffu : (unsigned)remaining0;
    const unsigned rem0 = rem;
    unsigned logpos = (unsigned)ctl->log_count, rounds = 0, slow = 0, prod_seen = head0;
    const unsigned lt_mask = (1u << lane) - 1u;
    const unsigned sh_amt = 32u - (unsigned)lane;
    const unsigned a_head = __shfl_sync(0xffffffffu, (unsigned)__cvta_generic_to_shared((const void *)&sh.head), 0);
    unsigned wpos = (h + (unsigned)lane) & (RING - 1);   // this lane's ring entry
    bool give_up = false;   // the attempt at the window's first position has unknown indices: the serial kernel takes over
    // a round may start while every attempt of its window has its index words and its uniform inside the pass
    while (rem > 0 && h + 32u + ANY_SCAN + 2u <= nwords) {
        if (prod_seen < h + 32u) {
            do { prod_seen = sh.prod; } while (prod_seen < h + 32u);   // the producer is behind (start of a pass)
            __threadfence_block();
        }
        rounds++;
        const unsigned w = wpos;
        const uint32_t ijl = ring_ijl[w], backmask = ring_bm[w];
        const double lu = ring_lu[w];
        const unsigned i = ijl & 0xfffu, j = (ijl >> 12) & 0xfffu, len = ijl >> 24;
        const bool unknown = len == 0u;
        const int si = s_perm[i], sj = s_perm[j];
        const unsigned a_ij = i * (unsigned)K + (unsigned)sj, a_ji = j * (unsigned)K + (unsigned)si;
        const double e_ij = u[a_ij];
        const double e_ji = u[a_ji];
        const double logp = swap_logp(e_ij, e_ji, s_diag[i], s_diag[j]);
        const double d = logp - lu;
        const bool ge0 = logp >= 0.0;
        bool acc = ge0 || d > 1e-9;
        const bool ambiguous = !ge0 && fabs(d) <= 1e-9 && !unknown;   // NaN compares false: rejected, like the reference
        if (__any_sync(0xffffffffu, ambiguous)) {
            if (ambiguous) {  // too close to call in the log domain: do exactly what the reference does
                const size_t p1 = (size_t)h + lane + len;
                acc = mt_double(words[p1], words[p1 + 1]) < rx_exp_cr(logp);
                slow++;
            }
        }
        // The visited chain by pointer jumping over the lanes: N = window position of the attempt after this one (>= 32:
        // beyond the window), R = set of positions the chain from here visits.  A hop is at least two words, so a window
        // holds at most 16 visited positions and four doublings resolve every chain; lane 0 holds the chain from h.
        unsigned N = unknown ? 64u : (unsigned)lane + len + (ge0 ? 0u : 2u);
        unsigned R = 1u << lane;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const unsigned src = N & 31u;
            const unsigned Rn = __shfl_sync(0xffffffffu, R, src), Nn = __shfl_sync(0xffffffffu, N, src);
            if (N < 32u) { R |= Rn; N = Nn; }
        }
        const unsigned V = __shfl_sync(0xffffffffu, R, 0);
        const unsigned c = __shfl_sync(0xffffffffu, N, 0);   // where the next attempt starts if the whole chain commits
        const unsigned A = __ballot_sync(0xffffffffu, acc && i != j && !unknown);   // accepted and really changing the permutation
        // a visited position is stale if an earlier visited state-changing swap of this window shares a replica with it
        const unsigned VA = V & A;
        unsigned earlier;   // bit 31-b: window position lane-1-b is a visited state-changing swap
        asm("shl.b32 %0, %1, %2;" : "=r"(earlier) : "r"(VA), "r"(sh_amt));
        const unsigned C = __ballot_sync(0xffffffffu, (earlier & backmask) != 0u || unknown) & V;
        const unsigned low = C & (0u - C);
        unsigned cm = V & (low - 1u);           // low == 0 -> all visited positions
        unsigned n = __popc(cm);
        unsigned advance = C ? (unsigned)__popc(low - 1u) : c;
        if (C & 1u) { give_up = true; break; }  // (only an unknown position can stop the window's first attempt)
        if (n > rem) {
            unsigned pos = 0;  // the first visited position we must NOT run: the (rem+1)-th set bit of cm
            for (unsigned cnt = 0; pos < 32; pos++)
                if ((cm >> pos) & 1u) { if (cnt == rem) break; cnt++; }
            cm &= (1u << pos) - 1u;
            n = rem;
            advance = pos;
        }
        // commit: everything is computed by every lane, only the stores are predicated
        const bool mine = (cm >> lane) & 1u;
        const unsigned log_at = logpos + __popc(cm & lt_mask);
        const uint32_t entry = (uint32_t)si | ((uint32_t)sj << LOG_STATE_BITS) | ((acc ? 1u : 0u) << LOG_ACC_BIT);
        const bool swaps = mine && acc && i != j;
        if (mine) commit_log[log_at] = entry;
        if (swaps) { s_perm[i] = sj; s_perm[j] = si; s_diag[i] = e_ij; s_diag[j] = e_ji; }
        logpos += n;
        h += advance;
        wpos = (wpos + advance) & (RING - 1);
        rem -= n;
        __syncwarp();
        if ((rounds & 3u) == 0u && lane == 0) {   // release (see k_mix_walk_pow2)
            __threadfence_block();
            asm volatile("st.volatile.shared.u32 [%0], %1;" :: "r"(a_head), "r"(h) : "memory");
        }
    }
    (void)give_up;
    if (lane == 0) sh.done = 1;
    for (int q = lane; q < K; q += 32) perm_g[q] = s_perm[q];
    slow = __reduce_add_sync(0xffffffffu, slow);
    if (lane == 0) {
        const long long remaining = remaining0 - (long long)(rem0 - rem);
        ctl->head = h;
        ctl->remaining = remaining;
        ctl->status = remaining > 0 ? 1 : 0;
        ctl->rounds += (int)rounds;
        ctl->slow_exp += slow;
        ctl->log_count = logpos;
    }
}
