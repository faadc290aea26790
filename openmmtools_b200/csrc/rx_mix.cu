// rx_mix.cu -- replica mixing (Gibbs / Metropolis state swaps) on the device.
//
// Replaces ReplicaExchangeSampler._mix_replicas (openmmtools/multistate/replicaexchange.py:255-292):
//   swap-all       _mix_all_replicas_numba  (replicaexchange.py:294-349)  -> k_mix_walk2 / k_mix_walk_pow2 (K a power of two),
//                                                                            k_mix_walk2c / k_mix_walk_any (any other K), k_mix_walk_serial
//   swap-neighbors _mix_neighboring_replicas (replicaexchange.py:366-406) -> k_mix_neighbors
// The results are bit-identical to the reference for the same MT19937 state: the random stream is numba's
// (numba/_random.c:37-73; randint = low bit_length(K-1) bits of one word with rejection, rand = 53-bit double
// from two words), reproduced on the device by k_mt_generate.
//
// Design (see DESIGN.md "mixing"): the K^3-long chain is data dependent (an attempt draws rand() only when
// log_p < 0), but the stream itself is state independent.  For power-of-two K every attempt starts on an
// even word ("slot"), so a parallel pre-pass turns the stream into slot records (i, j, log U, overlap mask)
// and ONE warp then walks the chain speculatively: 32 lanes evaluate 32 consecutive slots under the current
// permutation, the visited-slot chain is resolved with a carry-propagation bit trick, and the longest prefix
// in which no visited slot touches a replica swapped earlier in the same window is committed.
#include "rx_internal.cuh"
#include <type_traits>
#include <algorithm>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <vector>
#include <chrono>
static inline double rx_wall_us() { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// ------------------------------------------------------------------------------------------------------
// MT19937 generation: x[n+624] = x[n+397] ^ twist(x[n], x[n+1]); 227 words are independent per step and
// a thread's second consecutive step only needs its own previous output, so there is one barrier per 454
// words.  `window` holds the last 624 raw words and is advanced by exactly n.
// ------------------------------------------------------------------------------------------------------
#define MT_RING 2048

__device__ __forceinline__ uint32_t mt_temper(uint32_t y) {
    y ^= (y >> 11);
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    y ^= (y >> 18);
    return y;
}
__device__ __forceinline__ uint32_t mt_twist(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t y = (a & 0x80000000u) | (b & 0x7fffffffu);
    return c ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
}

__global__ void __launch_bounds__(256) k_mt_generate(uint32_t *__restrict__ window, uint32_t *__restrict__ out,
                                                     long long n) {
    __shared__ uint32_t buf[MT_RING];
    const int t = threadIdx.x;
    for (int q = t; q < 624; q += 256) buf[q] = window[q];
    __syncthreads();
    long long produced = 0;
    unsigned base = 0;
    while (produced < n) {
        if (t < 227) {
            uint32_t a = buf[(base + t) & (MT_RING - 1)], b = buf[(base + t + 1) & (MT_RING - 1)];
            uint32_t c = buf[(base + t + 397) & (MT_RING - 1)];
            uint32_t x = mt_twist(a, b, c);
            buf[(base + t + 624) & (MT_RING - 1)] = x;
            if (out && produced + t < n) out[produced + t] = mt_temper(x);
            // second step: x[n+227+t+624] needs x[n+227+t], x[n+228+t] (old) and this thread's x[n+624+t]
            a = buf[(base + 227 + t) & (MT_RING - 1)];
            b = buf[(base + 228 + t) & (MT_RING - 1)];
            uint32_t x2 = mt_twist(a, b, x);
            buf[(base + 227 + t + 624) & (MT_RING - 1)] = x2;
            if (out && produced + 227 + t < n) out[produced + 227 + t] = mt_temper(x2);
        }
        __syncthreads();
        produced += 454;
        base += 454;
    }
    // ring position of x_{n0 + n}: base - (produced - n)
    unsigned w0 = base - (unsigned)(produced - n);
    __syncthreads();
    uint32_t keep[3];
    for (int q = t, m = 0; q < 624; q += 256, m++) keep[m] = buf[(w0 + q) & (MT_RING - 1)];
    for (int q = t, m = 0; q < 624; q += 256, m++) window[q] = keep[m];
}

__global__ void k_copy_words(const uint32_t *__restrict__ src, uint32_t *__restrict__ dst, long long n) {
    long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    long long stride = (long long)gridDim.x * blockDim.x;
    for (; i < n; i += stride) dst[i] = src[i];
}

// numba/numpy double from two words: ((a >> 5) * 2^26 + (b >> 6)) / 2^53
__device__ __forceinline__ double mt_double(uint32_t w0, uint32_t w1) {
    return ((double)(w0 >> 5) * 67108864.0 + (double)(w1 >> 6)) * (1.0 / 9007199254740992.0);
}

// log_p exactly as the reference evaluates it: -(e_ij + e_ji) + e_ii + e_jj, left to right, no contraction.
__device__ __forceinline__ double swap_logp(double e_ij, double e_ji, double e_ii, double e_jj) {
    return __dadd_rn(__dadd_rn(-__dadd_rn(e_ij, e_ji), e_ii), e_jj);
}

// exp(x), correctly rounded (round to nearest) -- for the reference's own test `rand() < exp(log_p)` in the cases where
// it is not decided in the log domain.  CUDA's exp() may be off by one ulp; the host libm the reference calls (numba -> libm
// exp) is correctly rounded at all but ~1 % of the arguments: with a one-ulp error the decision differs from the
// reference's whenever U is the double next to exp(log_p) (tests/test_gpu_mixing.py constructs such matrices).
// Double-double evaluation: x = k ln2 + r (three-part ln 2, the first part fdlibm's ln2HI so that k ln2HI is exact),
// expm1(r / 256) by its Taylor series to the 9th power, eight squarings in the form m <- m (m + 2), result (1 + m) 2^k;
// relative error ~2^-95, so the rounding can only be wrong if exp(x) lies within ~2^-40 ulp of a midpoint between two doubles.
// Rare path only (guard band, plain loop): its speed is irrelevant.
struct rx_dd { double hi, lo; };
__device__ __forceinline__ rx_dd dd_fast_two_sum(double a, double b) {
    const double s = __dadd_rn(a, b);
    return {s, __dadd_rn(b, -__dadd_rn(s, -a))};
}
__device__ __forceinline__ rx_dd dd_two_sum(double a, double b) {
    const double s = __dadd_rn(a, b), bb = __dadd_rn(s, -a);
    return {s, __dadd_rn(__dadd_rn(a, -__dadd_rn(s, -bb)), __dadd_rn(b, -bb))};
}
__device__ __forceinline__ rx_dd dd_add(rx_dd a, rx_dd b) {
    rx_dd s = dd_two_sum(a.hi, b.hi);
    const rx_dd t = dd_two_sum(a.lo, b.lo);
    s = dd_fast_two_sum(s.hi, __dadd_rn(s.lo, t.hi));
    return dd_fast_two_sum(s.hi, __dadd_rn(s.lo, t.lo));
}
__device__ __forceinline__ rx_dd dd_mul(rx_dd a, rx_dd b) {
    const double p = __dmul_rn(a.hi, b.hi);
    double e = __fma_rn(a.hi, b.hi, -p);
    e = __fma_rn(a.hi, b.lo, e);
    e = __fma_rn(a.lo, b.hi, e);
    return dd_fast_two_sum(p, e);
}
__device__ __noinline__ double rx_exp_cr(double x) {
    if (!(x == x)) return x;
    if (x > 709.782712893384) return INFINITY;
    if (x < -745.1332191019412) return 0.0;      // exp(x) <= 2^-1075 rounds to zero
    const double kd = rint(__dmul_rn(x, 1.4426950408889634));
    const double ln2HI = 6.93147180369123816490e-01, ln2LO = 1.9082149292705877e-10, ln2LL = 1.1612227229362532e-26;
    const double r0 = __fma_rn(-kd, ln2HI, x);                  // exact
    const double p = __dmul_rn(kd, ln2LO), pe = __fma_rn(kd, ln2LO, -p);
    rx_dd r = dd_two_sum(r0, -p);
    r = dd_fast_two_sum(r.hi, __dadd_rn(r.lo, -__dadd_rn(pe, __dmul_rn(kd, ln2LL))));
    const rx_dd s = {__dmul_rn(r.hi, 0.00390625), __dmul_rn(r.lo, 0.00390625)};   // r / 256, exact
    const rx_dd c[8] = {   // 1/2! .. 1/9!
        {0.5, 0.0},
        {0.16666666666666666, 9.25185853854297e-18},
        {0.041666666666666664, 2.3129646346357427e-18},
        {0.008333333333333333, 1.1564823173178714e-19},
        {0.001388888888888889, -5.300543954373577e-20},
        {0.0001984126984126984, 1.7209558293420705e-22},
        {2.48015873015873e-05, 2.1511947866775882e-23},
        {2.7557319223985893e-06, -1.858393274046472e-22}};
    rx_dd acc = c[7];
#pragma unroll
    for (int n = 6; n >= 0; n--) acc = dd_add(c[n], dd_mul(s, acc));
    rx_dd m = dd_add(s, dd_mul(dd_mul(s, s), acc));                  // expm1(r / 256)
#pragma unroll
    for (int q = 0; q < 8; q++) m = dd_mul(m, dd_add(m, rx_dd{2.0, 0.0}));     // expm1(2 t) = expm1(t) (expm1(t) + 2)
    const rx_dd y = dd_add(rx_dd{1.0, 0.0}, m);
    return ldexp(y.hi, (int)kd);
}

__global__ void k_selftest_exp(const double *__restrict__ x, double *__restrict__ y, int n) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) y[t] = rx_exp_cr(x[t]);
}
int rxi_selftest_exp(rx_engine *h, const double *x, double *y, int n) {
    double *d = nullptr;
    if (n <= 0) return RX_OK;
    RX_CHECK_CUDA(h, cudaMalloc(&d, 2 * (size_t)n * sizeof(double)));
    RX_CHECK_CUDA(h, cudaMemcpy(d, x, (size_t)n * sizeof(double), cudaMemcpyHostToDevice));
    k_selftest_exp<<<(n + 127) / 128, 128, 0, h->stream>>>(d, d + n, n);
    RX_CHECK_CUDA(h, cudaGetLastError());
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    RX_CHECK_CUDA(h, cudaMemcpy(y, d + n, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost));
    cudaFree(d);
    return RX_OK;
}

// ------------------------------------------------------------------------------------------------------
// Slot records (state independent, fully parallel).
// ------------------------------------------------------------------------------------------------------
#define LOGU_ZERO (-745.5)  /* stands in for log(0): exp(x) == 0 <=> x < -745.13 */

__global__ void __launch_bounds__(256) k_slots_build(const uint32_t *__restrict__ words, long long nslots,
                                                     uint32_t mask, SlotRec *__restrict__ rec) {
    __shared__ uint32_t s_ij[256 + 32];
    long long s0 = (long long)blockIdx.x * 256;
    int t = threadIdx.x;
    // tile: slots s0-32 .. s0+255
    for (int q = t; q < 256 + 32; q += 256) {
        long long s = s0 - 32 + q;
        uint32_t ij = 0xffffffffu;
        if (s >= 0 && s < nslots) ij = (words[2 * s] & mask) | ((words[2 * s + 1] & mask) << 16);
        s_ij[q] = ij;
    }
    __syncthreads();
    long long s = s0 + t;
    if (s >= nslots) return;
    uint32_t w0 = words[2 * s], w1 = words[2 * s + 1];
    uint32_t ij = s_ij[t + 32];
    uint32_t i = ij & 0xffffu, j = ij >> 16;
    uint32_t bm = 0;
#pragma unroll
    for (int b = 0; b < 31; b++) {
        uint32_t o = s_ij[t + 32 - 1 - b];
        uint32_t oi = o & 0xffffu, oj = o >> 16;
        bool hit = (o != 0xffffffffu) && (oi == i || oi == j || oj == i || oj == j);
        bm |= (hit ? 1u : 0u) << (31 - b);
    }
    double U = mt_double(w0, w1);
    SlotRec r;
    r.ij = ij;
    r.backmask = bm;
    r.logU = (U == 0.0) ? LOGU_ZERO : log(U);
    rec[s] = r;
}

// ------------------------------------------------------------------------------------------------------
// The speculative chain walker.  K must be a power of two <= 16384.
//
// One warp walks (a second one only helps with the prologue).  The slot records come from DRAM (written once by the
// pre-pass, read once) into a 1024-slot shared-memory ring by cp.async that the walker issues itself, 512 slots ahead.
// Per round the warp (1) reads 32 records from the ring, (2) looks up the current states of both replicas, (3) fetches
// u[i,sj], u[j,si] and the maintained diagonal d[k] = u[k, perm[k]], (4) evaluates log_p and the accept test, (5) resolves
// the visited chain and staleness with ballots and bit tricks, (6) commits the valid prefix: permutation + diagonal
// in shared memory and ONE coalesced store of packed (si, sj, accepted) entries into a commit log (the count
// matrices are built from the log afterwards by k_mix_count, in parallel).
// (Round 1 had a producer warp and a ring synchronised by fences and volatile flags; the single warp with hardware-tracked
// copies is racecheck-clean and costs ~6 more instructions per round.)
//
// Where the energies live (FILTER):
//   true    K <= 256, where the image fits in shared memory (213 KB at K = 256); the kernel finishes the passes of
//           k_mix_walk2 on its SlotRec2 records.  Shared memory holds a 24-bit floating image of every row
//           (delta = u - rowmin as a float32 truncated to sign + 8 exponent + 15 mantissa bits) that gives log_p
//           to within a RIGOROUS bound eps = 3.2e-5 * sum|delta| + tiny; the decision is taken from the image, in
//           f32, whenever it is more than eps away from both thresholds (log_p = 0 and log_p = log U); a round
//           whose committed prefix contains an undecided lane is redone with the exact f64 values from L2.
//           The result is therefore still bit-identical.
//   false   exact f64 values from L2 every round, on SlotRec records (K >= 512)
//
// The walker's round is one dependent chain (~105 instructions, ~0.2 us); what was measured to matter, on one box:
// no f64 on the chain (-65 ns), no data-dependent branch besides the loop's (-60 ns: one loop condition, predicated
// commit), no sub-word shared stores (a byte-wide permutation table costs +40 ns), the absolute-to-relative lane
// conversion as one shift (back-mask bit order), and nothing re-derived from special registers inside the loop.
// ------------------------------------------------------------------------------------------------------
#define LOG_ACC_BIT 28
#define LOG_STATE_BITS 14
#define RING 1024
#include "rx_walk2.cuh"
#include "rx_walk_any.cuh"
#include "rx_walk2c.cuh"

// FILTER: the records are SlotRec2 (rx_walk2.cuh), otherwise SlotRec.
template <bool FILTER>
__global__ void __launch_bounds__(64) k_mix_walk_pow2(const SlotRec *__restrict__ rec, const uint32_t *__restrict__ words,
                                                      unsigned nslots, const double *__restrict__ u, int K, int logK,
                                                      int *__restrict__ perm_g, uint32_t *__restrict__ commit_log,
                                                      const unsigned char *__restrict__ filt,
                                                      const double *__restrict__ filt_rowabs, MixCtl *ctl) {
    extern __shared__ double s_mix[];
    // layout: ring[RING] 16-byte records | diag[K] f64 | (rowabs[K]) | perm[K] i32 | (image: u16[K*K] + u8[K*K])
    uint4 *s_ring = (uint4 *)s_mix;
    double *s_diag = s_mix + 2 * RING;
    double *s_rowabs = s_diag + K;                                   // [K] |row minimum| (FILTER only)
    int *s_perm = (int *)(s_rowabs + (FILTER ? K : 0));
    unsigned char *s_q = (unsigned char *)(s_perm + K);   // 24-bit image: int16 high plane [K*K] then uint8 low plane [K*K]
    // (the warp index through a shuffle: warp-uniform for the compiler, see k_mix_walk2)
    const int tid = threadIdx.x, lane = tid & 31, warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    for (int q = tid; q < K; q += 64) {
        const int st = perm_g[q];
        s_perm[q] = st;
        s_diag[q] = u[((size_t)q << logK) + st];
        // per-row share of the f64-rounding bound, f32 rounded up: 1.6e-14 (|row minimum| + 1/2)
        if (FILTER) ((float *)s_rowabs)[q] = __fmul_ru(1.6e-14f, __fadd_ru(__double2float_ru(filt_rowabs[q]), 0.5f));
    }
    if (FILTER) {
        const uint32_t *src = (const uint32_t *)filt;
        uint32_t *dst = (uint32_t *)s_q;
        for (int q = tid; q < (3 * K * K) / 4; q += 64) dst[q] = src[q];
    }
    const unsigned head0 = (unsigned)ctl->head;
    __syncthreads();
    if (warp != 0) return;   // (the second warp only helps with the prologue)

    // The records come into the ring by cp.async issued by the walker itself, 640 slots ahead, topped up every 8 rounds;
    // completion is tracked by the hardware (cp.async.wait_group), the warp barrier at the end of a round makes the data
    // visible to all lanes.  No second warp,
    // no flags, no fences: nothing for racecheck to find.
    // (32-bit shared address through a shuffle: it then lives in a register instead of being re-derived from SR_CgaCtaId
    // every round)
    const unsigned ring_addr = __shfl_sync(0xffffffffu, (unsigned)__cvta_generic_to_shared((const void *)s_ring), 0);
    const uint4 *recs = (const uint4 *)rec;
    unsigned filled = head0;
    auto refill = [&](unsigned h_now) {
        while (filled < h_now + 640u && filled < nslots) {
            if (filled + (unsigned)lane < nslots)
                w2_cp_async16(ring_addr + (((filled + (unsigned)lane) & (RING - 1)) << 4), recs + (filled + lane));
            filled += 32u;
        }
        w2_cp_async_commit();
    };
    refill(head0);
    w2_cp_async_wait<0>();
    __syncwarp();

    // ---------------- walker (warp 0).  The loop is latency bound (one warp, one dependent chain per round), so it is
    // written for a short instruction stream: 32-bit indices, cached producer position, head published every 8 rounds.
    unsigned h = head0;
    const long long remaining0 = ctl->remaining;
    unsigned rem = remaining0 > 0x7fffffffLL ? 0x7fffffffu : (unsigned)remaining0;   // attempts this launch may still do
    const unsigned rem0 = rem;
    unsigned logpos = (unsigned)ctl->log_count, rounds = 0, slow = 0;   // the log continues where k_mix_walk2 stopped
    const unsigned lt_mask = (1u << lane) - 1u;
    const unsigned sh_amt = 32u - (unsigned)lane;
    const unsigned short *s_qhi = (const unsigned short *)s_q;            // [K*K] sign, exponent, 7 mantissa bits
    const unsigned char *s_qlo = s_q + 2 * (size_t)K * K;                  // [K*K] next 8 mantissa bits
    unsigned wpos = (h + (unsigned)lane) & (RING - 1);   // this lane's ring slot
    // One round.  TAIL = the launch's attempt budget may end inside the window (checked only in the last rounds).
    auto round = [&](auto tail_tag) {
        constexpr bool TAIL = decltype(tail_tag)::value;
        rounds++;
        const unsigned w = wpos;   // (h + lane) & (RING - 1), carried from round to round
        const uint4 rq = w2_lds128(ring_addr + (w << 4));
        const uint32_t ij = rq.x, backmask = rq.y;
        // the uniform an attempt here would draw belongs to the NEXT slot (SlotRec: its f64 logU is words z, w of the record)
        double logU_next = 0.0;
        if (!FILTER) {
            const uint2 lw = w2_lds64(ring_addr + (((w + 1) & (RING - 1)) << 4) + 8u);
            logU_next = __hiloint2double((int)lw.y, (int)lw.x);
        }
        const unsigned i = ij & 0xffffu, j = ij >> 16;
        const int si = s_perm[i], sj = s_perm[j];
        const unsigned a_ij = (i << logK) | (unsigned)sj, a_ji = (j << logK) | (unsigned)si;
        bool ge0, acc, undecided = false;
        double e_ij = 0.0, e_ji = 0.0;   // exact off-diagonal values, needed by the commit (new diagonal)
        if (FILTER) {
            // image of u: 24-bit floats of delta = u - rowmin; logp~ = (d_ii - d_ij) + (d_jj - d_ji), |logp~ - logp_ref| <= eps
            const unsigned a_ii = (i << logK) | (unsigned)si, a_jj = (j << logK) | (unsigned)sj;
            // (hi << 16) | (lo << 8) in one byte permute
            const float f_ii = __uint_as_float(__byte_perm((unsigned)s_qhi[a_ii], (unsigned)s_qlo[a_ii], 0x1045));
            const float f_ij = __uint_as_float(__byte_perm((unsigned)s_qhi[a_ij], (unsigned)s_qlo[a_ij], 0x1045));
            const float f_jj = __uint_as_float(__byte_perm((unsigned)s_qhi[a_jj], (unsigned)s_qlo[a_jj], 0x1045));
            const float f_ji = __uint_as_float(__byte_perm((unsigned)s_qhi[a_ji], (unsigned)s_qlo[a_ji], 0x1045));
            // All in f32.  Every image value is within 2^-15 (relative) of the true delta (truncation to a 15-bit
            // mantissa + f32 rounding); the f32 additions below add at most 2^-23 of the magnitudes; the f64 rounding
            // of the reference's own three additions and of our centring is <= 64 ulp(f64) of the magnitudes.
            const float lp = (f_ii - f_ij) + (f_jj - f_ji);
            const float mag = (fabsf(f_ii) + fabsf(f_ij)) + (fabsf(f_jj) + fabsf(f_ji));
            // the guard band's 1e-9 rides in eps (a slightly wider eps for the sign test is only more conservative);
            // 1.6e-14 mag is inside the slack of 3.2e-5
            const float eps = fmaf(mag, 3.2e-5f, (((const float *)s_rowabs)[i] + ((const float *)s_rowabs)[j]) + 1e-9f);
            // log of the uniform, rounded to f32 by the producer: |lu - logU| <= 2^-24 |lu|; d carries one more rounding
            // (SlotRec2: the f32 log-uniform of the next slot is the third word of this slot's own record)
            const float lu = __uint_as_float(rq.z);
            const float d = lp - lu;
            const float mar = fmaf(fabsf(lp) + fabsf(lu), 1.3e-7f, eps);
            // |lp| > eps decides the sign of log_p, |d| > mar decides the comparison with the uniform (NaN: undecided)
            const bool dec_lp = fabsf(lp) > eps, dec_d = fabsf(d) > mar;
            // i == j: the reference's log_p is exactly 0 for finite energies (-(e+e)+e+e), accepted without a draw
            const bool same = (i == j) && (fabsf(f_ii) <= 3.0e38f);
            ge0 = (dec_lp && lp > 0.f) || same;
            acc = ge0 || (dec_lp && dec_d && d > 0.f);
            const bool decided = ge0 || (dec_lp && dec_d);
            undecided = !decided;   // resolved below, and only if the lane turns out to matter
        } else {
            e_ij = u[a_ij];
            e_ji = u[a_ji];
            const double logp = swap_logp(e_ij, e_ji, s_diag[i], s_diag[j]);
            const double d = logp - logU_next;
            ge0 = logp >= 0.0;
            acc = ge0 || d > 1e-9;
            const bool ambiguous = !ge0 && fabs(d) <= 1e-9;   // NaN compares false: rejected, like the reference
            if (__any_sync(0xffffffffu, ambiguous)) {
                if (ambiguous) {  // too close to call in the log domain: do exactly what the reference does
                    const unsigned s1 = h + lane + 1;
                    acc = mt_double(words[2 * (size_t)s1], words[2 * (size_t)s1 + 1]) < rx_exp_cr(logp);
                    slow++;
                }
            }
        }
        unsigned V, C, low, cm, n, advance;
        auto resolve = [&]() {
            const unsigned G = __ballot_sync(0xffffffffu, ge0);
            const unsigned A = __ballot_sync(0xffffffffu, acc && i != j);   // accepted and really changing the permutation
            // Visited chain: from a visited slot s the next attempt starts at s+1 if log_p >= 0 (no uniform drawn) else
            // at s+2.  skip[s+1] = NG[s] & ~skip[s]: inside a run of NG ones the skip flag alternates, so skip[s] =
            // parity of (s - run start); runs are split by the parity of their start with an add-carry (32-bit adds +
            // carry out).
            const unsigned X = ~G;
            const unsigned starts = X & ~(X << 1);
            const unsigned SE = starts & 0x55555555u, SO = starts & 0xAAAAAAAAu;
            const unsigned sumE = X + SE, sumO = X + SO;
            const unsigned skip = (((sumE ^ X) & ~SE) & 0xAAAAAAAAu) | (((sumO ^ X) & ~SO) & 0x55555555u);
            V = ~skip;
            const unsigned VA = V & A;  // visited, accepted, really changing the permutation
            // lane t is stale if an earlier visited state-changing swap in this window shares a replica with it
            unsigned earlier;   // bit 31-b: lane t-1-b is a visited state-changing swap (shl by 32 gives 0 for lane 0)
            asm("shl.b32 %0, %1, %2;" : "=r"(earlier) : "r"(VA), "r"(sh_amt));
            C = __ballot_sync(0xffffffffu, (earlier & backmask) != 0u) & V;
            low = C & (0u - C);
            cm = V & (low - 1u);           // low == 0 -> all lanes
            n = __popc(cm);
            // bit 32 (even position) of the skip word can only be set by the carry of an odd-start run
            advance = C ? (unsigned)__popc(low - 1u) : 32u + (sumO < X ? 1u : 0u);
        };
        if (FILTER) {
            // The filter's undecided lanes carry arbitrary ge0/acc.  Bits of V, C and cm below the lowest undecided
            // visited lane do not depend on them (the chain and the staleness test only look downwards), so the round
            // is resolved speculatively and redone with exact values only when such a lane lies inside the committed
            // prefix -- the ballot of the undecided lanes is off the critical path and rarely matters.
            const unsigned U = __ballot_sync(0xffffffffu, undecided);
            resolve();
            if (U & cm) {
                if (undecided) {   // exact path for this lane: the f64 values from L2
                    const unsigned a_ii = (i << logK) | (unsigned)si, a_jj = (j << logK) | (unsigned)sj;
                    const double logp = swap_logp(u[a_ij], u[a_ji], u[a_ii], u[a_jj]);
                    ge0 = logp >= 0.0;
                    acc = ge0;
                    if (!ge0) {
                        const double dd = logp - slot_logU(words, h + lane + 1);
                        if (dd > 1e-9) acc = true;
                        else if (dd < -1e-9) acc = false;
                        else { const unsigned s1 = h + lane + 1; acc = mt_double(words[2 * (size_t)s1], words[2 * (size_t)s1 + 1]) < rx_exp_cr(logp); }
                    }
                    slow++;
                }
                resolve();
            }
        } else {
            resolve();
        }
        if (TAIL && n > rem) {
            unsigned pos = 0;  // the first visited lane we must NOT run: the (rem+1)-th set bit of cm
            for (unsigned cnt = 0; pos < 32; pos++)
                if ((cm >> pos) & 1u) { if (cnt == rem) break; cnt++; }
            cm &= (1u << pos) - 1u;
            n = rem;
            advance = pos;
        }
        // commit: everything is computed by every lane, only the stores are predicated (no divergent block)
        const bool mine = (cm >> lane) & 1u;
        const unsigned log_at = logpos + __popc(cm & lt_mask);
        const uint32_t entry = (uint32_t)si | ((uint32_t)sj << LOG_STATE_BITS) | ((acc ? 1u : 0u) << LOG_ACC_BIT);
        const bool swaps = mine && acc && i != j;  // an i == j lane must not write: a later committed lane may swap this replica
        if (mine) commit_log[log_at] = entry;
        if (swaps) { s_perm[i] = sj; s_perm[j] = si; }
        if (!FILTER) { if (swaps) { s_diag[i] = e_ij; s_diag[j] = e_ji; } }   // the image needs no f64 diagonal
        logpos += n;
        h += advance;
        wpos = (wpos + advance) & (RING - 1);
        rem -= n;
        // every 8 rounds (at most 264 slots): top the ring up to 640 slots ahead and wait for all copies but the ones just
        // issued -- what the next 8 rounds read (< h + 298) was issued at the previous top-up or earlier (>= h + 376 then)
        if ((rounds & 7u) == 0u) { refill(h); w2_cp_async_wait<1>(); }
        __syncwarp();
    };
    while (rem > 0 && h + 33 <= nslots) {
        if (rem >= 33) {
            // main loop: a round commits at most 32 attempts, so the budget cannot end inside it
            do { round(std::false_type()); } while (rem >= 33u && h + 33u <= nslots);
        } else {
            round(std::true_type());
        }
    }
    w2_cp_async_wait<0>();
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

// 24-bit row image of the energy matrix for the filter walkers: delta = u[k,l] - min_l u[k,l] as a float32 truncated to
// its top 24 bits (sign, 8 exponent, 15 mantissa bits), stored as a uint16 plane followed by a uint8 plane.  Relative
// precision 2^-15 per entry, so huge entries (a decoupled atom overlapping another one evaluated at lambda = 1) cost no
// precision where the decisions are made.  absmax_out[k] = max |u[k,:]| (inf for rows with non-finite values).
__global__ void k_mix_filter_build(const double *__restrict__ u, int K, unsigned char *__restrict__ filt, double *__restrict__ scale,
                                   double *__restrict__ absmax_out) {
    __shared__ double s_lo[8], s_am[8];
    const int k = blockIdx.x, t = threadIdx.x;
    double lo = INFINITY, am = 0.0;
    bool bad = false;
    for (int l = t; l < K; l += blockDim.x) {
        const double v = u[(size_t)k * K + l];
        if (!isfinite(v)) bad = true;
        lo = fmin(lo, v); am = fmax(am, fabs(v));
    }
    for (int o = 16; o > 0; o >>= 1) {
        lo = fmin(lo, __shfl_down_sync(0xffffffffu, lo, o));
        am = fmax(am, __shfl_down_sync(0xffffffffu, am, o));
    }
    const int anybad = __syncthreads_or(bad ? 1 : 0);
    if ((t & 31) == 0) { s_lo[t >> 5] = lo; s_am[t >> 5] = am; }
    __syncthreads();
    lo = s_lo[0]; am = s_am[0];
    for (int q = 1; q < (int)(blockDim.x >> 5); q++) { lo = fmin(lo, s_lo[q]); am = fmax(am, s_am[q]); }
    if (!isfinite(lo)) lo = 0.0;
    for (int l = t; l < K; l += blockDim.x) {
        const float f = (float)(u[(size_t)k * K + l] - lo);     // round to nearest f32; inf/NaN stay inf/NaN
        const unsigned bits = __float_as_uint(f) & 0xffffff00u;  // truncate to 24 bits (toward zero)
        ((unsigned short *)filt)[(size_t)k * K + l] = (unsigned short)(bits >> 16);
        filt[2 * (size_t)K * K + (size_t)k * K + l] = (unsigned char)((bits >> 8) & 0xffu);
    }
    if (t == 0) { scale[k] = fabs(lo); absmax_out[k] = anybad ? INFINITY : am; }
}

// Build the (symmetric) proposal / acceptance count matrices from the commit log (replicaexchange.py:339-349).
__global__ void k_mix_count(const uint32_t *__restrict__ commit_log, long long n, int M, unsigned long long *__restrict__ nacc,
                            unsigned long long *__restrict__ nprop) {
    long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (; t < n; t += stride) {
        const uint32_t e = commit_log[t];
        const uint32_t si = e & ((1u << LOG_STATE_BITS) - 1u), sj = (e >> LOG_STATE_BITS) & ((1u << LOG_STATE_BITS) - 1u);
        atomicAdd(&nprop[(size_t)si * M + sj], 1ull);
        atomicAdd(&nprop[(size_t)sj * M + si], 1ull);
        if ((e >> LOG_ACC_BIT) & 1u) {
            atomicAdd(&nacc[(size_t)si * M + sj], 1ull);
            atomicAdd(&nacc[(size_t)sj * M + si], 1ull);
        }
    }
}

// ------------------------------------------------------------------------------------------------------
// Plain serial walker for any K (rejection sampling makes the slot structure state dependent).
// head counts WORDS here.  An attempt that would run out of words is rolled back.
// ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) k_mix_walk_serial(const uint32_t *__restrict__ words, long long nwords,
                                                        const double *__restrict__ u, int K, int M, int *perm_g,
                                                        unsigned long long *nacc, unsigned long long *nprop,
                                                        MixCtl *ctl) {
    extern __shared__ int s_perm[];
    const int lane = threadIdx.x;
    for (int q = lane; q < K; q += 32) s_perm[q] = perm_g[q];
    __syncwarp();
    if (lane == 0) {
        long long p = ctl->head, remaining = ctl->remaining;
        int nbits = 0;
        for (unsigned m = (unsigned)(K - 1); m; m >>= 1) nbits++;
        const uint32_t mask = nbits ? (0xffffffffu >> (32 - nbits)) : 0u;
        while (remaining > 0) {
            long long q = p;
            int i = 0, j = 0;
            bool ok = true;
            if (K > 1) {
                for (;;) { if (q >= nwords) { ok = false; break; } uint32_t r = words[q++] & mask; if ((int)r < K) { i = r; break; } }
                if (ok) for (;;) { if (q >= nwords) { ok = false; break; } uint32_t r = words[q++] & mask; if ((int)r < K) { j = r; break; } }
            }
            if (!ok) break;
            const int si = s_perm[i], sj = s_perm[j];
            const double logp = swap_logp(u[(size_t)i * M + sj], u[(size_t)j * M + si], u[(size_t)i * M + si],
                                          u[(size_t)j * M + sj]);
            bool acc = logp >= 0.0;
            if (!acc) {
                if (q + 2 > nwords) break;
                const double U = mt_double(words[q], words[q + 1]);
                q += 2;
                acc = U < rx_exp_cr(logp);
            }
            nprop[(size_t)si * M + sj] += 1;
            nprop[(size_t)sj * M + si] += 1;
            if (acc) {
                s_perm[i] = sj;
                s_perm[j] = si;
                nacc[(size_t)si * M + sj] += 1;
                nacc[(size_t)sj * M + si] += 1;
            }
            p = q;
            remaining--;
        }
        ctl->head = p;
        ctl->remaining = remaining;
        ctl->status = remaining > 0 ? 1 : 0;
    }
    __syncwarp();
    for (int q = lane; q < K; q += 32) perm_g[q] = s_perm[q];
}

// swap-neighbors (replicaexchange.py:366-406) on numpy's RandomState stream: offset = randint(2) is one
// masked word; each state pair (s, s+1) is attempted once; rand() (two words) only when log_p < 0.
__global__ void __launch_bounds__(32) k_mix_neighbors(const uint32_t *__restrict__ words, long long nwords,
                                                      const double *__restrict__ u, int K, int M, int *perm_g,
                                                      unsigned long long *nacc, unsigned long long *nprop,
                                                      MixCtl *ctl) {
    extern __shared__ int s_mem[];
    int *s_perm = s_mem, *s_inv = s_mem + K;
    const int lane = threadIdx.x;
    for (int q = lane; q < K; q += 32) { int s = perm_g[q]; s_perm[q] = s; if (s >= 0 && s < K) s_inv[s] = q; }
    __syncwarp();
    if (lane == 0) {
        long long p = 0;
        const int offset = (int)(words[p++] & 1u);
        for (int s = offset; s < K - 1; s += 2) {
            const int i = s_inv[s], j = s_inv[s + 1];
            const int si = s, sj = s + 1;
            const double logp = swap_logp(u[(size_t)i * M + sj], u[(size_t)j * M + si], u[(size_t)i * M + si],
                                          u[(size_t)j * M + sj]);
            bool acc = logp >= 0.0;
            if (!acc) {
                const double U = mt_double(words[p], words[p + 1]);
                p += 2;
                acc = U < rx_exp_cr(logp);
            }
            nprop[(size_t)si * M + sj] += 1;
            nprop[(size_t)sj * M + si] += 1;
            if (acc) {
                s_perm[i] = sj; s_perm[j] = si;
                s_inv[sj] = i; s_inv[si] = j;
                nacc[(size_t)si * M + sj] += 1;
                nacc[(size_t)sj * M + si] += 1;
            }
        }
        ctl->head = p;
        ctl->remaining = 0;
        ctl->status = 0;
    }
    __syncwarp();
    for (int q = lane; q < K; q += 32) perm_g[q] = s_perm[q];
}

// ------------------------------------------------------------------------------------------------------
// Host side: stream management
// ------------------------------------------------------------------------------------------------------
static int stream_reserve(rx_engine *h, MTStream &S, size_t cap) {
    if (cap <= S.cap) return RX_OK;
    uint32_t *a = nullptr, *b = nullptr;
    RX_CHECK_CUDA(h, cudaMalloc(&a, cap * sizeof(uint32_t)));
    RX_CHECK_CUDA(h, cudaMalloc(&b, cap * sizeof(uint32_t)));
    if (S.avail) RX_CHECK_CUDA(h, cudaMemcpyAsync(a, S.d_words, S.avail * sizeof(uint32_t), cudaMemcpyDeviceToDevice, h->stream));
    RX_CHECK_CUDA(h, cudaDeviceSynchronize());
    cudaFree(S.d_words);
    cudaFree(S.d_words_alt);
    S.d_words = a;
    S.d_words_alt = b;
    S.cap = cap;
    return RX_OK;
}

// make at least `need` unconsumed words available
static int stream_fill(rx_engine *h, MTStream &S, size_t need, int *launches, cudaStream_t st) {
    if (S.avail >= need) return RX_OK;
    int rc = stream_reserve(h, S, need);
    if (rc) return rc;
    long long n = (long long)(need - S.avail);
    k_mt_generate<<<1, 256, 0, st>>>(S.d_window, S.d_words + S.avail, n);
    RX_CHECK_CUDA(h, cudaGetLastError());
    S.avail = need;
    (*launches)++;
    return RX_OK;
}

static int stream_consume(rx_engine *h, MTStream &S, size_t c, int *launches) {
    if (c > S.avail) RX_FAIL(h, RX_ERR_INVALID, "internal: consumed more words than available");
    size_t left = S.avail - c;
    if (left && c) {
        k_copy_words<<<(unsigned)((left + 1023) / 1024 > 1184 ? 1184 : (left + 1023) / 1024), 1024, 0, h->stream>>>(
            S.d_words + c, S.d_words_alt, (long long)left);
        RX_CHECK_CUDA(h, cudaGetLastError());
        std::swap(S.d_words, S.d_words_alt);
        (*launches)++;
    }
    S.avail = left;
    S.consumed += c;
    return RX_OK;
}

int rxi_mix_seed(rx_engine *h, int stream, uint32_t seed) {
    if (stream < 0 || stream > 1) RX_FAIL(h, RX_ERR_INVALID, "rx_mix_seed: stream must be 0 (numba) or 1 (numpy)");
    MTStream &S = h->streams[stream];
    uint32_t mt[624];
    mt[0] = seed;  // init_genrand, numba/_random.c:59-73
    for (int i = 1; i < 624; i++) mt[i] = 1812433253u * (mt[i - 1] ^ (mt[i - 1] >> 30)) + (uint32_t)i;
    if (!S.d_window) RX_CHECK_CUDA(h, cudaMalloc(&S.d_window, 624 * sizeof(uint32_t)));
    RX_CHECK_CUDA(h, cudaMemcpy(S.d_window, mt, sizeof(mt), cudaMemcpyHostToDevice));
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream_rng));
    if (stream == RX_STREAM_NUMBA) { h->prepared = false; h->last_consumed = 0; }
    S.avail = 0;
    S.consumed = 0;
    S.seeded = true;
    return RX_OK;
}

int rxi_mix_skip(rx_engine *h, int stream, unsigned long long n) {
    if (stream < 0 || stream > 1) RX_FAIL(h, RX_ERR_INVALID, "rx_mix_skip: stream must be 0 (numba) or 1 (numpy)");
    MTStream &S = h->streams[stream];
    if (!S.seeded) RX_FAIL(h, RX_ERR_INVALID, "rx_mix_skip: seed the stream first");
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream_rng));
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    if (stream == RX_STREAM_NUMBA) h->prepared = false;
    // drop buffered words first, then advance the generator without storing
    unsigned long long todo = n;
    if (S.avail) {
        const size_t c = (size_t)(todo < S.avail ? todo : S.avail);
        {
            size_t left = S.avail - c;
            if (left && c) {
                k_copy_words<<<1184, 1024, 0, h->stream>>>(S.d_words + c, S.d_words_alt, (long long)left);
                RX_CHECK_CUDA(h, cudaGetLastError());
                std::swap(S.d_words, S.d_words_alt);
            }
            S.avail = left;
            S.consumed += c;
        }
        todo -= c;
    }
    while (todo > 0) {
        const long long chunk = todo > (1ull << 30) ? (1ll << 30) : (long long)todo;
        k_mt_generate<<<1, 256, 0, h->stream>>>(S.d_window, nullptr, chunk);
        RX_CHECK_CUDA(h, cudaGetLastError());
        todo -= (unsigned long long)chunk;
        S.consumed += (unsigned long long)chunk;
    }
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    return RX_OK;
}

struct MixTrace {   // RX_TRACE_MIX=1: device-time breakdown of one swap-all call (development aid)
    cudaEvent_t ev[10]; const char *name[10]; int n = 0; bool on = false; cudaStream_t st;
    void init(cudaStream_t s_) { st = s_; on = getenv("RX_TRACE_MIX") != nullptr; }
    void mark(const char *what) { if (!on || n >= 10) return; cudaEventCreate(&ev[n]); cudaEventRecord(ev[n], st); name[n++] = what; }
    void dump() {
        if (!on) return;
        cudaStreamSynchronize(st);
        for (int i = 1; i < n; i++) { float ms = 0; cudaEventElapsedTime(&ms, ev[i - 1], ev[i]); fprintf(stderr, "[mix trace] %-22s %9.3f ms\n", name[i], ms); }
        for (int i = 0; i < n; i++) cudaEventDestroy(ev[i]);
    }
};

static inline bool is_pow2(int k) { return k >= 2 && (k & (k - 1)) == 0; }

// Which walkers run a swap-all call, a function of K alone:
//   K                                 bulk of a pass          tail of a pass          records                counts from
//   power of two, 2 .. 256            k_mix_walk2             k_mix_walk_pow2<true>   SlotRec2               k_mix_count_slots + k_mix_count
//   power of two, 512 .. 16384        k_mix_walk_pow2<false>  (same kernel)           SlotRec                k_mix_count
//   not a power of two, 3 .. 255      k_mix_walk2c            k_mix_walk_serial       SlotRec2 per candidate k_mix_count_slots
//   not a power of two, 257 .. 4095   k_mix_walk_any          k_mix_walk_serial       WordRec                k_mix_count
//   anything else                     k_mix_walk_serial
// RX_WALK_SERIAL=1 gives every K that is not a power of two to the plain loop.
enum WalkPlan { PLAN_SERIAL = 0, PLAN_FILTER, PLAN_L2, PLAN_CAND, PLAN_WORDS };

// Dynamic shared memory of every walker launch.  The walker is one latency-bound CTA: it claims (almost) a whole SM's shared
// memory so that no other CTA -- in particular the stream generator that runs concurrently on the side stream -- is scheduled
// onto the same SM and steals issue slots (226 KB + the walker's static shared memory + the generator's 8 KB exceed 228 KB).
#define WALK_SMEM (226 * 1024)

static int walk_plan(rx_engine *h, int K, WalkPlan *plan) {
    if (is_pow2(K) && K <= (1 << LOG_STATE_BITS)) *plan = K <= 256 ? PLAN_FILTER : PLAN_L2;
    else if (K >= 3 && K <= ANY_MAX_K && !getenv("RX_WALK_SERIAL")) *plan = K < 256 ? PLAN_CAND : PLAN_WORDS;
    else *plan = PLAN_SERIAL;
    size_t image_smem = 0;   // the layouts that hold the 24-bit row image (213 KB at K = 256)
    if (*plan == PLAN_FILTER)   // k_mix_walk_pow2<true>: ring, diag, rowabs, perm, image; k_mix_walk2: ring, {state, diag}, image
        image_smem = std::max((size_t)RING * 16 + (size_t)K * (2 * sizeof(double) + sizeof(int)) + (size_t)3 * K * K,
                              (size_t)W2_RING * 16 + (size_t)K * sizeof(W2Replica) + (size_t)3 * K * K);
    if (*plan == PLAN_CAND)     // k_mix_walk2c: ring, {state, diag}, image rows padded to an even length
        image_smem = (size_t)W2_RING * 16 + (size_t)K * sizeof(W2Replica) + (size_t)((3 * K + 1) & ~1) * K;
    if (image_smem > WALK_SMEM) RX_FAIL(h, RX_ERR_INVALID, "internal: the row image does not fit the walker's shared memory");
    return RX_OK;
}

static inline size_t pass_need(long long remaining, WalkPlan plan) {
    const bool anyk = plan == PLAN_CAND || plan == PLAN_WORDS;
    const size_t chunk_words = anyk ? (size_t)1 << 25 : (size_t)1 << 26;  // words per pass (any K: 16 bytes of records per word)
    const bool slots = plan == PLAN_FILTER || plan == PLAN_L2;
    size_t need = slots ? (size_t)(4 * remaining + 160) : (size_t)(8 * remaining + 512);
    if (need > chunk_words) need = chunk_words;
    if (need < 512) need = 512;
    return need;
}

// Top the stream up to what a pass over `remaining` attempts may consume and build the plan's records from it, on stream
// `st`.  Both are state independent, so for the NEXT mixing call this runs on the side stream while the replicas are
// being propagated.
static int prepare_pass(rx_engine *h, MTStream &S, long long remaining, WalkPlan plan, int K, cudaStream_t st, int *launches) {
    const bool anyk = plan == PLAN_CAND || plan == PLAN_WORDS;   // records per word (candidate) rather than per slot
    const size_t need = pass_need(remaining, plan);
    int rc = stream_reserve(h, S, 2 * need + 1024);   // room for the words generated ahead while the walker runs
    if (rc) return rc;
    rc = stream_fill(h, S, need, launches, st);
    if (rc) return rc;
    if (plan != PLAN_SERIAL) {
        const long long nslots = anyk ? (long long)S.avail : (long long)(S.avail / 2);   // records: per slot, or per word
        if ((size_t)nslots > h->slots_cap) {
            // size for the largest stream the buffer can ever hold (2 * need + 1024 words), so that the slightly different
            // `avail` of every iteration never triggers another cudaFree/cudaMalloc (tens of ms each, device-synchronising)
            size_t want = anyk ? S.cap : (S.cap + 1) / 2;
            if (want < (size_t)nslots) want = (size_t)nslots;
            RX_CHECK_CUDA(h, cudaDeviceSynchronize());
            cudaFree(h->d_slots);
            cudaFree(h->d_log);
            h->d_slots = nullptr; h->d_log = nullptr;
            h->slots_cap = 0;
            RX_CHECK_CUDA(h, cudaMalloc(&h->d_slots, want * sizeof(SlotRec)));
            RX_CHECK_CUDA(h, cudaMalloc(&h->d_log, want * sizeof(uint32_t)));
            cudaFree(h->d_slotlog);
            h->d_slotlog = nullptr;
            RX_CHECK_CUDA(h, cudaMalloc(&h->d_slotlog, want * sizeof(uint32_t)));
            h->slots_cap = want;
        }
        if (plan == PLAN_CAND && (!h->d_cpos || h->ctile_cap < h->slots_cap)) {
            RX_CHECK_CUDA(h, cudaDeviceSynchronize());
            cudaFree(h->d_cpos); cudaFree(h->d_ctile);
            h->d_cpos = nullptr; h->d_ctile = nullptr;
            RX_CHECK_CUDA(h, cudaMalloc(&h->d_cpos, (h->slots_cap + 8) * sizeof(uint32_t)));
            RX_CHECK_CUDA(h, cudaMalloc(&h->d_ctile, (h->slots_cap / CAND_TILE + 8) * sizeof(uint32_t)));
            h->ctile_cap = h->slots_cap;
        }
        if (plan == PLAN_CAND) {
            // candidate coordinates (rx_walk2c.cuh): flag + count per tile, scan, scatter, one record per candidate index
            int nbits = 0;
            for (unsigned m = (unsigned)(K - 1); m; m >>= 1) nbits++;
            const uint32_t mask = 0xffffffffu >> (32 - nbits);
            const int ntiles = (int)((nslots + CAND_TILE - 1) / CAND_TILE);
            uint32_t *d_ncand = h->d_ctile + (h->ctile_cap / CAND_TILE + 4);
            k_cand_count<<<ntiles, 256, 0, st>>>(S.d_words, nslots, K, mask, h->d_ctile);
            k_cand_scan<<<1, 1024, 0, st>>>(h->d_ctile, ntiles, d_ncand);
            k_cand_scatter<<<ntiles, 256, 0, st>>>(S.d_words, nslots, K, mask, h->d_ctile, h->d_cpos);
            k_cand_records<<<(unsigned)((nslots + 255) / 256), 256, 0, st>>>(S.d_words, h->d_cpos, d_ncand, mask, (SlotRec2 *)h->d_slots);
            *launches += 3;
        } else if (plan == PLAN_WORDS) {
            static_assert(sizeof(WordRec) == sizeof(SlotRec), "all record formats share the d_slots buffer");
            int nbits = 0;
            for (unsigned m = (unsigned)(K - 1); m; m >>= 1) nbits++;
            k_words_build<<<(unsigned)((nslots + 255) / 256), 256, 0, st>>>(S.d_words, nslots, K, 0xffffffffu >> (32 - nbits), (WordRec *)h->d_slots);
        } else if (plan == PLAN_FILTER)
            k_slots_build2<<<(unsigned)((nslots + 255) / 256), 256, 0, st>>>(S.d_words, nslots, (uint32_t)(K - 1), (SlotRec2 *)h->d_slots);
        else
            k_slots_build<<<(unsigned)((nslots + 255) / 256), 256, 0, st>>>(S.d_words, nslots, (uint32_t)(K - 1), h->d_slots);
        RX_CHECK_CUDA(h, cudaGetLastError());
        (*launches)++;
    }
    h->slots_for_avail = S.avail;
    return RX_OK;
}

// Count matrices of a pass from a commit log: the sparse one indexed by slot or candidate (k_mix_walk2, k_mix_walk2c),
// entries [0, n), or the dense one of k_mix_walk_pow2 and k_mix_walk_any, n entries.
static int launch_count(rx_engine *h, bool sparse, long long n, int M, int *launches) {
    if (n <= 0) return RX_OK;
    long long nb = (n + 255) / 256;
    if (nb > 148 * 16) nb = 148 * 16;
    if (sparse) k_mix_count_slots<<<(unsigned)nb, 256, 0, h->stream>>>(h->d_slotlog, 0, n, M, h->d_nacc, h->d_nprop);
    else k_mix_count<<<(unsigned)nb, 256, 0, h->stream>>>(h->d_log, n, M, h->d_nacc, h->d_nprop);
    RX_CHECK_CUDA(h, cudaGetLastError());
    (*launches)++;
    return RX_OK;
}

// mix_stats[4]: device time of the walker launches between ev_walk[0] and ev_walk[1], in us (after a stream synchronise)
static void add_walker_time(rx_engine *h) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, h->ev_walk[0], h->ev_walk[1]) == cudaSuccess) h->mix_stats[4] += (long long)(ms * 1e3f);
}

int rxi_mix_swap_all(rx_engine *h, long long nswap, int *launches) {
    MTStream &S = h->streams[RX_STREAM_NUMBA];
    if (!S.seeded) RX_FAIL(h, RX_ERR_INVALID, "rx_mix_swap_all: the numba MT19937 stream has not been seeded (rx_mix_seed)");
    const int K = h->cfg.n_replicas, M = h->cfg.n_states;
    if (K != M) RX_FAIL(h, RX_ERR_INVALID, "rx_mix_swap_all: requires n_replicas == n_states");
    const size_t mm = (size_t)M * M * sizeof(unsigned long long);
    MixTrace tr; tr.init(h->stream); tr.mark("enter");
    RX_CHECK_CUDA(h, cudaMemsetAsync(h->d_nacc, 0, mm, h->stream));
    RX_CHECK_CUDA(h, cudaMemsetAsync(h->d_nprop, 0, mm, h->stream));
    tr.mark("memsets");
    if (nswap <= 0) return RX_OK;
    if (K == 1) {  // randint(1) draws nothing, log_p == 0: every attempt is an accepted no-op
        unsigned long long two_n = 2ull * (unsigned long long)nswap;
        RX_CHECK_CUDA(h, cudaMemcpyAsync(h->d_nacc, &two_n, 8, cudaMemcpyHostToDevice, h->stream));
        RX_CHECK_CUDA(h, cudaMemcpyAsync(h->d_nprop, &two_n, 8, cudaMemcpyHostToDevice, h->stream));
        RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
        return RX_OK;
    }
    WalkPlan plan;
    int rc = walk_plan(h, K, &plan);
    if (rc) return rc;
    const bool pow2 = plan == PLAN_FILTER || plan == PLAN_L2;   // slot records; the walkers finish every pass themselves
    int logK = 0;
    while ((1 << logK) < K) logK++;
    const size_t smem_serial = (size_t)K * sizeof(int);
    if (smem_serial > 48 * 1024) RX_CHECK_CUDA(h, cudaFuncSetAttribute(k_mix_walk_serial, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_serial));
    auto claim = [](const void *walker) { return cudaFuncSetAttribute(walker, cudaFuncAttributeMaxDynamicSharedMemorySize, WALK_SMEM); };
    if (plan == PLAN_FILTER) {
        RX_CHECK_CUDA(h, claim((const void *)k_mix_walk2));
        RX_CHECK_CUDA(h, claim((const void *)k_mix_walk_pow2<true>));
    }
    if (plan == PLAN_L2) RX_CHECK_CUDA(h, claim((const void *)k_mix_walk_pow2<false>));
    if (plan == PLAN_CAND) RX_CHECK_CUDA(h, claim((const void *)k_mix_walk2c));
    if (plan == PLAN_WORDS) RX_CHECK_CUDA(h, claim((const void *)k_mix_walk_any));
    tr.mark("func attributes");
    if (plan == PLAN_FILTER || plan == PLAN_CAND) {
        if (!h->d_filt) {
            RX_CHECK_CUDA(h, cudaMalloc(&h->d_filt, (size_t)3 * K * K + 16));
            RX_CHECK_CUDA(h, cudaMalloc(&h->d_filt_scale, sizeof(double) * 2 * K));
        }
        // row image + |row minimum| for the per-lane error bound; non-finite or astronomically large entries only send the
        // lanes that touch them to the exact path (no host round trip, no global fallback)
        k_mix_filter_build<<<K, 256, 0, h->stream>>>(h->d_u, K, h->d_filt, h->d_filt_scale, h->d_filt_scale + K);
        RX_CHECK_CUDA(h, cudaGetLastError());
        (*launches)++;
    }
    tr.mark("filter build");
    long long remaining = nswap;
    h->mix_stats[0] = h->mix_stats[1] = h->mix_stats[2] = h->mix_stats[4] = h->mix_stats[5] = 0;
    const uint64_t consumed0 = S.consumed;
    const size_t chunk_words = (size_t)1 << 26;
    while (remaining > 0) {
        const size_t need = pass_need(remaining, plan);
        if (h->prepared && h->prepared_plan == plan && S.avail >= need && h->slots_for_avail == S.avail) {
            // produced on the side stream while the replicas were propagating
            RX_CHECK_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_prepared, 0));
            float ms = 0;
            const double tw0 = rx_wall_us();
            if (cudaEventSynchronize(h->ev[7]) == cudaSuccess && cudaEventElapsedTime(&ms, h->ev[6], h->ev[7]) == cudaSuccess)
                h->phase_ms[3] += ms;
            h->mix_stats[5] += (long long)(rx_wall_us() - tw0);
        } else {
            if (h->prepared) RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream_rng));
            rc = prepare_pass(h, S, remaining, plan, K, h->stream, launches);
            if (rc) return rc;
        }
        h->prepared = false;
        tr.mark("prepared/built");
        MixCtl ctl = {0, remaining, 0, 0, 0, 0, 0};
        RX_CHECK_CUDA(h, cudaMemcpyAsync(h->d_ctl, &ctl, sizeof(ctl), cudaMemcpyHostToDevice, h->stream));
        size_t consumed_words;
        if (pow2) {
            const long long nslots = (long long)(S.avail / 2);
            // While the walker runs (it only reads words [0, avail)), generate on the side stream about as many words
            // as the previous call consumed: they are appended behind the valid region and adopted afterwards.
            size_t ahead = 0;
            if (!getenv("RX_NO_ASYNC_RNG") && h->last_consumed > 0 && S.avail + h->last_consumed <= S.cap) {
                ahead = h->last_consumed;
                k_mt_generate<<<1, 256, 0, h->stream_rng>>>(S.d_window, S.d_words + S.avail, (long long)ahead);
                RX_CHECK_CUDA(h, cudaGetLastError());
                RX_CHECK_CUDA(h, cudaEventRecord(h->ev_prepared, h->stream_rng));
                *launches += 1;
            }
            RX_CHECK_CUDA(h, cudaEventRecord(h->ev_walk[0], h->stream));
            if (plan == PLAN_FILTER) {
                static_assert(sizeof(SlotRec2) == sizeof(SlotRec), "both record formats share the d_slots buffer");
                // sparse commit log: one word per slot, zero = no attempt started there
                RX_CHECK_CUDA(h, cudaMemsetAsync(h->d_slotlog, 0, (size_t)nslots * sizeof(uint32_t), h->stream));
                k_mix_walk2<<<1, W2_THREADS, WALK_SMEM, h->stream>>>((const SlotRec2 *)h->d_slots, S.d_words, (unsigned)nslots, h->d_u, K, logK, h->d_perm, h->d_slotlog, h->d_filt, h->d_filt_scale, h->d_ctl);
                RX_CHECK_CUDA(h, cudaGetLastError());
                *launches += 1;
                k_mix_walk_pow2<true><<<1, 64, WALK_SMEM, h->stream>>>(h->d_slots, S.d_words, (unsigned)nslots, h->d_u, K, logK, h->d_perm, h->d_log, h->d_filt, h->d_filt_scale, h->d_ctl);
            } else
                k_mix_walk_pow2<false><<<1, 64, WALK_SMEM, h->stream>>>(h->d_slots, S.d_words, (unsigned)nslots, h->d_u, K, logK, h->d_perm, h->d_log, nullptr, nullptr, h->d_ctl);
            RX_CHECK_CUDA(h, cudaGetLastError());
            RX_CHECK_CUDA(h, cudaEventRecord(h->ev_walk[1], h->stream));
            tr.mark("walker");
            *launches += 1;
            RX_CHECK_CUDA(h, cudaMemcpyAsync(&ctl, h->d_ctl, sizeof(ctl), cudaMemcpyDeviceToHost, h->stream));
            RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
            add_walker_time(h);
            consumed_words = (size_t)(2 * ctl.head);
            if (ahead) {   // adopt the words generated during the walk
                RX_CHECK_CUDA(h, cudaStreamWaitEvent(h->stream, h->ev_prepared, 0));
                S.avail += ahead;
            }
            if (plan == PLAN_FILTER) {   // k_mix_walk2 logs by slot, up to the one it reached
                rc = launch_count(h, true, ctl.head, M, launches);
                if (rc) return rc;
            }
            rc = launch_count(h, false, ctl.log_count, M, launches);
            if (rc) return rc;
            tr.mark("adopt-ahead + count");
        } else {
            if (plan != PLAN_SERIAL) {
                // bulk of the pass; what the walker leaves -- the last words of the pass -- is finished by the plain loop below
                RX_CHECK_CUDA(h, cudaEventRecord(h->ev_walk[0], h->stream));
                if (plan == PLAN_CAND) {
                    RX_CHECK_CUDA(h, cudaMemsetAsync(h->d_slotlog, 0, S.avail * sizeof(uint32_t), h->stream));
                    k_mix_walk2c<<<1, W2_THREADS, WALK_SMEM, h->stream>>>((const SlotRec2 *)h->d_slots, S.d_words, h->d_cpos,
                                                                          h->d_ctile + (h->ctile_cap / CAND_TILE + 4), h->d_u, K, h->d_perm,
                                                                          h->d_slotlog, h->d_filt, h->d_filt_scale, h->d_ctl);
                } else
                    k_mix_walk_any<<<1, 64, WALK_SMEM, h->stream>>>((const WordRec *)h->d_slots, S.d_words, (unsigned)S.avail, h->d_u, K, h->d_perm, h->d_log, h->d_ctl);
                RX_CHECK_CUDA(h, cudaGetLastError());
                RX_CHECK_CUDA(h, cudaEventRecord(h->ev_walk[1], h->stream));
                *launches += 1;
            }
            k_mix_walk_serial<<<1, 32, smem_serial, h->stream>>>(S.d_words, (long long)S.avail, h->d_u, K, M, h->d_perm, h->d_nacc,
                                                               h->d_nprop, h->d_ctl);
            RX_CHECK_CUDA(h, cudaGetLastError());
            *launches += 1;
            RX_CHECK_CUDA(h, cudaMemcpyAsync(&ctl, h->d_ctl, sizeof(ctl), cudaMemcpyDeviceToHost, h->stream));
            RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
            consumed_words = (size_t)ctl.head;
            if (plan != PLAN_SERIAL) {
                add_walker_time(h);
                // k_mix_walk2c logs by candidate index, up to the one it reached
                rc = plan == PLAN_CAND ? launch_count(h, true, ctl.aux, M, launches) : launch_count(h, false, ctl.log_count, M, launches);
                if (rc) return rc;
            }
        }
        if (ctl.remaining == remaining && consumed_words == 0 && need >= chunk_words)
            RX_FAIL(h, RX_ERR_INVALID, "internal: mixing made no progress");
        remaining = ctl.remaining;
        h->mix_stats[0] += ctl.rounds;
        h->mix_stats[1] += ctl.slow_exp;
        h->mix_stats[2] += 1;
        rc = stream_consume(h, S, consumed_words, launches);
        if (rc) return rc;
        tr.mark("consume copy");
    }
    tr.dump();
    h->mix_stats[3] = (long long)(S.consumed - consumed0);
    h->last_consumed = (size_t)(S.consumed - consumed0);
    if (!getenv("RX_NO_ASYNC_RNG")) {
        // overlap the next call's stream generation + slot records with whatever runs next on the main stream
        RX_CHECK_CUDA(h, cudaEventRecord(h->ev_consumed, h->stream));
        RX_CHECK_CUDA(h, cudaStreamWaitEvent(h->stream_rng, h->ev_consumed, 0));
        RX_CHECK_CUDA(h, cudaEventRecord(h->ev[6], h->stream_rng));
        int l2 = 0;
        int rc2 = prepare_pass(h, S, nswap, plan, K, h->stream_rng, &l2);
        h->prepared_plan = plan;
        if (rc2) return rc2;
        RX_CHECK_CUDA(h, cudaEventRecord(h->ev[7], h->stream_rng));
        RX_CHECK_CUDA(h, cudaEventRecord(h->ev_prepared, h->stream_rng));
        h->phase_launches[3] += l2;
        h->prepared = true;
    }
    return RX_OK;
}

int rxi_mix_swap_neighbors(rx_engine *h, int *launches) {
    MTStream &S = h->streams[RX_STREAM_NUMPY];
    if (!S.seeded) RX_FAIL(h, RX_ERR_INVALID, "rx_mix_swap_neighbors: the numpy MT19937 stream has not been seeded (rx_mix_seed)");
    const int K = h->cfg.n_replicas, M = h->cfg.n_states;
    if (K != M) RX_FAIL(h, RX_ERR_INVALID, "rx_mix_swap_neighbors: requires n_replicas == n_states");
    const size_t mm = (size_t)M * M * sizeof(unsigned long long);
    RX_CHECK_CUDA(h, cudaMemsetAsync(h->d_nacc, 0, mm, h->stream));
    RX_CHECK_CUDA(h, cudaMemsetAsync(h->d_nprop, 0, mm, h->stream));
    int rc = stream_fill(h, S, (size_t)K + 64, launches, h->stream);
    if (rc) return rc;
    const size_t smem = 2 * (size_t)K * sizeof(int);
    if (smem > 48 * 1024)
        RX_CHECK_CUDA(h, cudaFuncSetAttribute(k_mix_neighbors, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    MixCtl ctl = {0, 0, 0, 0, 0, 0};
    RX_CHECK_CUDA(h, cudaMemcpyAsync(h->d_ctl, &ctl, sizeof(ctl), cudaMemcpyHostToDevice, h->stream));
    k_mix_neighbors<<<1, 32, smem, h->stream>>>(S.d_words, (long long)S.avail, h->d_u, K, M, h->d_perm, h->d_nacc, h->d_nprop,
                                              h->d_ctl);
    RX_CHECK_CUDA(h, cudaGetLastError());
    (*launches)++;
    RX_CHECK_CUDA(h, cudaMemcpyAsync(&ctl, h->d_ctl, sizeof(ctl), cudaMemcpyDeviceToHost, h->stream));
    RX_CHECK_CUDA(h, cudaStreamSynchronize(h->stream));
    return stream_consume(h, S, (size_t)ctl.head, launches);
}

void rxi_mix_free(rx_engine *h) {
    for (int s = 0; s < 2; s++) {
        cudaFree(h->streams[s].d_window);
        cudaFree(h->streams[s].d_words);
        cudaFree(h->streams[s].d_words_alt);
    }
    cudaFree(h->d_slots);
    cudaFree(h->d_log);
    cudaFree(h->d_slotlog);
    cudaFree(h->d_cpos);
    cudaFree(h->d_ctile);
    cudaFree(h->d_filt);
    cudaFree(h->d_filt_scale);
    cudaFree(h->d_ctl);
}

#include "rx_sams.cuh"
