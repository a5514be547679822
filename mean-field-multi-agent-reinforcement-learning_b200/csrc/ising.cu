// K6: Ising-model tabular mean-field Q-learning, one fused sweep per launch.
//
// Reference (pure Python): main_MFQ_Ising.py:105-134 (loop body), :55-67 (boltzman_explore),
// examples/ising_model/Ising.py:7-58 (4-neighbour torus mask), :101-111 (reward), :113-118 (observation),
// multiagent/core.py:99-125 (spin <- action), multiagent/environment.py:49-78.
// Per site i of an L x L torus, per step:
//     s   = number of up neighbours in the OLD lattice            (obs of the previous step)
//     p_a = exp(Q[i,s,a] / T) / sum_a' exp(Q[i,s,a'] / T);  a = [u >= p_0]   (np.random.choice(2, 1, p))
//     spin_i <- a                                                  (all sites, synchronously)
//     r   = 0.5 * sigma_i * sum_nbr sigma_j on the NEW lattice,  sigma = 2 spin - 1
//     Q[i,s,a] <- Q[i,s,a] + lr * (r - Q[i,s,a])                   (sites in the act group)
//
// Layout in HBM:  spins int8 [B][L][L];  Q  T [B][5][L*L][2]  (one plane per neighbour count s, the action
// pair of a site adjacent: a site reads its pair with ONE 8-byte load and rewrites one half of it, and a
// warp walking a lattice row touches consecutive pairs of one plane whenever neighbouring sites share s.
// Measured on B200 against the [5][2][N] split-plane layout in the disordered phase: fewer partially
// used 32-byte sectors; an AoS [site][5][2] row (40 B) would cost a full sector read + write per site).
//
// Mapping: one CTA per lattice, one thread per lattice COLUMN, warps = ceil(L / 32).  Both the old and
// the new lattice live in shared memory bit-packed (__ballot_sync packs a warp's 32 columns into one
// word), so a 256 x 256 lattice costs 2 x 8 KB and eight CTAs fit per SM.  Rows are swept in bands of
// RB rows: the band's Q pairs are loaded with 2*RB independent loads per thread in flight, actions are
// drawn and the band's new bits published, and after one barrier the rows whose three new neighbour
// rows are known are finalised from registers (reward, Q update) -- Q is read once and written once per
// site.  Row 0 waits in registers for row L-1 (torus wrap).  Algorithmic traffic per site-step:
// 2 x 4 (Q read) + 4 (Q write) + 1 + 1 (spin) = 14 B in fp32.
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cstdlib>
#include <map>
#include <mutex>
#include <type_traits>

#include "../../include/mfmarl_batched.h"
#include "rng.cuh"
#include "engine.h"

namespace mfmarl {

constexpr int kIsingRB = 4;   // rows per band == uniforms per Philox call

template <typename T>
struct IsingArgs {
    int B, L;
    int8_t *spins;          // [B][L][L] in/out
    T *Q;                   // [B][5][L*L][2] in/out
    T temperature, lr;
    const T *u;             // optional injected uniforms [B][L*L] (test hook); else Philox
    const uint8_t *mask;    // optional act-group mask [B][L*L]; null = every site updates Q
    uint32_t seed, lattice_base, step;
    int32_t *n_up;          // [B] out: up spins after the sweep
    T *reward_sum;          // [B] out: sum_i r_i
    T *mse;                 // [B] out: sum over updated sites (Q_new - target)^2 / N   (main_MFQ_Ising.py:127-134)
};

template <typename T> struct Pair;
template <> struct Pair<float> { typedef float2 type; };
template <> struct Pair<double> { typedef double2 type; };

template <typename T> __device__ __forceinline__ T uniform_from_bits(uint32_t hi, uint32_t lo);
template <> __device__ __forceinline__ float uniform_from_bits<float>(uint32_t hi, uint32_t) {
    return __uint2float_rz(hi) * (1.0f / 4294967296.0f);                  // round toward zero keeps it in [0, 1)
}
template <> __device__ __forceinline__ double uniform_from_bits<double>(uint32_t hi, uint32_t lo) {
    return ((double)(hi >> 5) * 67108864.0 + (double)(lo >> 6)) * (1.0 / 9007199254740992.0);   // 53 bits
}

// p_0 after numpy's own renormalisation: np.random.choice builds cdf = cumsum(p); cdf /= cdf[-1] and
// returns searchsorted(cdf, u, 'right')  =>  a = [u >= cdf_0].
__device__ __forceinline__ double action_threshold(double q0, double q1, double T) {
    const double e0 = exp(q0 / T), e1 = exp(q1 / T);
    const double denom = 0.0 + e0 + e1;                                   // denom = 0; denom += val (x2)
    const double p0 = e0 / denom, p1 = e1 / denom;
    return p0 / (p0 + p1);
}
// fp32 production mode.  a = [u >= p0] with p0 = e0/(e0+e1) = 1/(1 + e), e = exp((q1-q0)/T), is evaluated as
// u*(1 + e) >= 1, which needs neither the reciprocal nor the division: c = log2(e)/T is computed once per sweep,
// e = ex2.approx((q1-q0)*c), and u*e + u is one fma.  |error| of the
// implied threshold < 4e-6 for |q| <= 2, T >= 0.25, i.e. an action can differ from the fp64 reference only for
// draws that close to the threshold -- the same order as the fp32 rounding of u itself (2^-24).  Both fp32
// kernels (streaming and resident) share this function, so they agree bit for bit.
__device__ __forceinline__ float temperature_param(float T) { return __fdiv_rn(1.4426950408889634f, T); }
__device__ __forceinline__ double temperature_param(double T) { return T; }
__device__ __forceinline__ int draw_action(float u, float q0, float q1, float c) {
    float e;                                   // e = +inf at tiny T is fine: u * inf + u >= 1 for every u > 0
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"((q1 - q0) * c));
    return __fmaf_rn(u, e, u) >= 1.0f ? 1 : 0;
}
// the same decision with the uniform still scaled by 2^32 (m = u * 2^32, exactly): saves the rescaling multiply
__device__ __forceinline__ int draw_action_scaled(float m, float q0, float q1, float c) {
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"((q1 - q0) * c));
    return __fmaf_rn(m, e, m) >= 4294967296.0f ? 1 : 0;
}
// fp64 mode replays the reference's operation sequence
__device__ __forceinline__ int draw_action(double u, double q0, double q1, double T) {
    return u >= action_threshold(q0, q1, T) ? 1 : 0;
}

__device__ __forceinline__ int bit_at(const uint32_t *rows, int wpr, int r, int x) {
    return (rows[r * wpr + (x >> 5)] >> (x & 31)) & 1;
}

// PL: per-lattice temperatures, lattice b draws at temps[b] instead of A.temperature (mfi_step_lattices)
template <typename T, bool PL>
__device__ __forceinline__ void ising_sweep(const IsingArgs<T> A, const T *temps) {
    extern __shared__ __align__(16) uint32_t s_bits[];
    const int L = A.L, N = L * L, wpr = (L + 31) >> 5;
    uint32_t *s_old = s_bits, *s_new = s_bits + L * wpr;
    __shared__ int s_nup;
    __shared__ T s_rsum, s_mse;

    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int x = tid;                       // this thread's column
    const bool active = x < L;
    const size_t lbase = (size_t)b * N;
    int8_t *spins = A.spins + lbase;
    T *Q = A.Q + lbase * 10;
    const int xl = x == 0 ? L - 1 : x - 1, xr = x == L - 1 ? 0 : x + 1;

    if (tid == 0) { s_nup = 0; s_rsum = (T)0; s_mse = (T)0; }
    // ---- old lattice -> bits ----
#pragma unroll 8
    for (int r = 0; r < L; r++) {
        const int v = active ? spins[r * L + x] : 0;
        const uint32_t word = __ballot_sync(0xFFFFFFFFu, v != 0);
        if (lane == 0) s_old[r * wpr + w] = word;
    }
    __syncthreads();

    const T tparam = temperature_param(PL ? temps[b] : A.temperature);
    T keep_q[kIsingRB]; int keep_sa[kIsingRB];     // this band: selected Q value, s | a << 3
    T prev_q = (T)0; int prev_sa = 0;              // last row of the previous band
    T row0_q = (T)0; int row0_sa = 0;              // row 0, finalised last (needs row L-1)
    int nup = 0; T rsum = (T)0, mse = (T)0;

    auto finalize = [&](int r, T qsel, int sa) {
        const int s = sa & 7, a = sa >> 3, i = r * L + x;
        const int ru = r == 0 ? L - 1 : r - 1, rd = r == L - 1 ? 0 : r + 1;
        const int ups = bit_at(s_new, wpr, ru, x) + bit_at(s_new, wpr, rd, x) + bit_at(s_new, wpr, r, xl) +
                        bit_at(s_new, wpr, r, xr);
        const T reward = (T)0.5 * (T)(2 * a - 1) * (T)(2 * ups - 4);      // Ising.py:101-111
        spins[i] = (int8_t)a;
        nup += a; rsum += reward;
        if (A.mask == nullptr || A.mask[lbase + i]) {
            const T qn = qsel + A.lr * (reward - qsel);                    // main_MFQ_Ising.py:129-131
            Q[((size_t)s * N + i) * 2 + a] = qn;
            const T d = qn - (T)((2 - s) * (1 - 2 * a));                   // reward_target[s][a], :77-81
            mse += d * d;
        }
    };

    for (int r0 = 0; r0 < L; r0 += kIsingRB) {
        const int nrows = min(kIsingRB, L - r0);
        T q0[kIsingRB], q1[kIsingRB]; int sv[kIsingRB];
        // ---- neighbour counts on the OLD lattice and the band's Q pairs: 2*RB loads in flight ----
#pragma unroll
        for (int j = 0; j < kIsingRB; j++) {
            sv[j] = 0; q0[j] = (T)0; q1[j] = (T)0;
            if (j < nrows && active) {
                const int r = r0 + j, ru = r == 0 ? L - 1 : r - 1, rd = r == L - 1 ? 0 : r + 1;
                sv[j] = bit_at(s_old, wpr, ru, x) + bit_at(s_old, wpr, rd, x) + bit_at(s_old, wpr, r, xl) +
                        bit_at(s_old, wpr, r, xr);                         // Ising.py:113-118 + count_nonzero
                const size_t i = (size_t)r * L + x;
                const typename Pair<T>::type pr = *(const typename Pair<T>::type *)(Q + ((size_t)sv[j] * N + i) * 2);
                q0[j] = pr.x; q1[j] = pr.y;
            }
        }
        // ---- uniforms: one Philox call per thread per band, keyed (seed, lattice) x (column, band, step) ----
        T uu[kIsingRB];
        if (A.u != nullptr) {
#pragma unroll
            for (int j = 0; j < kIsingRB; j++)
                uu[j] = (j < nrows && active) ? A.u[lbase + (size_t)(r0 + j) * L + x] : (T)0;
        } else if (sizeof(T) == 4) {
            const uint4 rnd = philox4x32_10(make_uint4((uint32_t)x, (uint32_t)(r0 / kIsingRB), A.step, 0u),
                                            make_uint2(A.seed, A.lattice_base + (uint32_t)b));
            uu[0] = uniform_from_bits<T>(rnd.x, 0); uu[1] = uniform_from_bits<T>(rnd.y, 0);
            uu[2] = uniform_from_bits<T>(rnd.z, 0); uu[3] = uniform_from_bits<T>(rnd.w, 0);
        } else {
            const uint2 key = make_uint2(A.seed, A.lattice_base + (uint32_t)b);
            const uint4 r1 = philox4x32_10(make_uint4((uint32_t)x, (uint32_t)(r0 / kIsingRB), A.step, 0u), key);
            const uint4 r2 = philox4x32_10(make_uint4((uint32_t)x, (uint32_t)(r0 / kIsingRB), A.step, 1u), key);
            uu[0] = uniform_from_bits<T>(r1.x, r1.y); uu[1] = uniform_from_bits<T>(r1.z, r1.w);
            uu[2] = uniform_from_bits<T>(r2.x, r2.y); uu[3] = uniform_from_bits<T>(r2.z, r2.w);
        }
        // ---- Boltzmann draw, publish the band's new bits ----
#pragma unroll
        for (int j = 0; j < kIsingRB; j++) {
            int a = 0;
            if (j < nrows && active) a = draw_action(uu[j], q0[j], q1[j], tparam);
            const uint32_t word = __ballot_sync(0xFFFFFFFFu, a != 0);
            if (j < nrows && lane == 0) s_new[(r0 + j) * wpr + w] = word;
            keep_q[j] = a ? q1[j] : q0[j];
            keep_sa[j] = sv[j] | (a << 3);
        }
        __syncthreads();
        // ---- finalise every row whose three new neighbour rows are now known ----
        if (active) {
            if (r0 > 0) {
                if (r0 - 1 > 0) finalize(r0 - 1, prev_q, prev_sa);
            }
#pragma unroll
            for (int j = 0; j < kIsingRB; j++) {
                const int r = r0 + j;
                if (j < nrows - 1) {
                    if (r == 0) { row0_q = keep_q[j]; row0_sa = keep_sa[j]; }
                    else finalize(r, keep_q[j], keep_sa[j]);
                }
            }
        }
        // remember the band's last row for the next iteration
#pragma unroll
        for (int j = 0; j < kIsingRB; j++)
            if (j == nrows - 1) { prev_q = keep_q[j]; prev_sa = keep_sa[j]; }
    }
    if (active) {
        if (L > 1) finalize(L - 1, prev_q, prev_sa);   // needs row 0, published in the first band
        finalize(0, row0_q, row0_sa);                  // needs row L-1, published in the last band
    }

    // ---- per-lattice statistics: up count, reward sum, mse ----
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        nup += __shfl_xor_sync(0xFFFFFFFFu, nup, o);
        rsum += __shfl_xor_sync(0xFFFFFFFFu, rsum, o);
        mse += __shfl_xor_sync(0xFFFFFFFFu, mse, o);
    }
    if (lane == 0) { atomicAdd(&s_nup, nup); atomicAdd(&s_rsum, rsum); atomicAdd(&s_mse, mse); }
    __syncthreads();
    if (tid == 0) {
        if (A.n_up) A.n_up[b] = s_nup;
        if (A.reward_sum) A.reward_sum[b] = s_rsum;
        if (A.mse) A.mse[b] = s_mse / (T)N;
    }
}

template <typename T>
__global__ void __launch_bounds__(sizeof(T) == 8 ? 512 : 1024) k_ising(const IsingArgs<T> A) { ising_sweep<T, false>(A, nullptr); }
template <typename T>
__global__ void __launch_bounds__(sizeof(T) == 8 ? 512 : 1024) k_ising_lattices(const IsingArgs<T> A, const T *temps) {
    ising_sweep<T, true>(A, temps);
}

// temps: null = A.temperature for every lattice, else T [B] device (one temperature per lattice)
template <typename T>
static void launch_ising(const IsingArgs<T> &A, cudaStream_t st, const T *temps = nullptr) {
    const int L = A.L, wpr = (L + 31) >> 5;
    if (L < 3 || L > 1024) throw Fatal("ising: lattice side must be in [3, 1024]");
    if ((size_t)2 * L * wpr * sizeof(uint32_t) > 200 * 1024) throw Fatal("ising: lattice too large for the shared-memory bit planes");
    if (A.B < 1) throw Fatal("ising: need at least one lattice");
    if (sizeof(T) == 8 && L > 512) throw Fatal("ising: fp64 mode supports lattice sides up to 512");
    const int threads = wpr * 32;
    const size_t smem = (size_t)2 * L * wpr * sizeof(uint32_t);
    if (temps) {
        if (smem > 48 * 1024)
            MF_CUDA(cudaFuncSetAttribute(k_ising_lattices<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_ising_lattices<T><<<A.B, threads, smem, st>>>(A, temps);
    } else {
        if (smem > 48 * 1024)
            MF_CUDA(cudaFuncSetAttribute(k_ising<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_ising<T><<<A.B, threads, smem, st>>>(A);
    }
    MF_CUDA(cudaGetLastError());
}


// ----------------------------------------------------------------------------------------------
// K6r: RESIDENT variant -- K sweeps per launch with the Q table in shared memory.
//
// The streaming kernel above moves every site's Q pair through HBM once per sweep (14 B/site-step
// algorithmic, 45-60 B real in the disordered phase because the plane index s is data dependent and
// 32-byte sectors are only partly used).  Here a lattice is cut into C horizontal strips, one CTA each,
// the C CTAs forming one thread-block cluster; a CTA keeps its strip of Q ([5][rows*L][2], up to 160 KB) and
// two bit-packed spin buffers (ping-pong, each with one halo row above and below) in shared memory for all
// K sweeps.  HBM traffic drops to (80 B load + 80 B store) / K per site-step; the kernel is bound by issue
// slots, so the sweep is written to need few instructions and ONE cluster barrier:
//   * the up-neighbour count of the lattice after sweep k-1 is both the reward input of sweep k-1 and the
//     Q-row index s of sweep k, so one fused phase per barrier does: count -> finish sweep k-1 (reward,
//     Q update in shared memory, statistics) -> draw sweep k (Q pair, Boltzmann draw) -> publish the new bits;
//   * a CTA PUSHES its two boundary rows into the neighbours' halo rows (st.shared::cluster is fire and
//     forget), so every read is local -- no 200-cycle DSMEM load sits on the critical path;
//   * the barrier is split (barrier.cluster.arrive.release ... wait.acquire) and the Philox draws of the next
//     sweep plus the statistics flush are computed between the two halves;
//   * left/right neighbours come from the row's ballot word (kept in a register) and the two adjacent words
//     with one funnel shift each; up/down inside a thread's 4-row band come from its own registers.
// A sweep reads buffer `cur` and writes buffer `cur^1`; a CTA can be at most one barrier ahead of its
// neighbours and by then they have finished reading, so the ping-pong needs no second barrier.
// Draws use the same Philox keys as the streaming kernel -- (seed, lattice) x (column, global row band, step) --
// so K resident sweeps equal K streaming launches bit for bit.
// C = 1 covers lattices whose whole Q fits one CTA (L <= 64 in fp32; the reference's 20 x 20 case);
// 256 x 256 uses C = 16 (16 rows per CTA, 1024 threads = 256 columns x 4 bands).
// ----------------------------------------------------------------------------------------------
}  // namespace mfmarl
#include <cooperative_groups.h>
namespace mfmarl {
namespace cg = cooperative_groups;

template <typename T>
struct IsingRunArgs {
    int B, L, K, rows_per;         // lattices, side, sweeps, rows per CTA (= L / cluster size)
    int8_t *spins; T *Q;
    const T *temperatures;          // [K] device
    T lr;
    const T *u;                     // optional injected uniforms [K][B][L*L]
    const uint8_t *mask;            // optional act groups [K][B][L*L] (act_rate < 1): which sites update Q in sweep k
    uint32_t seed, lattice_base, step0;
    int32_t *n_up;                  // [K][B] out, must be zeroed by the caller
    T *reward_sum;                  // [K][B] out or null, zeroed by the caller
};

__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }

template <typename T>
__device__ __forceinline__ void ising_uniforms(T (&uu)[kIsingRB], uint32_t x, uint32_t gband, uint32_t step, uint2 key) {
    if (sizeof(T) == 4) {
        const uint4 rnd = philox4x32_10(make_uint4(x, gband, step, 0u), key);
        uu[0] = uniform_from_bits<T>(rnd.x, 0); uu[1] = uniform_from_bits<T>(rnd.y, 0);
        uu[2] = uniform_from_bits<T>(rnd.z, 0); uu[3] = uniform_from_bits<T>(rnd.w, 0);
    } else {
        const uint4 r1 = philox4x32_10(make_uint4(x, gband, step, 0u), key);
        const uint4 r2 = philox4x32_10(make_uint4(x, gband, step, 1u), key);
        uu[0] = uniform_from_bits<T>(r1.x, r1.y); uu[1] = uniform_from_bits<T>(r1.z, r1.w);
        uu[2] = uniform_from_bits<T>(r2.x, r2.y); uu[3] = uniform_from_bits<T>(r2.z, r2.w);
    }
}

// FAST: L % 32 == 0 and rows % 4 == 0 -- every thread owns 4 live sites and a row's x-wrap is a word wrap.
// PL: A.temperatures is [K][B] (lattice b draws sweep k at row k, column b) instead of [K].
template <typename T, bool FAST, bool PL>
__device__ __forceinline__ void ising_resident_sweeps(const IsingRunArgs<T> A) {
    extern __shared__ __align__(16) unsigned char s_raw[];
    cg::cluster_group cluster = cg::this_cluster();
    const int C = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
    const int L = A.L, N = L * L, wpr = (L + 31) >> 5, LP = wpr * 32, rows = A.rows_per;
    const int b = blockIdx.x / C, row0 = rank * rows;
    const int strip = rows * L;                          // sites in this CTA's strip
    const int HR = rows + 2;                             // bit rows per buffer: halo, rows, halo

    T *s_q = (T *)s_raw;                                 // [5][strip][2]
    uint32_t *s_bits = (uint32_t *)(s_raw + (size_t)5 * strip * 2 * sizeof(T));   // [2][HR][wpr]
    int *s_stat = (int *)(s_bits + 2 * HR * wpr);        // [2][2]: (up count, reward sum) of sweep parity

    const int tid = threadIdx.x, lane = tid & 31;
    const int x = tid % LP, band = tid / LP, w = x >> 5;  // column, band (4 rows) inside the strip
    const bool active = FAST || x < L;
    const int xl = x == 0 ? L - 1 : x - 1, xr = x == L - 1 ? 0 : x + 1;
    const int wl = w == 0 ? wpr - 1 : w - 1, wr = w == wpr - 1 ? 0 : w + 1;
    const size_t lbase = (size_t)b * N;
    const int rb = band * kIsingRB;                       // first local row of this thread
    const int up_rank = (rank + C - 1) % C, dn_rank = (rank + 1) % C;
    uint32_t *up_bits = cluster.map_shared_rank(s_bits, up_rank);   // == s_bits when C == 1
    uint32_t *dn_bits = cluster.map_shared_rank(s_bits, dn_rank);

    // publish one 32-column word of local row r into buffer `which`: own copy + the neighbour's halo row
    auto publish = [&](int which, int r, uint32_t word) {
        const int o = which * HR * wpr + w;
        s_bits[o + (r + 1) * wpr] = word;
        if (r == 0) up_bits[o + (rows + 1) * wpr] = word;            // I am the row below up_rank's last row
        if (r == rows - 1) dn_bits[o] = word;                         // ... and the row above dn_rank's first
    };

    if (tid < 4) s_stat[tid] = 0;
    // ---- load: Q strip (5 contiguous plane slices) and spins -> bits (buffer 0) ----
    for (int sp = 0; sp < 5; sp++) {
        const T *src = A.Q + (lbase * 5 + (size_t)sp * N + (size_t)row0 * L) * 2;
        T *dst = s_q + (size_t)sp * strip * 2;
        if (sizeof(T) == 4 && (strip & 1) == 0) {
            const float4 *s4 = (const float4 *)src; float4 *d4 = (float4 *)dst;
            for (int i = tid; i < strip / 2; i += blockDim.x) d4[i] = s4[i];
        } else {
            for (int i = tid; i < strip * 2; i += blockDim.x) dst[i] = src[i];
        }
    }
    int a_cur[kIsingRB];            // this thread's spins in the current lattice
    uint32_t w_cur[kIsingRB];       // the 32-column words those spins live in (ballot result)
    cluster.sync();                 // everybody's shared memory exists before the first remote store
#pragma unroll
    for (int j = 0; j < kIsingRB; j++) {
        const int r = rb + j;
        const bool live = FAST || (r < rows && active);
        a_cur[j] = live ? (int)A.spins[lbase + (size_t)(row0 + r) * L + x] : 0;
        w_cur[j] = __ballot_sync(0xFFFFFFFFu, a_cur[j] != 0);
        if ((FAST || r < rows) && lane == 0) publish(0, r, w_cur[j]);
    }
    cluster_arrive();

    const uint2 key = make_uint2(A.seed, A.lattice_base + (uint32_t)b);
    const uint32_t gband = (uint32_t)((row0 >> 2) + band);            // global band index: same counter as k_ising
    T uu[kIsingRB];
    if (A.u == nullptr) ising_uniforms<T>(uu, (uint32_t)x, gband, A.step0, key);

    T keep_q[kIsingRB]; int keep_s[kIsingRB];     // pending sweep: chosen Q value and its row index s (a is a_cur)
#pragma unroll
    for (int j = 0; j < kIsingRB; j++) { keep_q[j] = (T)0; keep_s[j] = 0; }

    int cur = 0;
    for (int k = 0; k <= A.K; k++, cur ^= 1) {
        cluster_wait();                                   // lattice after sweep k-1 is complete in buffer `cur`
        const uint32_t *ob = s_bits + cur * HR * wpr;
        if (tid == 0 && k >= 2) {                         // statistics of sweep k-2: all warps added before this barrier
            int *st = s_stat + (k & 1) * 2;
            atomicAdd(&A.n_up[(size_t)(k - 2) * A.B + b], st[0]);
            if (A.reward_sum) atomicAdd(&A.reward_sum[(size_t)(k - 2) * A.B + b], (T)st[1]);
            st[0] = 0; st[1] = 0;
        }
        // ---- up-neighbour counts of the current lattice ----
        int ups[kIsingRB];
        {
            const int v_top = (int)((ob[rb * wpr + w] >> lane) & 1u);                  // local row rb-1 (or halo)
            const int v_bot = (int)((ob[(rb + kIsingRB + 1) * wpr + w] >> lane) & 1u);  // local row rb+4 (or halo)
#pragma unroll
            for (int j = 0; j < kIsingRB; j++) {
                const int r = rb + j;
                int up, dn, lf, rt;
                if (FAST) {
                    up = j == 0 ? v_top : a_cur[j - 1];
                    dn = j == kIsingRB - 1 ? v_bot : a_cur[j + 1];
                    const uint32_t Wl = ob[(r + 1) * wpr + wl], Wr = ob[(r + 1) * wpr + wr];
                    lf = (int)((__funnelshift_l(Wl, w_cur[j], 1) >> lane) & 1u);
                    rt = (int)((__funnelshift_r(w_cur[j], Wr, 1) >> lane) & 1u);
                } else {
                    const bool live = r < rows && active;
                    up = live ? bit_at(ob, wpr, r, x) : 0;            // halo-indexed: local row r-1 is row r
                    dn = live ? bit_at(ob, wpr, r + 2, x) : 0;
                    lf = live ? bit_at(ob, wpr, r + 1, xl) : 0;
                    rt = live ? bit_at(ob, wpr, r + 1, xr) : 0;
                }
                ups[j] = up + dn + lf + rt;
            }
        }
        // ---- finish sweep k-1: reward on the new lattice, Q update in shared memory ----
        if (k > 0) {
            int nup = 0, rsum = 0;
#pragma unroll
            for (int j = 0; j < kIsingRB; j++) {
                const int r = rb + j;
                if (FAST || (r < rows && active)) {
                    const int a = a_cur[j];
                    const int ri = (2 * a - 1) * (ups[j] - 2);                       // Ising.py:101-111, in {-2..2}
                    const T reward = (T)0.5 * (T)(2 * a - 1) * (T)(2 * ups[j] - 4);
                    if (A.mask == nullptr || A.mask[((size_t)(k - 1) * A.B + b) * N + (size_t)(row0 + r) * L + x])
                        s_q[((size_t)keep_s[j] * strip + r * L + x) * 2 + a] = keep_q[j] + A.lr * (reward - keep_q[j]);
                    nup += a; rsum += ri;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                nup += __shfl_xor_sync(0xFFFFFFFFu, nup, o);
                rsum += __shfl_xor_sync(0xFFFFFFFFu, rsum, o);
            }
            if (lane == 0) { int *st = s_stat + ((k - 1) & 1) * 2; atomicAdd(&st[0], nup); atomicAdd(&st[1], rsum); }
        }
        if (k == A.K) break;
        // ---- draw sweep k: s = the count just computed, Boltzmann action, publish into buffer cur^1 ----
        const T tparam = temperature_param(PL ? A.temperatures[(size_t)k * A.B + b] : A.temperatures[k]);
        if (A.u != nullptr) {
#pragma unroll
            for (int j = 0; j < kIsingRB; j++) {
                const int r = rb + j;
                uu[j] = (FAST || (r < rows && active)) ? A.u[((size_t)k * A.B + b) * N + (size_t)(row0 + r) * L + x] : (T)0;
            }
        }
#pragma unroll
        for (int j = 0; j < kIsingRB; j++) {
            const int r = rb + j;
            int a = 0; T q0 = (T)0, q1 = (T)0;
            if (FAST || (r < rows && active)) {
                const typename Pair<T>::type pr =
                    *(const typename Pair<T>::type *)(s_q + ((size_t)ups[j] * strip + r * L + x) * 2);
                q0 = pr.x; q1 = pr.y;
                a = draw_action(uu[j], q0, q1, tparam);
            }
            const uint32_t word = __ballot_sync(0xFFFFFFFFu, a != 0);
            if ((FAST || r < rows) && lane == 0) publish(cur ^ 1, r, word);
            keep_q[j] = a ? q1 : q0; keep_s[j] = ups[j];
            a_cur[j] = a; w_cur[j] = word;
        }
        cluster_arrive();
        // ---- under the barrier: the next sweep's Philox draws ----
        if (A.u == nullptr && k + 1 < A.K) ising_uniforms<T>(uu, (uint32_t)x, gband, A.step0 + (uint32_t)(k + 1), key);
    }
    __syncthreads();
    if (tid == 0) {                                       // sweeps K-1 (and K-2 when it was not flushed in the loop)
        for (int kk = max(0, A.K - 1); kk < A.K; kk++) {
            int *st = s_stat + (kk & 1) * 2;
            atomicAdd(&A.n_up[(size_t)kk * A.B + b], st[0]);
            if (A.reward_sum) atomicAdd(&A.reward_sum[(size_t)kk * A.B + b], (T)st[1]);
        }
    }

    // ---- store: Q strip and the final spins ----
    for (int sp = 0; sp < 5; sp++) {
        T *dst = A.Q + (lbase * 5 + (size_t)sp * N + (size_t)row0 * L) * 2;
        const T *src = s_q + (size_t)sp * strip * 2;
        if (sizeof(T) == 4 && (strip & 1) == 0) {
            float4 *d4 = (float4 *)dst; const float4 *s4 = (const float4 *)src;
            for (int i = tid; i < strip / 2; i += blockDim.x) d4[i] = s4[i];
        } else {
            for (int i = tid; i < strip * 2; i += blockDim.x) dst[i] = src[i];
        }
    }
#pragma unroll
    for (int j = 0; j < kIsingRB; j++) {
        const int r = rb + j;
        if (FAST || (r < rows && active)) A.spins[lbase + (size_t)(row0 + r) * L + x] = (int8_t)a_cur[j];
    }
    cluster.sync();       // nobody leaves while a neighbour's last remote store may still be in flight
}

template <typename T, bool FAST>
__global__ void __launch_bounds__(1024, 1) k_ising_resident(const IsingRunArgs<T> A) { ising_resident_sweeps<T, FAST, false>(A); }
template <typename T, bool FAST>
__global__ void __launch_bounds__(1024, 1) k_ising_resident_lattices(const IsingRunArgs<T> A) {
    ising_resident_sweeps<T, FAST, true>(A);
}

// ---- K6r specialised for fp32 and compile-time shapes (the bench shape 256 x 256 / 16 rows per CTA and the other
// power-of-two sides): same algorithm, same bits as the generic kernel above, written for instruction count -- the
// kernel is issue-bound (ncu: ALU pipe busiest, no DRAM traffic).  Shapes fold to constants, shared memory is
// addressed with 32-bit shared-window addresses (ld.shared / st.shared / mapa + st.shared::cluster), the Q slot
// to update is remembered as an address, the reward is (float)((2a-1)(ups-2)) (exact), and the two per-sweep
// statistics travel through ONE packed shuffle tree and one shared atomic.  RPT = rows per thread (4 or 8).
__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
    uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v;
}
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" :: "r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ float2 lds_f32x2(uint32_t a) {
    float2 v; asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a) : "memory"); return v;
}
__device__ __forceinline__ void sts_f32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" :: "r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ uint32_t map_to_rank(uint32_t a, uint32_t rank) {
    uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank)); return r;
}
__device__ __forceinline__ void sts_cluster_u32(uint32_t a, uint32_t v) {
    asm volatile("st.shared::cluster.u32 [%0], %1;" :: "r"(a), "r"(v) : "memory");
}

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    } while (!ok);
}
// remote 4-byte store that also counts 4 bytes on the TARGET CTA's mbarrier: data and signal in one message, no fence
__device__ __forceinline__ void st_async_u32(uint32_t remote_addr, uint32_t v, uint32_t remote_bar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.u32 [%0], %1, [%2];"
                 :: "r"(remote_addr), "r"(v), "r"(remote_bar) : "memory");
}

template <int L, int ROWS, int RPT, bool MASK>
__global__ void __launch_bounds__(L * (ROWS / RPT), 1) k_ising_resident_f32(const IsingRunArgs<float> A) {
    static_assert(L % 32 == 0 && ROWS % RPT == 0 && RPT % kIsingRB == 0, "shape");
    constexpr int N = L * L, WPR = L / 32, HR = ROWS + 2, STRIP = ROWS * L, NT = L * (ROWS / RPT);
    constexpr int NPH = RPT / kIsingRB;                         // Philox calls per thread per sweep
    constexpr uint32_t PLANE = (uint32_t)STRIP * 8u;            // bytes between the Q planes of consecutive s
    constexpr uint32_t BUF = (uint32_t)HR * WPR * 4u;           // bytes per bit buffer
    extern __shared__ __align__(16) unsigned char s_raw[];
    cg::cluster_group cluster = cg::this_cluster();
    const int C = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
    const int b = blockIdx.x / C, row0 = rank * ROWS;
    float *s_q = (float *)s_raw;                                                    // [5][STRIP][2]
    uint32_t *s_bits = (uint32_t *)(s_raw + (size_t)5 * STRIP * 8);                 // [2][HR][WPR]
    unsigned long long *s_bar = (unsigned long long *)(s_bits + 2 * HR * WPR);      // [2] halo-arrival mbarrier per buffer
    int *s_stat = (int *)(s_bar + 2);                                               // [2] packed statistics per sweep parity

    const int tid = threadIdx.x, lane = tid & 31;
    const int x = tid % L, band = tid / L, w = x >> 5;
    const int rb = band * RPT;
    const int wl = w == 0 ? WPR - 1 : w - 1, wr = w == WPR - 1 ? 0 : w + 1;
    const size_t lbase = (size_t)b * N;
    const uint32_t up_rank = (uint32_t)((rank + C - 1) % C), dn_rank = (uint32_t)((rank + 1) % C);
    const uint32_t bits0 = smem_addr(s_bits);
    const uint32_t q_site0 = smem_addr(s_q) + (uint32_t)(rb * L + x) * 8u;          // Q pair of (s = 0, row rb, column x)
    const uint32_t own_w = bits0 + (uint32_t)((rb + 1) * WPR + w) * 4u;             // this thread's word of local row rb, buffer 0
    const uint32_t own_l = bits0 + (uint32_t)((rb + 1) * WPR + wl) * 4u, own_r = bits0 + (uint32_t)((rb + 1) * WPR + wr) * 4u;
    // remote halo slots (buffer 0): up neighbour's bottom halo row, down neighbour's top halo row
    const uint32_t halo_up = map_to_rank(bits0 + (uint32_t)((ROWS + 1) * WPR + w) * 4u, up_rank);
    const uint32_t halo_dn = map_to_rank(bits0 + (uint32_t)w * 4u, dn_rank);
    const uint32_t bar0 = smem_addr(s_bar);                                          // + 8 * buffer
    const uint32_t bar_up = map_to_rank(bar0, up_rank), bar_dn = map_to_rank(bar0, dn_rank);
    const bool first_band = rb == 0, last_band = rb + RPT == ROWS;
    constexpr uint32_t HALO_BYTES = 2u * WPR * 4u;                                   // one row from above, one from below

    if (tid < 2) s_stat[tid] = 0;
    if (tid == 0) {
        mbar_init(bar0, 1); mbar_init(bar0 + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_expect_tx(bar0, HALO_BYTES);                                            // the initial lattice arrives in buffer 0
    }
    for (int sp = 0; sp < 5; sp++) {
        const float4 *s4 = (const float4 *)(A.Q + (lbase * 5 + (size_t)sp * N + (size_t)row0 * L) * 2);
        float4 *d4 = (float4 *)(s_q + (size_t)sp * STRIP * 2);
#pragma unroll 4
        for (int i = tid; i < STRIP / 2; i += NT) d4[i] = s4[i];
    }
    int a_cur[RPT]; uint32_t w_cur[RPT];
    cluster.sync();                 // everybody's shared memory exists before the first remote store
#pragma unroll
    for (int j = 0; j < RPT; j++) {
        a_cur[j] = (int)A.spins[lbase + (size_t)(row0 + rb + j) * L + x];
        w_cur[j] = __ballot_sync(0xFFFFFFFFu, a_cur[j] != 0);
        if (lane == 0) {
            sts_u32(own_w + (uint32_t)j * WPR * 4u, w_cur[j]);
            if (first_band && j == 0) st_async_u32(halo_up, w_cur[j], bar_up);
            if (last_band && j == RPT - 1) st_async_u32(halo_dn, w_cur[j], bar_dn);
        }
    }

    const uint2 key = make_uint2(A.seed, A.lattice_base + (uint32_t)b);
    const uint32_t gband = (uint32_t)((row0 + rb) >> 2);
    float uu[RPT];
    auto draw_uniforms = [&](uint32_t step) {
#pragma unroll
        for (int h = 0; h < NPH; h++) {
            const uint4 rnd = philox4x32_10(make_uint4((uint32_t)x, gband + (uint32_t)h, step, 0u), key);
            uu[4 * h + 0] = __uint2float_rz(rnd.x); uu[4 * h + 1] = __uint2float_rz(rnd.y);   // u * 2^32
            uu[4 * h + 2] = __uint2float_rz(rnd.z); uu[4 * h + 3] = __uint2float_rz(rnd.w);
        }
    };
    if (A.u == nullptr) draw_uniforms(A.step0);
    float tparam = temperature_param(A.temperatures[0]);

    float keep_q[RPT]; uint32_t keep_addr[RPT];       // pending sweep: chosen Q value and the shared address it came from
#pragma unroll
    for (int j = 0; j < RPT; j++) { keep_q[j] = 0.0f; keep_addr[j] = q_site0; }

    // Synchronisation per sweep: ONE __syncthreads (the CTA's own words) plus, for the two boundary bands only, a wait
    // on the mbarrier that counts the halo bytes the neighbours pushed with st.async -- point to point, no cluster-wide
    // barrier and no fence.  A neighbour cannot overwrite a halo row still being read: it only reaches the draw
    // that writes buffer X again after receiving this CTA's next words, which are sent after these reads.
    uint32_t cur = 0;                                 // byte offset of the buffer holding the current lattice (0 or BUF)
    for (int k = 0; k <= A.K; k++, cur ^= BUF) {
        __syncthreads();                              // own words of the lattice after sweep k-1 are in buffer `cur`
        const uint32_t cur_bar = bar0 + (cur ? 8u : 0u);
        if (tid == 0) mbar_expect_tx(bar0 + (cur ? 0u : 8u), HALO_BYTES);   // the other buffer fills during this iteration
        if (first_band || last_band) mbar_wait(cur_bar, (uint32_t)(k >> 1) & 1u);
        if (tid == 0 && k >= 2) {                     // statistics of sweep k-2: all warps added before this barrier
            const int pk = s_stat[k & 1];
            s_stat[k & 1] = 0;
            atomicAdd(&A.n_up[(size_t)(k - 2) * A.B + b], pk & 0xFFFF);
            if (A.reward_sum) atomicAdd(&A.reward_sum[(size_t)(k - 2) * A.B + b], (float)((pk >> 16) - 2 * RPT * NT));
        }
        // ---- up-neighbour counts of the current lattice ----
        int ups[RPT];
        {
            const int v_top = (int)((lds_u32(own_w + cur - WPR * 4u) >> lane) & 1u);
            const int v_bot = (int)((lds_u32(own_w + cur + (uint32_t)RPT * WPR * 4u) >> lane) & 1u);
#pragma unroll
            for (int j = 0; j < RPT; j++) {
                const int up = j == 0 ? v_top : a_cur[j - 1];
                const int dn = j == RPT - 1 ? v_bot : a_cur[j + 1];
                const uint32_t Wl = lds_u32(own_l + cur + (uint32_t)j * WPR * 4u), Wr = lds_u32(own_r + cur + (uint32_t)j * WPR * 4u);
                const uint32_t lf = __funnelshift_l(Wl, w_cur[j], 1), rt = __funnelshift_r(w_cur[j], Wr, 1);
                ups[j] = up + dn + (int)((lf >> lane) & 1u) + (int)((rt >> lane) & 1u);
            }
        }
        // ---- finish sweep k-1: reward on the new lattice, Q update in shared memory, statistics ----
        if (k > 0) {
            int packed = 0;
            uint32_t upd = 0xFFFFFFFFu;                                            // bit j: site j updates Q this sweep
            if (MASK) {                                                            // act_rate < 1
                const uint8_t *m = A.mask + ((size_t)(k - 1) * A.B + b) * N + (size_t)(row0 + rb) * L + x;
                upd = 0;
#pragma unroll
                for (int j = 0; j < RPT; j++) upd |= (m[j * L] ? 1u : 0u) << j;
            }
#pragma unroll
            for (int j = 0; j < RPT; j++) {
                const int d = ups[j] - 2;
                const int ri = a_cur[j] ? d : -d;                                  // (2a-1)(ups-2) = Ising.py:101-111
                const float reward = (float)ri;                                    // == 0.5f * (2a-1) * (2 ups - 4), exactly
                if (!MASK || ((upd >> j) & 1u)) sts_f32(keep_addr[j], keep_q[j] + A.lr * (reward - keep_q[j]));
                packed += a_cur[j] + ((ri + 2) << 16);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) packed += __shfl_xor_sync(0xFFFFFFFFu, packed, o);
            if (lane == 0) atomicAdd(&s_stat[(k - 1) & 1], packed);
        }
        if (k == A.K) break;
        // ---- draw sweep k: s = the count just computed, Boltzmann action, publish into the other buffer ----
        if (A.u != nullptr) {
#pragma unroll
            for (int j = 0; j < RPT; j++)
                uu[j] = A.u[((size_t)k * A.B + b) * N + (size_t)(row0 + rb + j) * L + x] * 4294967296.0f;
        }
        const uint32_t nxt = cur ^ BUF;
        // staged so that the RPT sites' load -> exp -> compare -> ballot chains overlap instead of running one after
        // the other (the shared-memory stores of one site would otherwise order the next site's load behind them)
        float2 pr[RPT];
#pragma unroll
        for (int j = 0; j < RPT; j++) {
            keep_addr[j] = q_site0 + (uint32_t)ups[j] * PLANE + (uint32_t)j * (L * 8u);
            pr[j] = lds_f32x2(keep_addr[j]);
        }
#pragma unroll
        for (int j = 0; j < RPT; j++) a_cur[j] = draw_action_scaled(uu[j], pr[j].x, pr[j].y, tparam);
#pragma unroll
        for (int j = 0; j < RPT; j++) w_cur[j] = __ballot_sync(0xFFFFFFFFu, a_cur[j] != 0);
        if (lane == 0) {
#pragma unroll
            for (int j = 0; j < RPT; j++) sts_u32(own_w + nxt + (uint32_t)j * WPR * 4u, w_cur[j]);
            if (first_band) st_async_u32(halo_up + nxt, w_cur[0], bar_up + (nxt ? 8u : 0u));
            if (last_band) st_async_u32(halo_dn + nxt, w_cur[RPT - 1], bar_dn + (nxt ? 8u : 0u));
        }
#pragma unroll
        for (int j = 0; j < RPT; j++) {
            keep_q[j] = a_cur[j] ? pr[j].y : pr[j].x;
            keep_addr[j] += (uint32_t)a_cur[j] * 4u;
        }
        // ---- the next sweep's Philox draws and temperature (independent of the lattice) ----
        if (k + 1 < A.K) {
            if (A.u == nullptr) draw_uniforms(A.step0 + (uint32_t)(k + 1));
            tparam = temperature_param(A.temperatures[k + 1]);
        }
    }
    __syncthreads();
    if (tid == 0) {
        const int kk = A.K - 1, pk = s_stat[kk & 1];
        atomicAdd(&A.n_up[(size_t)kk * A.B + b], pk & 0xFFFF);
        if (A.reward_sum) atomicAdd(&A.reward_sum[(size_t)kk * A.B + b], (float)((pk >> 16) - 2 * RPT * NT));
    }
    for (int sp = 0; sp < 5; sp++) {
        float4 *d4 = (float4 *)(A.Q + (lbase * 5 + (size_t)sp * N + (size_t)row0 * L) * 2);
        const float4 *s4 = (const float4 *)(s_q + (size_t)sp * STRIP * 2);
#pragma unroll 4
        for (int i = tid; i < STRIP / 2; i += NT) d4[i] = s4[i];
    }
#pragma unroll
    for (int j = 0; j < RPT; j++) A.spins[lbase + (size_t)(row0 + rb + j) * L + x] = (int8_t)a_cur[j];
    cluster.sync();       // nobody leaves while a neighbour's last remote store may still be in flight
}

// ---- K6p: the same sweep as K6r-f32, PERSISTENT and without thread-block clusters --------------------------------
// A 16-CTA cluster has to sit inside one GPC, and the B200's GPCs (16-20 SMs) hold one such cluster each: only 7 of
// them are resident, 112 of 148 SMs (ncu launch__waves_per_multiprocessor, round 1).  Here a lattice is still cut into
// C = L / ROWS strips, one CTA each, but the CTAs are ordinary ones: the grid is exactly n_slots * C <= (resident CTAs)
// co-scheduled CTAs (cooperative launch, so they are guaranteed to be resident together), slot s sweeps lattices
// s, s + n_slots, ... one after the other, and the halo words travel through L2.  One 8-byte store carries a halo
// word and a sequence number -- data and flag in one single-copy-atomic message, so neither side needs a fence -- and
// the receiving warp polls exactly the word it needs with ld.relaxed.gpu (all lanes the same address: one request).
// Sequence numbers count lattice states over the whole launch (state k of the it-th lattice of a slot has number
// it * (K + 1) + k + 1); the parity of that number picks the buffer, in shared memory as in L2, so the last state of
// one lattice and the first of the next never share a buffer.  A strip can be at most one state ahead of its
// neighbours (it needs their halo of state k to publish state k + 1), which is what makes two buffers enough.
// Same Philox keys, same arithmetic, same bits as K6 / K6r.
__device__ __forceinline__ void st_halo(unsigned long long *p, uint32_t word, uint32_t seq) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" :: "l"(p), "l"(((unsigned long long)seq << 32) | word) : "memory");
}
__device__ __forceinline__ unsigned long long ld_halo(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

template <int L, int ROWS, int RPT, bool MASK>
__global__ void __launch_bounds__(L * (ROWS / RPT), 1) k_ising_persist_f32(const IsingRunArgs<float> A, const int n_slots,
                                                                           unsigned long long *const halo) {
    static_assert(L % 32 == 0 && ROWS % RPT == 0 && RPT % kIsingRB == 0 && L % ROWS == 0 && ROWS > RPT, "shape");
    constexpr int N = L * L, WPR = L / 32, HR = ROWS + 2, STRIP = ROWS * L, NT = L * (ROWS / RPT), C = L / ROWS;
    constexpr int NPH = RPT / kIsingRB;                         // Philox calls per thread per sweep
    constexpr uint32_t PLANE = (uint32_t)STRIP * 8u;            // bytes between the Q planes of consecutive s
    constexpr uint32_t BUF = (uint32_t)HR * WPR * 4u;           // bytes per bit buffer
    extern __shared__ __align__(16) unsigned char s_raw[];
    const int slot = blockIdx.x / C, rank = blockIdx.x % C, row0 = rank * ROWS;
    float *s_q = (float *)s_raw;                                                    // [5][STRIP][2]
    uint32_t *s_bits = (uint32_t *)(s_raw + (size_t)5 * STRIP * 8);                 // [2][HR][WPR]
    int *s_stat = (int *)(s_bits + 2 * HR * WPR);                                   // [2] packed statistics per sweep parity
    float *s_tparam = (float *)(s_stat + 4);                                        // [K] log2(e) / T_k, computed once per launch

    const int tid = threadIdx.x, lane = tid & 31;
    const int x = tid % L, band = tid / L, w = x >> 5;
    const int rb = band * RPT;
    const int wl = w == 0 ? WPR - 1 : w - 1, wr = w == WPR - 1 ? 0 : w + 1;
    const int up_rank = (rank + C - 1) % C, dn_rank = (rank + 1) % C;
    const uint32_t bits0 = smem_addr(s_bits);
    const uint32_t q_site0 = smem_addr(s_q) + (uint32_t)(rb * L + x) * 8u;          // Q pair of (s = 0, row rb, column x)
    const uint32_t own_w = bits0 + (uint32_t)((rb + 1) * WPR + w) * 4u;             // this thread's word of local row rb, buffer 0
    const uint32_t own_l = bits0 + (uint32_t)((rb + 1) * WPR + wl) * 4u, own_r = bits0 + (uint32_t)((rb + 1) * WPR + wr) * 4u;
    const bool first_band = rb == 0, last_band = rb + RPT == ROWS;                  // (never both: ROWS > RPT)
    // halo mailboxes in L2: [slot][rank][parity][top | bottom][WPR] -- rank r READS its own, its neighbours write into it.
    // A boundary warp reads one word (its 32 columns of the row above / below the strip) and writes one word.
    constexpr size_t MB_PARITY = 2 * WPR;                                            // mailbox words between the two parities
    const unsigned long long *const mb_in =
        halo + (((size_t)slot * C + rank) * 2 * 2 + (last_band ? 1 : 0)) * WPR + w;
    unsigned long long *const mb_out =
        halo + (((size_t)slot * C + (first_band ? up_rank : dn_rank)) * 2 * 2 + (first_band ? 1 : 0)) * WPR + w;
    const bool boundary = first_band || last_band;

    for (int i = threadIdx.x; i < A.K; i += NT) s_tparam[i] = temperature_param(A.temperatures[i]);
    uint32_t state_no = 0;                                      // lattice states published so far by this slot
    for (int b = slot; b < A.B; b += n_slots, state_no += (uint32_t)A.K + 1u) {
        const size_t lbase = (size_t)b * N;
        __syncthreads();                                        // the previous lattice's Q strip has been stored
        if (tid < 2) s_stat[tid] = 0;
        for (int sp = 0; sp < 5; sp++) {
            const float4 *s4 = (const float4 *)(A.Q + (lbase * 5 + (size_t)sp * N + (size_t)row0 * L) * 2);
            float4 *d4 = (float4 *)(s_q + (size_t)sp * STRIP * 2);
#pragma unroll 4
            for (int i = tid; i < STRIP / 2; i += NT) d4[i] = s4[i];
        }
        int a_cur[RPT]; uint32_t w_cur[RPT];
        unsigned long long hv = 0;                              // the halo word last read from the mailbox (word | seq << 32)
        {
            const uint32_t par = state_no & 1u, seq = state_no + 1u;
#pragma unroll
            for (int j = 0; j < RPT; j++) {
                a_cur[j] = (int)A.spins[lbase + (size_t)(row0 + rb + j) * L + x];
                w_cur[j] = __ballot_sync(0xFFFFFFFFu, a_cur[j] != 0);
                if (lane == 0) sts_u32(own_w + par * BUF + (uint32_t)j * WPR * 4u, w_cur[j]);
            }
            if (boundary) {
                if (lane == 0) st_halo(mb_out + par * MB_PARITY, first_band ? w_cur[0] : w_cur[RPT - 1], seq);
                hv = ld_halo(mb_in + par * MB_PARITY);
            }
        }
        const uint2 key = make_uint2(A.seed, A.lattice_base + (uint32_t)b);
        const uint32_t gband = (uint32_t)((row0 + rb) >> 2);
        float uu[RPT];
        auto draw_uniforms = [&](uint32_t step) {
#pragma unroll
            for (int h = 0; h < NPH; h++) {
                const uint4 rnd = philox4x32_10(make_uint4((uint32_t)x, gband + (uint32_t)h, step, 0u), key);
                uu[4 * h + 0] = __uint2float_rz(rnd.x); uu[4 * h + 1] = __uint2float_rz(rnd.y);   // u * 2^32
                uu[4 * h + 2] = __uint2float_rz(rnd.z); uu[4 * h + 3] = __uint2float_rz(rnd.w);
            }
        };
        if (A.u == nullptr) draw_uniforms(A.step0);
        float keep_q[RPT]; uint32_t keep_addr[RPT];
#pragma unroll
        for (int j = 0; j < RPT; j++) { keep_q[j] = 0.0f; keep_addr[j] = q_site0; }

        // Order inside a sweep.  Only the strip's BOUNDARY row needs the neighbour (its halo word), and only the
        // boundary row is needed by the neighbour.  It is therefore handled LAST: the interior rows of sweep k are
        // finished and drawn first, while the halo word of state k -- sent by the neighbour at the end of ITS interior
        // work of the previous sweep -- travels through L2; it is asked for half-way through the interior work and looked
        // at only when the boundary row's turn comes, and the boundary row's new word leaves right after.  Between a
        // send and the moment the neighbour needs the word lies most of a sweep, which is what absorbs the L2 round
        // trip and the jitter between the 16 strips of a lattice (ncu, boundary row first: 11 % of the samples sat in
        // the halo poll and 14 % at the barrier behind it).
        auto is_boundary_row = [&](int j) { return (j == 0 && first_band) || (j == RPT - 1 && last_band); };
        for (int k = 0; k <= A.K; k++) {
            const uint32_t par = (state_no + (uint32_t)k) & 1u, seq = state_no + (uint32_t)k + 1u;
            const uint32_t cur = par * BUF, nxt = cur ^ BUF;
            __syncthreads();                              // own words of the lattice after sweep k-1 are in buffer `cur`
            if (tid == 0 && k >= 2) {                     // statistics of sweep k-2: all warps added before this barrier
                const int pk = s_stat[k & 1];
                s_stat[k & 1] = 0;
                atomicAdd(&A.n_up[(size_t)(k - 2) * A.B + b], pk & 0xFFFF);
                if (A.reward_sum) atomicAdd(&A.reward_sum[(size_t)(k - 2) * A.B + b], (float)((pk >> 16) - 2 * RPT * NT));
            }
            const bool draw = k < A.K;
            const float tparam = s_tparam[draw ? k : 0];      // (written before the first barrier of the first lattice)
            if (draw && A.u != nullptr) {
#pragma unroll
                for (int j = 0; j < RPT; j++)
                    uu[j] = A.u[((size_t)k * A.B + b) * N + (size_t)(row0 + rb + j) * L + x] * 4294967296.0f;
            }
            uint32_t upd = 0xFFFFFFFFu;                                            // bit j: site j updates Q (sweep k-1)
            if (MASK && k > 0) {
                const uint8_t *m = A.mask + ((size_t)(k - 1) * A.B + b) * N + (size_t)(row0 + rb) * L + x;
                upd = 0;
#pragma unroll
                for (int j = 0; j < RPT; j++) upd |= (m[j * L] ? 1u : 0u) << j;
            }
            // the state-k spins the boundary row's count will need, before the interior rows are redrawn
            const int a_next_to_boundary = first_band ? a_cur[1] : a_cur[RPT - 2];
            int packed = 0;
            int ups[RPT];
            float2 pr[RPT];
            // ---- interior rows: neighbour counts of state k (own registers + own shared-memory words) ----
            {
                const uint32_t top_word = first_band ? 0u : lds_u32(own_w + cur - WPR * 4u);
                const uint32_t bot_word = last_band ? 0u : lds_u32(own_w + cur + (uint32_t)RPT * WPR * 4u);
                const int v_top = (int)((top_word >> lane) & 1u), v_bot = (int)((bot_word >> lane) & 1u);
#pragma unroll
                for (int j = 0; j < RPT; j++) {
                    if (is_boundary_row(j)) continue;
                    const int up = j == 0 ? v_top : a_cur[j - 1];
                    const int dn = j == RPT - 1 ? v_bot : a_cur[j + 1];
                    const uint32_t Wl = lds_u32(own_l + cur + (uint32_t)j * WPR * 4u), Wr = lds_u32(own_r + cur + (uint32_t)j * WPR * 4u);
                    const uint32_t lf = __funnelshift_l(Wl, w_cur[j], 1), rt = __funnelshift_r(w_cur[j], Wr, 1);
                    ups[j] = up + dn + (int)((lf >> lane) & 1u) + (int)((rt >> lane) & 1u);
                }
            }
            // ---- interior rows: finish sweep k-1 (reward on state k, Q update in shared memory, statistics) ----
            if (k > 0) {
#pragma unroll
                for (int j = 0; j < RPT; j++) {
                    if (is_boundary_row(j)) continue;
                    const int d = ups[j] - 2;
                    const int ri = a_cur[j] ? d : -d;                                  // (2a-1)(ups-2) = Ising.py:101-111
                    if (!MASK || ((upd >> j) & 1u)) sts_f32(keep_addr[j], keep_q[j] + A.lr * ((float)ri - keep_q[j]));
                    packed += a_cur[j] + ((ri + 2) << 16);
                }
            }
            // the halo word of state k: asked for now, looked at after the interior draws
            if (boundary && (uint32_t)(hv >> 32) != seq) hv = ld_halo(mb_in + par * MB_PARITY);
            // ---- interior rows: draw sweep k (staged: all Q-pair loads, all decisions, all ballots) ----
            if (draw) {
#pragma unroll
                for (int j = 0; j < RPT; j++) {
                    if (is_boundary_row(j)) continue;
                    keep_addr[j] = q_site0 + (uint32_t)ups[j] * PLANE + (uint32_t)j * (L * 8u);
                    pr[j] = lds_f32x2(keep_addr[j]);
                }
#pragma unroll
                for (int j = 0; j < RPT; j++)
                    if (!is_boundary_row(j)) a_cur[j] = draw_action_scaled(uu[j], pr[j].x, pr[j].y, tparam);
#pragma unroll
                for (int j = 0; j < RPT; j++)
                    if (!is_boundary_row(j)) w_cur[j] = __ballot_sync(0xFFFFFFFFu, a_cur[j] != 0);
                if (lane == 0) {
#pragma unroll
                    for (int j = 0; j < RPT; j++)
                        if (!is_boundary_row(j)) sts_u32(own_w + nxt + (uint32_t)j * WPR * 4u, w_cur[j]);
                }
#pragma unroll
                for (int j = 0; j < RPT; j++) {
                    if (is_boundary_row(j)) continue;
                    keep_q[j] = a_cur[j] ? pr[j].y : pr[j].x;
                    keep_addr[j] += (uint32_t)a_cur[j] * 4u;
                }
            }
            // ---- the boundary row: halo word of state k, count, finish, draw, and its new word straight to the neighbour ----
            if (boundary) {
                while ((uint32_t)(hv >> 32) != seq) hv = ld_halo(mb_in + par * MB_PARITY);
                const int v_halo = (int)(((uint32_t)hv >> lane) & 1u);
                auto boundary_row = [&](auto jc) {
                    constexpr int j = decltype(jc)::value;
                    const int up = j == 0 ? v_halo : a_next_to_boundary, dn = j == 0 ? a_next_to_boundary : v_halo;
                    const uint32_t Wl = lds_u32(own_l + cur + (uint32_t)j * WPR * 4u), Wr = lds_u32(own_r + cur + (uint32_t)j * WPR * 4u);
                    const uint32_t lf = __funnelshift_l(Wl, w_cur[j], 1), rt = __funnelshift_r(w_cur[j], Wr, 1);
                    const int u = up + dn + (int)((lf >> lane) & 1u) + (int)((rt >> lane) & 1u);
                    if (k > 0) {
                        const int d = u - 2;
                        const int ri = a_cur[j] ? d : -d;
                        if (!MASK || ((upd >> j) & 1u)) sts_f32(keep_addr[j], keep_q[j] + A.lr * ((float)ri - keep_q[j]));
                        packed += a_cur[j] + ((ri + 2) << 16);
                    }
                    if (draw) {
                        keep_addr[j] = q_site0 + (uint32_t)u * PLANE + (uint32_t)j * (L * 8u);
                        const float2 q = lds_f32x2(keep_addr[j]);
                        a_cur[j] = draw_action_scaled(uu[j], q.x, q.y, tparam);
                        w_cur[j] = __ballot_sync(0xFFFFFFFFu, a_cur[j] != 0);
                        if (lane == 0) {
                            st_halo(mb_out + (par ^ 1u) * MB_PARITY, w_cur[j], seq + 1u);
                            sts_u32(own_w + nxt + (uint32_t)j * WPR * 4u, w_cur[j]);
                        }
                        keep_q[j] = a_cur[j] ? q.y : q.x;
                        keep_addr[j] += (uint32_t)a_cur[j] * 4u;
                    }
                };
                if (first_band) boundary_row(std::integral_constant<int, 0>{});
                else boundary_row(std::integral_constant<int, RPT - 1>{});
            }
            if (k > 0) {
                packed = __reduce_add_sync(0xFFFFFFFFu, packed);           // one REDUX instead of a five-step shuffle tree
                if (lane == 0) atomicAdd(&s_stat[(k - 1) & 1], packed);
            }
            if (!draw) break;
            // ---- the next sweep's Philox draws and temperature (independent of the lattice) ----
            if (k + 1 < A.K && A.u == nullptr) draw_uniforms(A.step0 + (uint32_t)(k + 1));
        }
        __syncthreads();
        if (tid == 0) {
            const int kk = A.K - 1, pk = s_stat[kk & 1];
            atomicAdd(&A.n_up[(size_t)kk * A.B + b], pk & 0xFFFF);
            if (A.reward_sum) atomicAdd(&A.reward_sum[(size_t)kk * A.B + b], (float)((pk >> 16) - 2 * RPT * NT));
        }
        for (int sp = 0; sp < 5; sp++) {
            float4 *d4 = (float4 *)(A.Q + (lbase * 5 + (size_t)sp * N + (size_t)row0 * L) * 2);
            const float4 *s4 = (const float4 *)(s_q + (size_t)sp * STRIP * 2);
#pragma unroll 4
            for (int i = tid; i < STRIP / 2; i += NT) d4[i] = s4[i];
        }
#pragma unroll
        for (int j = 0; j < RPT; j++) A.spins[lbase + (size_t)(row0 + rb + j) * L + x] = (int8_t)a_cur[j];
    }
}

// ---- K6s: K6p with the per-site integer work done for a thread's RPT rows AT ONCE (SWAR) -------------------------
// ncu on K6p v5: 69 thread instructions per site-step, 9 % of them branches, 8 ballots + 16 word loads + 16 funnel
// shifts per thread per sweep only to count neighbours.  Here a thread keeps its RPT <= 8 spins as ONE word of 4-bit
// fields (field i = slot i), so
//   * the left / right neighbours of all its rows arrive with two warp shuffles (lanes 0 and 31 take the word the
//     neighbouring warp's edge lane left in shared memory),
//   * up / down are the word shifted by one field,
//   * the neighbour counts of all rows are three SWAR additions (a field never exceeds 4),
//   * the per-sweep statistics are a popcount and two horizontal field sums,
//   * the reward as a float is (2^23 + count) reinterpreted, minus (2^23 + 2): no integer-to-float conversion,
//   * only the two rows other threads' columns look at from above / below are still published as ballot words.
// Shape: exactly two bands per strip (ROWS == 2 RPT; RPT = 8 at sides 64 / 128 / 256, 4 at 512 where 16 rows do not fit).  The lower band holds its rows in REVERSE order (slot i = local
// row ROWS-1-i, in registers and in the shared-memory Q strip), which makes the two bands mirror images: slot 0 is
// always the strip's boundary row (the one that needs the halo word and feeds the neighbouring strip), slot RPT-1
// always the row facing the other band, and the neighbour sum is symmetric in up / down -- one code path, no
// per-row "is this the boundary row" branches.  The sweep loop is peeled (first sweep: nothing to finish; after the
// last: nothing to draw) and has NO CTA barrier: the three words a warp reads from other warps are 8-byte
// {word, sequence number} messages in shared memory (see `sweep` below), the per-warp statistics stay in registers and
// meet every 32 sweeps.  Same Philox keys, same float operations in the same order as K6 / K6r / K6p: same bits.
// Measured (C5, B200): K6p 3.27e11 -> 4.59e11 site-steps/s; 69 -> 50 thread instructions per site-step (profiles/r02).
template <int I0, int I1, class F> __device__ __forceinline__ void static_for(F &&f) {
    if constexpr (I0 < I1) { f(std::integral_constant<int, I0>{}); static_for<I0 + 1, I1>(f); }
}
template <uint32_t OFF> __device__ __forceinline__ float2 lds_f32x2_at(uint32_t a) {
    float2 v; asm volatile("ld.shared.v2.f32 {%0, %1}, [%2+%3];" : "=f"(v.x), "=f"(v.y) : "r"(a), "n"(OFF) : "memory"); return v;
}
template <uint32_t OFF> __device__ __forceinline__ void sts_f32_at(uint32_t a, float v) {
    asm volatile("st.shared.f32 [%0+%1], %2;" :: "r"(a), "n"(OFF), "f"(v) : "memory");
}
// 8-byte shared-memory messages {word, sequence number}: data and flag in one single-copy-atomic access
__device__ __forceinline__ void sts_msg(uint32_t a, uint32_t word, uint32_t seq) {
    asm volatile("st.relaxed.cta.shared.u64 [%0], %1;" :: "r"(a), "l"(((unsigned long long)seq << 32) | word) : "memory");
}
__device__ __forceinline__ unsigned long long lds_msg(uint32_t a) {
    unsigned long long v; asm volatile("ld.relaxed.cta.shared.u64 %0, [%1];" : "=l"(v) : "r"(a) : "memory"); return v;
}
__device__ __forceinline__ uint32_t field_sum(uint32_t x) {            // sum of the eight 4-bit fields (each <= 15)
    return (((x & 0x0F0F0F0Fu) + ((x >> 4) & 0x0F0F0F0Fu)) * 0x01010101u) >> 24;
}

// PL: A.temperatures is [K][B]; the log2e / T table is refilled from lattice b's column (prefetched during the previous lattice) when a slot takes lattice b up
template <int L, int RPT, bool MASK, bool PL>
__global__ void __launch_bounds__(2 * L, 512 / (2 * L) > 0 ? 512 / (2 * L) : 1) k_ising_persist_swar_f32(const IsingRunArgs<float> A, const int n_slots,
                                                                     unsigned long long *const halo) {
    static_assert(L % 32 == 0 && RPT % kIsingRB == 0 && RPT <= 8 && L % (2 * RPT) == 0, "shape");
    static_assert(((uint64_t)0x4B000000u * ((uint64_t)2 * RPT * L * 8)) % (1ull << 32) == 0, "plane stride must clear the float exponent bits");
    constexpr int ROWS = 2 * RPT, N = L * L, WPR = L / 32, STRIP = ROWS * L, NT = 2 * L, C = L / ROWS, NW = NT / 32;
    constexpr int NPH = RPT / kIsingRB;
    constexpr uint32_t PLANE = (uint32_t)STRIP * 8u;            // bytes between the Q planes of consecutive s
    constexpr uint32_t ROWB = (uint32_t)L * 8u;                 // bytes between consecutive rows of a plane
    constexpr uint32_t TOP = 4u * (RPT - 1);                    // bit position of the last slot's field
    constexpr uint32_t FIELDS = RPT == 8 ? 0xFFFFFFFFu : ((1u << (4 * RPT)) - 1u);
    extern __shared__ __align__(16) unsigned char s_raw[];
    const int slot = blockIdx.x / C, rank = blockIdx.x % C, row0 = rank * ROWS;
    float *s_q = (float *)s_raw;                                                    // [5][ROWS (lower band reversed)][L][2]
    unsigned long long *s_inner = (unsigned long long *)(s_raw + (size_t)5 * STRIP * 8);   // [2 parity][2 band][WPR] {ballot of slot RPT-1, seq}
    unsigned long long *s_edge = s_inner + 2 * 2 * WPR;                             // [2 parity][2 band][WPR][2] {field word of lane 0 / 31, seq}
    int *s_wstat = (int *)(s_edge + 2 * 2 * WPR * 2);                               // [NW][32] packed statistics of up to 32 sweeps per warp
    float *s_tparam = (float *)(s_wstat + NW * 32);                                 // [K]
    float *s_traw = s_tparam + A.K;                     // PL: [K] the raw temperatures of the slot's next lattice
    constexpr uint32_t INNER_BUF = 2u * WPR * 8u, EDGE_BUF = 2u * WPR * 2u * 8u;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int x = tid % L, band = tid / L, w = x >> 5;
    const bool upper = band == 0;
    const int wl = w == 0 ? WPR - 1 : w - 1, wr = w == WPR - 1 ? 0 : w + 1;
    const int up_rank = (rank + C - 1) % C, dn_rank = (rank + 1) % C;
    const uint32_t q_site0 = smem_addr(s_q) + (uint32_t)(band * RPT * L + x) * 8u;  // Q pair of (s = 0, slot 0, column x)
    const uint32_t inner_out = smem_addr(s_inner) + (uint32_t)(band * WPR + w) * 8u;
    const uint32_t inner_in = smem_addr(s_inner) + (uint32_t)((band ^ 1) * WPR + w) * 8u;
    const uint32_t edge_out = smem_addr(s_edge) + (uint32_t)(((band * WPR + w) * 2 + (lane == 31 ? 1 : 0))) * 8u;
    const uint32_t edge_in = smem_addr(s_edge) +
        (uint32_t)(lane == 0 ? (band * WPR + wl) * 2 + 1 : lane == 31 ? (band * WPR + wr) * 2 : (band * WPR + w) * 2) * 8u;
    const bool edge_lane = lane == 0 || lane == 31;
    // halo mailboxes in L2 as in K6p: [slot][rank][parity][top | bottom][WPR]
    constexpr size_t MB_PARITY = 2 * WPR;
    const unsigned long long *const mb_in = halo + (((size_t)slot * C + rank) * 2 * 2 + (upper ? 0 : 1)) * WPR + w;
    unsigned long long *const mb_out = halo + (((size_t)slot * C + (upper ? up_rank : dn_rank)) * 2 * 2 + (upper ? 1 : 0)) * WPR + w;

    if (!PL) for (int i = tid; i < A.K; i += NT) s_tparam[i] = temperature_param(A.temperatures[i]);
    // PL: lattice bb's column of the [K][B] table, copied into s_traw with cp.async while the slot still sweeps the
    // lattice before it (a strided gather of K words: its latency would otherwise stall every hand-over).  Thread tid
    // copies, and later converts, exactly the entries i = tid + j NT, so it only waits for its own copies.
    auto prefetch_column = [&](int bb) {
        for (int i = tid; i < A.K; i += NT)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;"
                         :: "r"(smem_addr(s_traw + i)), "l"(A.temperatures + (size_t)i * A.B + bb) : "memory");
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    if (PL && slot < A.B) prefetch_column(slot);
    for (int i = tid; i < 2 * 2 * WPR * 3; i += NT) s_inner[i] = 0ull;              // (s_inner and s_edge are contiguous) sequence numbers start at 1

    // everything a lattice needs, for the upper band (slot i = row i of the strip) or the lower one (slot i = row ROWS-1-i)
    auto run_lattice = [&](auto upper_c, const int b, const uint32_t state_no) {
        constexpr bool UPPER = decltype(upper_c)::value;
        auto local_row = [](int i) { return UPPER ? i : ROWS - 1 - i; };
        const size_t lbase = (size_t)b * N;
        uint32_t own = 0;                                       // this thread's spins of the current state, 4 bits per slot
        float sgn[RPT];                                         // the same spins as sigma = +-1
        unsigned long long hv = 0;
        {
            const uint32_t par = state_no & 1u, seq = state_no + 1u;
            int a0 = 0, aN = 0;
#pragma unroll
            for (int i = 0; i < RPT; i++) {
                const int a = (int)A.spins[lbase + (size_t)(row0 + local_row(i)) * L + x] != 0;
                own |= (uint32_t)a << (4 * i);
                sgn[i] = a ? 1.0f : -1.0f;
                if (i == 0) a0 = a;
                if (i == RPT - 1) aN = a;
            }
            const uint32_t w0 = __ballot_sync(0xFFFFFFFFu, a0 != 0), wN = __ballot_sync(0xFFFFFFFFu, aN != 0);
            if (lane == 0) {
                sts_msg(inner_out + par * INNER_BUF, wN, seq);
                st_halo(mb_out + par * MB_PARITY, w0, seq);
            }
            if (edge_lane) sts_msg(edge_out + par * EDGE_BUF, own, seq);
            hv = ld_halo(mb_in + par * MB_PARITY);
        }
        const uint2 key = make_uint2(A.seed, A.lattice_base + (uint32_t)b);
        const uint32_t gband = (uint32_t)((row0 + band * RPT) >> 2);
        float uu[RPT];                                          // uniforms * 2^32, by slot
        auto draw_uniforms = [&](uint32_t step) {
#pragma unroll
            for (int h = 0; h < NPH; h++) {                     // component c of call h belongs to row 4h + c of the band
                const uint4 rnd = philox4x32_10(make_uint4((uint32_t)x, gband + (uint32_t)h, step, 0u), key);
                uu[UPPER ? 4 * h + 0 : RPT - 1 - (4 * h + 0)] = __uint2float_rz(rnd.x);
                uu[UPPER ? 4 * h + 1 : RPT - 1 - (4 * h + 1)] = __uint2float_rz(rnd.y);
                uu[UPPER ? 4 * h + 2 : RPT - 1 - (4 * h + 2)] = __uint2float_rz(rnd.z);
                uu[UPPER ? 4 * h + 3 : RPT - 1 - (4 * h + 3)] = __uint2float_rz(rnd.w);
            }
        };
        if (A.u == nullptr) draw_uniforms(A.step0);
        float keep_q[RPT]; uint32_t keep_addr[RPT];
#pragma unroll
        for (int i = 0; i < RPT; i++) { keep_q[i] = 0.0f; keep_addr[i] = q_site0; }
        int acc = 0;                                            // lane l: packed statistics of the sweep with (sweep & 31) == l

        // One pass: finish sweep k-1 on state k (FIN), draw sweep k (DRAW).  No CTA barrier: a warp waits only for the
        // three messages it reads -- the edge words of its left / right neighbour warps and the other band's ballot --
        // each an 8-byte {word, sequence number} in shared memory, double-buffered by state parity like the halo
        // mailboxes (a warp can be at most one state ahead of a warp it exchanges messages with).  Interior slots
        // first, the boundary slot 0 last (its halo word travels through L2 meanwhile), as in K6p.
        auto sweep = [&](auto fin_c, auto draw_c, const int k) {
            constexpr bool FIN = decltype(fin_c)::value, DRAW = decltype(draw_c)::value;
            const uint32_t par = (state_no + (uint32_t)k) & 1u, seq = state_no + (uint32_t)k + 1u;
            float tparam = 0.0f;
            if (DRAW) {
                tparam = s_tparam[k];
                if (A.u != nullptr) {
#pragma unroll
                    for (int i = 0; i < RPT; i++)
                        uu[i] = A.u[((size_t)k * A.B + b) * N + (size_t)(row0 + local_row(i)) * L + x] * 4294967296.0f;
                }
            }
            uint32_t upd = 0xFFFFFFFFu;                                            // bit i: slot i updates Q (sweep k-1)
            if (MASK && FIN) {
                const uint8_t *m = A.mask + ((size_t)(k - 1) * A.B + b) * N + (size_t)row0 * L + x;
                upd = 0;
#pragma unroll
                for (int i = 0; i < RPT; i++) upd |= (m[local_row(i) * L] ? 1u : 0u) << i;
            }
            // neighbour counts of state k for all slots at once (the boundary slot still lacks its halo neighbour)
            uint32_t left = __shfl_up_sync(0xFFFFFFFFu, own, 1), right = __shfl_down_sync(0xFFFFFFFFu, own, 1);
            unsigned long long e, inner;
            for (;;) {
                e = lds_msg(edge_in + par * EDGE_BUF);
                inner = lds_msg(inner_in + par * INNER_BUF);
                const bool ok = (uint32_t)(inner >> 32) == seq && (!edge_lane || (uint32_t)(e >> 32) == seq);
                if (__all_sync(0xFFFFFFFFu, ok)) break;
            }
            if (lane == 0) left = (uint32_t)e;
            if (lane == 31) right = (uint32_t)e;
            uint32_t cnt = (own << 4) + (own >> 4) + left + right + ((((uint32_t)inner >> lane) & 1u) << TOP);
            uint32_t nxt_own = 0;
            // the halo word of state k: asked for now, looked at after the interior slots
            if ((uint32_t)(hv >> 32) != seq) hv = ld_halo(mb_in + par * MB_PARITY);

            uint32_t qaddr[RPT];
            auto finish = [&](auto ic) {
                constexpr int i = decltype(ic)::value;
                // g = 2^23 + ups as float bits.  g - (2^23 + 2) = (float)(ups - 2) exactly, and g * PLANE = ups * PLANE
                // modulo 2^32 (0x4B000000 * PLANE is a multiple of 2^32): one word serves the reward and the address.
                const uint32_t g = ((cnt >> (4 * i)) & 15u) | 0x4B000000u;
                if constexpr (FIN) {
                    const float t = __fmaf_rn(__uint_as_float(g) - 8388610.0f, sgn[i], -keep_q[i]);   // (2a-1)(ups-2) - q: one rounding
                    if (!MASK || ((upd >> i) & 1u)) sts_f32_at<(uint32_t)i * ROWB>(keep_addr[i], keep_q[i] + A.lr * t);
                }
                asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(qaddr[i]) : "r"(g), "n"(PLANE), "r"(q_site0));
            };
            auto decide = [&](auto ic, const float2 q) {
                constexpr int i = decltype(ic)::value;
                const int a = draw_action_scaled(uu[i], q.x, q.y, tparam);
                keep_q[i] = a ? q.y : q.x;
                keep_addr[i] = qaddr[i] + (a ? 4u : 0u);                               // (+ i * ROWB in the store instruction)
                sgn[i] = a ? 1.0f : -1.0f;
                nxt_own |= a ? (1u << (4 * i)) : 0u;
                return a;
            };
            // ---- interior slots 1 .. RPT-1 (staged: all finishes, all Q-pair loads, all decisions) ----
            float2 pr[RPT];
            int a_top = 0;
            static_for<1, RPT>([&](auto ic) { finish(ic); });
            if (DRAW) {
                static_for<1, RPT>([&](auto ic) {
                    constexpr int i = decltype(ic)::value;
                    pr[i] = lds_f32x2_at<(uint32_t)i * ROWB>(qaddr[i]);
                });
                static_for<1, RPT>([&](auto ic) {
                    constexpr int i = decltype(ic)::value;
                    const int a = decide(ic, pr[i]);
                    if (i == RPT - 1) a_top = a;
                });
                const uint32_t wN = __ballot_sync(0xFFFFFFFFu, a_top != 0);         // slot RPT-1: the row the other band looks at
                if (lane == 0) sts_msg(inner_out + (par ^ 1u) * INNER_BUF, wN, seq + 1u);
            }
            // ---- the boundary slot 0: halo word of state k, count, finish, draw, its new word straight to the neighbour ----
            while ((uint32_t)(hv >> 32) != seq) hv = ld_halo(mb_in + par * MB_PARITY);
            cnt += ((uint32_t)hv >> lane) & 1u;
            finish(std::integral_constant<int, 0>{});
            if (DRAW) {
                const float2 q = lds_f32x2_at<0>(qaddr[0]);
                const int a = decide(std::integral_constant<int, 0>{}, q);
                const uint32_t w0 = __ballot_sync(0xFFFFFFFFu, a != 0);
                if (lane == 0) st_halo(mb_out + (par ^ 1u) * MB_PARITY, w0, seq + 1u);
                if (edge_lane) sts_msg(edge_out + (par ^ 1u) * EDGE_BUF, nxt_own, seq + 1u);
            }
            if (FIN) {                                    // statistics of sweep k-1 from the complete counts of state k
                const uint32_t n_up = (uint32_t)__popc(own);
                const uint32_t s_all = field_sum(cnt & FIELDS), s_up = field_sum(cnt & (own * 15u));
                // sum_i (2a-1)(ups-2) + 2 RPT  (>= 0), packed above the up count
                int packed = (int)(n_up + ((2u * s_up - s_all - 4u * n_up + 4u * RPT) << 16));
                packed = __reduce_add_sync(0xFFFFFFFFu, packed);
                if (lane == ((k - 1) & 31)) acc = packed;
                // every 32 sweeps and after the last one: the warps' sums meet in shared memory, warp 0 adds them up
                if ((k & 31) == 0 || !DRAW) {
                    s_wstat[warp * 32 + lane] = acc;
                    acc = 0;
                    __syncthreads();
                    const int ks = ((k - 1) & ~31) + lane;
                    if (warp == 0 && ks < k) {
                        int pk = 0;
#pragma unroll
                        for (int ww = 0; ww < NW; ww++) pk += s_wstat[ww * 32 + lane];
                        atomicAdd(&A.n_up[(size_t)ks * A.B + b], pk & 0xFFFF);
                        if (A.reward_sum) atomicAdd(&A.reward_sum[(size_t)ks * A.B + b], (float)((pk >> 16) - 2 * RPT * NT));
                    }
                    __syncthreads();
                }
            }
            if (DRAW) own = nxt_own;
        };
        sweep(std::false_type{}, std::true_type{}, 0);
        for (int k = 1; k < A.K; k++) {
            if (A.u == nullptr) draw_uniforms(A.step0 + (uint32_t)k);
            sweep(std::true_type{}, std::true_type{}, k);
        }
        sweep(std::true_type{}, std::false_type{}, A.K);        // (ends with a barrier: every warp's Q updates are in shared memory)
#pragma unroll
        for (int i = 0; i < RPT; i++)
            A.spins[lbase + (size_t)(row0 + local_row(i)) * L + x] = (int8_t)((own >> (4 * i)) & 1u);
    };

    uint32_t state_no = 0;                                      // lattice states published so far by this slot
    for (int b = slot; b < A.B; b += n_slots, state_no += (uint32_t)A.K + 1u) {
        const size_t lbase = (size_t)b * N;
        __syncthreads();                                        // the previous lattice's Q strip has been stored (first pass: the tables are set)
        if (PL) {                                               // (every warp has left the previous lattice's last draw)
            asm volatile("cp.async.wait_all;" ::: "memory");
            for (int i = tid; i < A.K; i += NT) s_tparam[i] = temperature_param(s_traw[i]);
            if (b + n_slots < A.B) prefetch_column(b + n_slots);
        }
        for (int sp = 0; sp < 5; sp++) {
            const float4 *s4 = (const float4 *)(A.Q + (lbase * 5 + (size_t)sp * N + (size_t)row0 * L) * 2);
            float4 *d4 = (float4 *)(s_q + (size_t)sp * STRIP * 2);
#pragma unroll 4
            for (int i = tid; i < STRIP / 2; i += NT) {
                const int sr = i / (L / 2), c4 = i % (L / 2);
                d4[i] = s4[(sr < RPT ? sr : ROWS - 1 - sr + RPT) * (L / 2) + c4];
            }
        }
        __syncthreads();                                        // the strip and the table are complete before anybody draws
        if (upper) run_lattice(std::true_type{}, b, state_no);
        else run_lattice(std::false_type{}, b, state_no);
        for (int sp = 0; sp < 5; sp++) {
            float4 *d4 = (float4 *)(A.Q + (lbase * 5 + (size_t)sp * N + (size_t)row0 * L) * 2);
            const float4 *s4 = (const float4 *)(s_q + (size_t)sp * STRIP * 2);
#pragma unroll 4
            for (int i = tid; i < STRIP / 2; i += NT) {
                const int sr = i / (L / 2), c4 = i % (L / 2);
                d4[(sr < RPT ? sr : ROWS - 1 - sr + RPT) * (L / 2) + c4] = s4[i];
            }
        }
    }
}


template <typename T>
static size_t resident_smem_bytes(int L, int rows) {
    const int wpr = (L + 31) >> 5;
    return (size_t)5 * rows * L * 2 * sizeof(T) + (size_t)2 * (rows + 2) * wpr * 4 + 48;   // bit buffers, 2 mbarriers, statistics
}

// cluster size for a lattice side, 0 = the resident kernel does not apply
template <typename T>
static int resident_cluster_size(int L) {
    const int wpr = (L + 31) >> 5, LP = wpr * 32;
    for (int C = 1; C <= 16; C *= 2) {
        if (L % C) continue;
        const int rows = L / C;
        if (C > 1 && rows % kIsingRB) continue;
        const int bands = (rows + kIsingRB - 1) / kIsingRB;
        if (LP * bands <= 1024 && resident_smem_bytes<T>(L, rows) <= 200 * 1024) return C;
    }
    return 0;
}

// fp32 shapes with a compile-time specialisation (rows per thread from MFMARL_ISING_RPT, default 8: measured 11 % faster than 4)
static void specialised_resident_kernel(const IsingRunArgs<double> &, void (*&)(const IsingRunArgs<double>), unsigned &) {}
static void specialised_resident_kernel(const IsingRunArgs<float> &A, void (*&kern)(const IsingRunArgs<float>), unsigned &threads) {
    const char *env = getenv("MFMARL_ISING_RPT");
    const int rpt = env ? atoi(env) : 8;
    if (env && atoi(env) == 0) return;                 // 0 = force the generic kernel (tests)
#define MF_PICK(LL, RR) \
    if (A.L == LL && A.rows_per == RR) { \
        if (rpt == 8) { kern = A.mask ? k_ising_resident_f32<LL, RR, 8, true> : k_ising_resident_f32<LL, RR, 8, false>; threads = LL * (RR / 8); } \
        else { kern = A.mask ? k_ising_resident_f32<LL, RR, 4, true> : k_ising_resident_f32<LL, RR, 4, false>; threads = LL * (RR / 4); } \
        return; \
    }
    MF_PICK(256, 16) MF_PICK(128, 32) MF_PICK(64, 64)
#undef MF_PICK
}

// K6p launcher (fp32, C > 1 strips per lattice): false = no persistent specialisation for this shape / switched off.
// pl: per-lattice temperature table [K][B]; only K6s has such a variant (launch_ising_resident refuses the overrides
// that would select K6p before it gets here)
static bool launch_ising_persistent(const IsingRunArgs<double> &, cudaStream_t, bool) { return false; }
static bool launch_ising_persistent(const IsingRunArgs<float> &A, cudaStream_t st, bool pl) {
    const char *env = getenv("MFMARL_ISING_PERSIST");
    const char *renv = getenv("MFMARL_ISING_RPT");
    if (A.L != 512) {                                               // (512: K6s is the only resident kernel, see below)
        if (env && atoi(env) == 0) return false;                    // 0 = the cluster kernel K6r (tests, comparisons)
        if (renv && atoi(renv) == 0) return false;                  // the generic kernel was asked for
    }
    const int rpt = renv ? atoi(renv) : 8;
    void (*kern)(const IsingRunArgs<float>, int, unsigned long long *) = nullptr;
    unsigned threads = 0;
#define MF_PICK(LL, RR) \
    if (A.L == LL && A.rows_per == RR) { \
        if (rpt == 8) { kern = A.mask ? k_ising_persist_f32<LL, RR, 8, true> : k_ising_persist_f32<LL, RR, 8, false>; threads = LL * (RR / 8); } \
        else { kern = A.mask ? k_ising_persist_f32<LL, RR, 4, true> : k_ising_persist_f32<LL, RR, 4, false>; threads = LL * (RR / 4); } \
    }
    if (!pl) { MF_PICK(256, 16) MF_PICK(128, 32) }
#undef MF_PICK
    // K6s (SWAR neighbour counts): strips of two bands of 8 rows whatever K6r's cluster would be (no cluster here, so
    // the strip height is free); MFMARL_ISING_PERSIST=1 keeps K6p
    int rows_per = A.rows_per;
    bool swar = false;
    if (!(env && atoi(env) == 1) && rpt == 8) {
#define MF_PICK(LL) \
        if (A.L == LL) { kern = pl ? (A.mask ? k_ising_persist_swar_f32<LL, 8, true, true> : k_ising_persist_swar_f32<LL, 8, false, true>) \
                                   : (A.mask ? k_ising_persist_swar_f32<LL, 8, true, false> : k_ising_persist_swar_f32<LL, 8, false, false>); \
                         threads = 2 * LL; rows_per = 16; swar = true; }
        MF_PICK(256) MF_PICK(128) MF_PICK(64)
#undef MF_PICK
    }
    // 512 x 512: a 16-row strip's Q (327 KB) does not fit, so strips of 8 rows with 4 rows per thread (1024 threads, 64
    // registers); no cluster kernel exists for this side, so neither MFMARL_ISING_PERSIST nor _RPT (other than 0) applies
    if (A.L == 512) {
        kern = pl ? (A.mask ? k_ising_persist_swar_f32<512, 4, true, true> : k_ising_persist_swar_f32<512, 4, false, true>)
                  : (A.mask ? k_ising_persist_swar_f32<512, 4, true, false> : k_ising_persist_swar_f32<512, 4, false, false>);
        threads = 1024; rows_per = 8; swar = true;
    }
    if (!kern) return false;
    const int C = A.L / rows_per, wpr = A.L / 32;
    constexpr int kMaxSweeps = 4096;                                 // per launch: the temperature table lives in shared memory
    if (A.K > kMaxSweeps) {
        for (int k0 = 0; k0 < A.K; k0 += kMaxSweeps) {
            IsingRunArgs<float> part = A;
            part.K = std::min(kMaxSweeps, A.K - k0);
            part.temperatures = A.temperatures + (size_t)k0 * (pl ? A.B : 1); part.step0 = A.step0 + (uint32_t)k0;
            if (A.u) part.u = A.u + (size_t)k0 * A.B * A.L * A.L;
            if (A.mask) part.mask = A.mask + (size_t)k0 * A.B * A.L * A.L;
            part.n_up = A.n_up + (size_t)k0 * A.B;
            if (A.reward_sum) part.reward_sum = A.reward_sum + (size_t)k0 * A.B;
            if (!launch_ising_persistent(part, st, pl)) return false;
        }
        return true;
    }
    // K6p: bit buffers + statistics; K6s: message slots [2][2][wpr] x (1 + 2) of 8 bytes + [warps][32] statistics
    const size_t smem = (swar ? (size_t)5 * rows_per * A.L * 8 + (size_t)2 * 2 * wpr * 3 * 8 + (size_t)(threads / 32) * 32 * 4
                              : resident_smem_bytes<float>(A.L, rows_per)) + (size_t)A.K * sizeof(float) * (pl ? 2 : 1);
    MF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int dev = 0, n_sm = 0, per_sm = 0;
    MF_CUDA(cudaGetDevice(&dev));
    MF_CUDA(cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev));
    MF_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, (int)threads, smem));
    const int n_slots = std::min(A.B, per_sm * n_sm / C);           // lattices in flight: 9 of 16 strips on 148 SMs
    if (n_slots < 1) return false;
    // mailboxes [slot][rank][parity][top|bottom][wpr]: one buffer per (device, stream), kept for the life of the process
    // (launches on one stream are ordered, so they can share it; a stream-ordered allocation per launch made the
    // host-synchronised loop of bench.py's e2e leg jitter by hundreds of milliseconds)
    const size_t halo_bytes = (size_t)n_slots * C * 2 * 2 * wpr * sizeof(unsigned long long);
    unsigned long long *halo = nullptr;
    {
        static std::mutex mu;
        static std::map<std::pair<int, cudaStream_t>, std::pair<unsigned long long *, size_t>> pool;
        std::lock_guard<std::mutex> lock(mu);
        auto &slot = pool[std::make_pair(dev, st)];
        if (slot.second < halo_bytes) {
            if (slot.first) { MF_CUDA(cudaStreamSynchronize(st)); cudaFree(slot.first); }
            MF_CUDA(cudaMalloc(&slot.first, halo_bytes));
            slot.second = halo_bytes;
        }
        halo = slot.first;
    }
    MF_CUDA(cudaMemsetAsync(halo, 0, halo_bytes, st));              // sequence numbers start at 1
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(n_slots * C)); cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;                    // the strips of a lattice wait for each other: the
    attr[0].val.cooperative = 1;                                    // whole grid must be resident at once
    cfg.attrs = attr; cfg.numAttrs = 1;
    const cudaError_t err = cudaLaunchKernelEx(&cfg, kern, A, n_slots, halo);
    if (err == cudaErrorCooperativeLaunchTooLarge && A.L != 512) {
        // fewer SMs are available to this process than the device reports (MPS with a limited SM share, ...): the
        // co-scheduled grid cannot be resident at once -- leave the launch to the cluster kernel K6r, same bits
        (void)cudaGetLastError();
        return false;
    }
    MF_CUDA(err);
    return true;
}

// The environment overrides that select a kernel without per-lattice temperature tables (K6p, the specialised K6r)
// refuse a per-lattice call instead of running another kernel.  They only ever apply to fp32 below side 512.
static void refuse_per_lattice_overrides(int L) {
    const char *penv = getenv("MFMARL_ISING_PERSIST"), *renv = getenv("MFMARL_ISING_RPT");
    if (L == 512) return;
    if (penv && atoi(penv) == 1)
        throw Fatal("MFMARL_ISING_PERSIST=1 selects K6p, which has no per-lattice temperature tables");
    if (renv && atoi(renv) != 0 && atoi(renv) != 8)
        throw Fatal(std::string("MFMARL_ISING_RPT=") + renv + " selects a specialised kernel without per-lattice temperature tables");
    if (penv && atoi(penv) == 0 && !(renv && atoi(renv) == 0) && (L == 64 || L == 128 || L == 256))
        throw Fatal("MFMARL_ISING_PERSIST=0 selects the specialised cluster kernel k_ising_resident_f32, which has no per-lattice "
                    "temperature tables (MFMARL_ISING_RPT=0 selects the generic one)");
}

// pl: A.temperatures is [K][B] (per-lattice schedules, mfi_run_lattices) instead of [K]
template <typename T>
static void launch_ising_resident(const IsingRunArgs<T> &A0, cudaStream_t st, bool pl = false) {
    IsingRunArgs<T> A = A0;
    const int L = A.L, wpr = (L + 31) >> 5, LP = wpr * 32;
    const int C = resident_cluster_size<T>(L);
    A.rows_per = C > 0 ? L / C : 0;
    if (pl && sizeof(T) == 4) refuse_per_lattice_overrides(L);
    if (launch_ising_persistent(A, st, pl)) return;                 // (declines shapes it has no specialisation for)
    if (C == 0) throw Fatal("ising resident kernel: lattice side " + std::to_string(L) + " not supported (use mfi_step)");
    const int bands = (A.rows_per + kIsingRB - 1) / kIsingRB;
    const size_t smem = resident_smem_bytes<T>(L, A.rows_per);
    const bool fast = (L % 32 == 0) && (A.rows_per % kIsingRB == 0);
    void (*kern)(const IsingRunArgs<T>) = pl ? (fast ? k_ising_resident_lattices<T, true> : k_ising_resident_lattices<T, false>)
                                             : (fast ? k_ising_resident<T, true> : k_ising_resident<T, false>);
    unsigned threads = (unsigned)(LP * bands);
    if (!pl) specialised_resident_kernel(A, kern, threads);
    MF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (C > 8) MF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(A.B * C)); cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    MF_CUDA(cudaLaunchKernelEx(&cfg, kern, A));
}

// ----------------------------------------------------------------------------------------------
// The Ising ENVIRONMENT step on its own (examples/ising_model/multiagent/environment.py:49-92, core.py:99-125,
// Ising.py:101-118): a caller-supplied action vector is applied, then every site gets its reward and observation
// on the NEW lattice.  This is what IsingMultiAgentEnv.step / reset return, for callers that bring their own policy
// (the unmodified main_MFQ_Ising.py); the fused kernels above are the same step with the tabular policy inside.
//   k_ising_env_apply    spin_i <- [action_i > 0]                     (environment.py:112-114, core.py:118-125)
//   k_ising_env_observe  obs_i = the 4 torus neighbours' spins in ascending flat-index order (Ising.py:113-118 returns
//                        global_state.flatten()[np.where(mask == 1)]), reward_i = 0.5 sigma_i sum_nbr sigma_j
//                        (Ising.py:101-111), n_up (core.py:106-110)
// ----------------------------------------------------------------------------------------------
__global__ void k_ising_env_apply(int8_t *__restrict__ spins, const int32_t *__restrict__ actions, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) spins[i] = actions[i] <= 0 ? 0 : 1;
}

__global__ void k_ising_env_observe(const int8_t *__restrict__ spins, int L, uint8_t *__restrict__ obs,
                                    float *__restrict__ reward, int32_t *__restrict__ n_up) {
    const int b = blockIdx.y, N = L * L;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int8_t *sp = spins + (size_t)b * N;
    int a = 0;
    if (i < N) {
        const int r = i / L, c = i - r * L;
        const int ru = r == 0 ? L - 1 : r - 1, rd = r == L - 1 ? 0 : r + 1;
        const int cl = c == 0 ? L - 1 : c - 1, cr = c == L - 1 ? 0 : c + 1;
        int id[4] = {ru * L + c, rd * L + c, r * L + cl, r * L + cr};
        // np.where(mask == 1) lists the neighbours by ascending flat index: sort the four (5-comparator network)
#define MF_CSWAP(x, y) { const int lo = min(id[x], id[y]), hi = max(id[x], id[y]); id[x] = lo; id[y] = hi; }
        MF_CSWAP(0, 1) MF_CSWAP(2, 3) MF_CSWAP(0, 2) MF_CSWAP(1, 3) MF_CSWAP(1, 2)
#undef MF_CSWAP
        int ups = 0;
        uint32_t packed = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) { const int v = sp[id[k]] != 0; ups += v; packed |= (uint32_t)v << (8 * k); }
        a = sp[i] != 0;
        if (obs) ((uint32_t *)obs)[(size_t)b * N + i] = packed;
        if (reward) reward[(size_t)b * N + i] = 0.5f * (float)(2 * a - 1) * (float)(2 * ups - 4);
    }
    const unsigned up_mask = __ballot_sync(0xFFFFFFFFu, a != 0);
    if (n_up && (threadIdx.x & 31) == 0 && up_mask) atomicAdd(&n_up[b], __popc(up_mask));
}

}  // namespace mfmarl

using namespace mfmarl;

extern "C" int mfi_env_step(int n_lattices, int side, int8_t *d_spins, const int32_t *d_actions, uint8_t *d_obs,
                            float *d_reward, int32_t *d_n_up, void *stream) {
    try {
        if (n_lattices < 1 || side < 3) throw Fatal("mfi_env_step: need at least one lattice of side >= 3");
        if (!d_spins) throw Fatal("mfi_env_step: null lattice");
        if (d_obs && ((uintptr_t)d_obs & 3)) throw Fatal("mfi_env_step: d_obs must be 4-byte aligned");
        cudaStream_t st = (cudaStream_t)stream;
        const size_t n = (size_t)n_lattices * side * side;
        if (d_actions) {
            k_ising_env_apply<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_spins, d_actions, n);
            MF_CUDA(cudaGetLastError());
        }
        if (d_obs || d_reward || d_n_up) {
            if (d_n_up) MF_CUDA(cudaMemsetAsync(d_n_up, 0, (size_t)n_lattices * sizeof(int32_t), st));
            const dim3 grid((unsigned)((side * side + 255) / 256), (unsigned)n_lattices);
            k_ising_env_observe<<<grid, 256, 0, st>>>(d_spins, side, d_obs, d_reward, d_n_up);
            MF_CUDA(cudaGetLastError());
        }
    } catch (const std::exception &ex) {
        set_last_error(std::string("mfi_env_step: ") + ex.what());
        return -1;
    }
    return 0;
}


extern "C" int mfi_step(int dtype, int n_lattices, int side, int8_t *d_spins, void *d_q, double temperature,
                        double lr, const void *d_uniforms, const uint8_t *d_update_mask, unsigned seed,
                        unsigned lattice_base, unsigned step, int32_t *d_n_up, void *d_reward_sum, void *d_mse,
                        void *stream) {
    try {
        if (dtype == 0) {
            IsingArgs<float> A{n_lattices, side, d_spins, (float *)d_q, (float)temperature, (float)lr,
                               (const float *)d_uniforms, d_update_mask, seed, lattice_base, step, d_n_up,
                               (float *)d_reward_sum, (float *)d_mse};
            launch_ising(A, (cudaStream_t)stream);
        } else if (dtype == 1) {
            IsingArgs<double> A{n_lattices, side, d_spins, (double *)d_q, temperature, lr,
                                (const double *)d_uniforms, d_update_mask, seed, lattice_base, step, d_n_up,
                                (double *)d_reward_sum, (double *)d_mse};
            launch_ising(A, (cudaStream_t)stream);
        } else throw Fatal("mfi_step: dtype must be 0 (f32) or 1 (f64)");
    } catch (const std::exception &ex) {
        set_last_error(std::string("mfi_step: ") + ex.what());
        return -1;
    }
    return 0;
}

extern "C" int mfi_step_lattices(int dtype, int n_lattices, int side, int8_t *d_spins, void *d_q,
                                 const void *d_temperatures, double lr, const void *d_uniforms,
                                 const uint8_t *d_update_mask, unsigned seed, unsigned lattice_base, unsigned step,
                                 int32_t *d_n_up, void *d_reward_sum, void *d_mse, void *stream) {
    try {
        if (!d_temperatures) throw Fatal("need a device temperature table [n_lattices]");
        if (dtype == 0) {
            IsingArgs<float> A{n_lattices, side, d_spins, (float *)d_q, 0.0f, (float)lr,
                               (const float *)d_uniforms, d_update_mask, seed, lattice_base, step, d_n_up,
                               (float *)d_reward_sum, (float *)d_mse};
            launch_ising(A, (cudaStream_t)stream, (const float *)d_temperatures);
        } else if (dtype == 1) {
            IsingArgs<double> A{n_lattices, side, d_spins, (double *)d_q, 0.0, lr,
                                (const double *)d_uniforms, d_update_mask, seed, lattice_base, step, d_n_up,
                                (double *)d_reward_sum, (double *)d_mse};
            launch_ising(A, (cudaStream_t)stream, (const double *)d_temperatures);
        } else throw Fatal("dtype must be 0 (f32) or 1 (f64)");
    } catch (const std::exception &ex) {
        set_last_error(std::string("mfi_step_lattices: ") + ex.what());
        return -1;
    }
    return 0;
}

extern "C" int mfi_resident_cluster_size(int dtype, int side) {
    if (dtype != 1 && side == 512) return 64;          // K6s only: 64 strips of 8 rows (no cluster kernel at this side)
    return dtype == 1 ? resident_cluster_size<double>(side) : resident_cluster_size<float>(side);
}

extern "C" int mfi_run(int dtype, int n_lattices, int side, int n_sweeps, int8_t *d_spins, void *d_q,
                       const void *d_temperatures, double lr, const void *d_uniforms, const uint8_t *d_update_mask,
                       unsigned seed, unsigned lattice_base, unsigned step0, int32_t *d_n_up, void *d_reward_sum,
                       void *stream) {
    try {
        if (n_sweeps < 1 || n_lattices < 1) throw Fatal("mfi_run: need at least one sweep and one lattice");
        if (dtype == 0) {
            IsingRunArgs<float> A{n_lattices, side, n_sweeps, 0, d_spins, (float *)d_q, (const float *)d_temperatures,
                                  (float)lr, (const float *)d_uniforms, d_update_mask, seed, lattice_base, step0, d_n_up,
                                  (float *)d_reward_sum};
            launch_ising_resident(A, (cudaStream_t)stream);
        } else if (dtype == 1) {
            IsingRunArgs<double> A{n_lattices, side, n_sweeps, 0, d_spins, (double *)d_q, (const double *)d_temperatures,
                                   lr, (const double *)d_uniforms, d_update_mask, seed, lattice_base, step0, d_n_up,
                                   (double *)d_reward_sum};
            launch_ising_resident(A, (cudaStream_t)stream);
        } else throw Fatal("mfi_run: dtype must be 0 (f32) or 1 (f64)");
    } catch (const std::exception &ex) {
        set_last_error(std::string("mfi_run: ") + ex.what());
        return -1;
    }
    return 0;
}

extern "C" int mfi_run_lattices(int dtype, int n_lattices, int side, int n_sweeps, int8_t *d_spins, void *d_q,
                                const void *d_temperatures, double lr, const void *d_uniforms,
                                const uint8_t *d_update_mask, unsigned seed, unsigned lattice_base, unsigned step0,
                                int32_t *d_n_up, void *d_reward_sum, void *stream) {
    try {
        if (n_sweeps < 1 || n_lattices < 1) throw Fatal("need at least one sweep and one lattice");
        if (!d_temperatures) throw Fatal("need a device temperature table [n_sweeps][n_lattices]");
        if (dtype == 0) {
            IsingRunArgs<float> A{n_lattices, side, n_sweeps, 0, d_spins, (float *)d_q, (const float *)d_temperatures,
                                  (float)lr, (const float *)d_uniforms, d_update_mask, seed, lattice_base, step0, d_n_up,
                                  (float *)d_reward_sum};
            launch_ising_resident(A, (cudaStream_t)stream, true);
        } else if (dtype == 1) {
            IsingRunArgs<double> A{n_lattices, side, n_sweeps, 0, d_spins, (double *)d_q, (const double *)d_temperatures,
                                   lr, (const double *)d_uniforms, d_update_mask, seed, lattice_base, step0, d_n_up,
                                   (double *)d_reward_sum};
            launch_ising_resident(A, (cudaStream_t)stream, true);
        } else throw Fatal("dtype must be 0 (f32) or 1 (f64)");
    } catch (const std::exception &ex) {
        set_last_error(std::string("mfi_run_lattices: ") + ex.what());
        return -1;
    }
    return 0;
}
