// K8: checkerboard single-spin-flip Metropolis on batches of L x L tori -- the MCMC reference that MF-Q's Ising
// curve (order parameter against temperature) is compared with.
//
// Model: H = -1/2 sum_bonds sigma_i sigma_j = -1/2 sum_i r_i with r_i = 1/2 sigma_i sum_nbr sigma_j the environment's
// reward (Ising.py:101-111): coupling J = 1/2, Tc = 1 / ln(1 + sqrt 2) ~ 1.1346 on MF-Q's temperature axis.  Flipping
// site i changes the energy by h = sigma_i sum_nbr sigma_j in {-4, -2, 0, 2, 4}: a flip with h <= 0 is always accepted, one with h in {2, 4}
// when the site's 32-bit Philox word is below floor(exp(-h / T) * 2^32), computed on the host in double with the C
// library's exp -- no device transcendental takes part in a decision, so a CPU restatement reproduces every bit.
// One sweep = all sites with (x + y) even, then all with (x + y) odd (L even: the torus is bipartite).
//
// Mapping: one CTA per lattice, the lattice bit-packed in shared memory for the whole launch (row-major words of 32
// columns, 512 x 512 = 32 KB).  A thread owns whole words.  Per word and colour it forms the four neighbour words
// (up / down: same word of the adjacent rows; left / right: the word shifted by one column, the bit that crosses the
// word or wraps the row fetched on its own), the bit-sliced count of aligned neighbours (3 and 4 aligned = h 2 and 4),
// one Philox4x32-10 call per 4 sites of the colour that may need a draw, and writes the flips back.  Only the owner
// writes a word; the other threads read from it only bits of the colour that is not being updated.  The statistics
// come from the odd half: after it, sum_{odd i} sigma_i sum_nbr sigma_j is the whole bond sum (every bond has one odd
// end), and the word holds its final spins.
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "../../include/mfmarl_batched.h"
#include "rng.cuh"
#include "engine.h"

namespace mfmarl {

constexpr uint32_t kMetropolisTag = 2u;      // counter word 3: MF-Q uses 0 and 1 there
constexpr int kMetropolisThreads = 256;

struct MetropolisArgs {
    int B, L, K;
    int8_t *spins;                 // [B][L][L] in/out
    const uint32_t *thr;           // [K][B][2]: acceptance thresholds for h = 2 and h = 4
    uint32_t seed, lattice_base, step0;
    int32_t *n_up, *bond_sum;      // [K][B] out (or null)
};

__global__ void __launch_bounds__(kMetropolisThreads) k_ising_metropolis(const MetropolisArgs A) {
    extern __shared__ uint32_t s_w[];                       // [L][wpr]
    __shared__ int s_stat[2][2];                            // (up count, bond sum) by sweep parity
    const int L = A.L, wpr = (L + 31) >> 5, nw = L * wpr;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = blockDim.x >> 5;
    const size_t lbase = (size_t)b * L * L;
    const uint2 key = make_uint2(A.seed, A.lattice_base + (uint32_t)b);

    if (tid < 4) (&s_stat[0][0])[tid] = 0;
    for (int wi = warp; wi < nw; wi += nwarp) {             // a warp packs one word: lane = column
        const int y = wi / wpr, x = (wi - y * wpr) * 32 + lane;
        const uint32_t word = __ballot_sync(0xFFFFFFFFu, x < L && A.spins[lbase + (size_t)y * L + x] != 0);
        if (lane == 0) s_w[wi] = word;
    }
    __syncthreads();

    auto bit = [&](int y, int x) { return (s_w[y * wpr + (x >> 5)] >> (x & 31)) & 1u; };
    for (int k = 0; k < A.K; k++) {
        const uint32_t thr2 = A.thr[((size_t)k * A.B + b) * 2], thr4 = A.thr[((size_t)k * A.B + b) * 2 + 1];
        const uint32_t step = A.step0 + (uint32_t)k;
        int nup = 0, bonds = 0;
        for (int c = 0; c < 2; c++) {
            for (int wi = tid; wi < nw; wi += blockDim.x) {
                const int y = wi / wpr, w = wi - y * wpr, x0 = w * 32;
                const int nvalid = min(32, L - x0);
                const uint32_t valid = nvalid == 32 ? 0xFFFFFFFFu : (1u << nvalid) - 1u;
                const uint32_t cmask = (((uint32_t)c ^ (uint32_t)y) & 1u ? 0xAAAAAAAAu : 0x55555555u) & valid;
                const int yu = y == 0 ? L - 1 : y - 1, yd = y == L - 1 ? 0 : y + 1;
                const uint32_t cur = s_w[wi], up = s_w[yu * wpr + w], dn = s_w[yd * wpr + w];
                const uint32_t in_l = bit(y, x0 == 0 ? L - 1 : x0 - 1);                 // column left of the word
                const uint32_t in_r = bit(y, x0 + nvalid == L ? 0 : x0 + nvalid);       // column right of its last one
                const uint32_t lf = (cur << 1) | in_l, rt = (cur >> 1) | (in_r << (nvalid - 1));
                // aligned-neighbour indicators and their bit-sliced count
                const uint32_t e1 = ~(cur ^ up), e2 = ~(cur ^ dn), e3 = ~(cur ^ lf), e4 = ~(cur ^ rt);
                const uint32_t x1 = e1 ^ e2, c1 = e1 & e2, x2 = e3 ^ e4, c2 = e3 & e4;
                const uint32_t h2 = (x1 ^ x2) & (c1 ^ c2 ^ (x1 & x2)) & cmask;          // 3 aligned: h = 2
                const uint32_t h4 = c1 & c2 & cmask;                                     // 4 aligned: h = 4
                uint32_t flip = cmask & ~(h2 | h4);                                      // h <= 0
                const uint32_t need = h2 | h4, par = ((uint32_t)c ^ (uint32_t)y) & 1u;
#pragma unroll
                for (int q = 0; q < 4; q++) {                     // sites 2m + par, m = 4q .. 4q+3, of this colour
                    if (((need >> (8 * q)) & 0xFFu) == 0u) continue;
                    const uint4 r = philox4x32_10(make_uint4((uint32_t)wi * 4u + (uint32_t)q, step, (uint32_t)c, kMetropolisTag), key);
                    const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const int i = 8 * q + 2 * j + (int)par;
                        const uint32_t t = ((h4 >> i) & 1u) ? thr4 : thr2;
                        flip |= (((need >> i) & 1u) && rr[j] < t) ? (1u << i) : 0u;
                    }
                }
                const uint32_t nw_ = cur ^ flip;
                s_w[wi] = nw_;
                if (c == 1) {
                    // bond sum over the odd sites with their final spins (the even neighbours are final too)
                    const uint32_t a = __popc(~(nw_ ^ up) & cmask) + __popc(~(nw_ ^ dn) & cmask) +
                                       __popc(~(nw_ ^ lf) & cmask) + __popc(~(nw_ ^ rt) & cmask);
                    bonds += 2 * (int)a - 4 * __popc(cmask);
                    nup += __popc(nw_ & valid);
                }
            }
            __syncthreads();
        }
        // here every warp is past the odd half of sweep k; the totals of sweep k-1 were complete one barrier ago
        nup = __reduce_add_sync(0xFFFFFFFFu, nup);
        bonds = __reduce_add_sync(0xFFFFFFFFu, bonds);
        if (lane == 0 && (nup | bonds)) { atomicAdd(&s_stat[k & 1][0], nup); atomicAdd(&s_stat[k & 1][1], bonds); }
        if (tid == 0 && k > 0) {
            if (A.n_up) A.n_up[(size_t)(k - 1) * A.B + b] = s_stat[(k - 1) & 1][0];
            if (A.bond_sum) A.bond_sum[(size_t)(k - 1) * A.B + b] = s_stat[(k - 1) & 1][1];
            s_stat[(k - 1) & 1][0] = 0; s_stat[(k - 1) & 1][1] = 0;
        }
    }
    __syncthreads();
    if (tid == 0) {
        const int k = A.K - 1;
        if (A.n_up) A.n_up[(size_t)k * A.B + b] = s_stat[k & 1][0];
        if (A.bond_sum) A.bond_sum[(size_t)k * A.B + b] = s_stat[k & 1][1];
    }
    for (int wi = warp; wi < nw; wi += nwarp) {
        const int y = wi / wpr, x = (wi - y * wpr) * 32 + lane;
        if (x < L) A.spins[lbase + (size_t)y * L + x] = (int8_t)((s_w[wi] >> lane) & 1u);
    }
}

}  // namespace mfmarl

using namespace mfmarl;

extern "C" int mfi_metropolis(int n_lattices, int side, int n_sweeps, int8_t *d_spins, const double *h_temperatures,
                              unsigned seed, unsigned lattice_base, unsigned step0, int32_t *d_n_up,
                              int32_t *d_bond_sum, void *stream) {
    try {
        if (n_lattices < 1 || n_sweeps < 1) throw Fatal("need at least one lattice and one sweep");
        if (side < 2 || side > 512 || side % 2) throw Fatal("side must be even and in [2, 512], got " + std::to_string(side));
        if (!d_spins || !h_temperatures) throw Fatal("null spins or temperatures");
        const size_t n = (size_t)n_sweeps * n_lattices;
        std::vector<uint32_t> thr(2 * n);
        double last_T = 0.0;                          // neighbouring entries mostly repeat a temperature
        for (size_t i = 0; i < n; i++) {
            const double T = h_temperatures[i];
            if (!(T > 0.0) || !std::isfinite(T))
                throw Fatal("temperature " + std::to_string(T) + " at index " + std::to_string(i) + " is not finite and > 0");
            if (i > 0 && T == last_T) { thr[2 * i] = thr[2 * i - 2]; thr[2 * i + 1] = thr[2 * i - 1]; continue; }
            for (int j = 0; j < 2; j++) {
                const double t = std::floor(std::exp(-(double)(2 * (j + 1)) / T) * 4294967296.0);
                thr[2 * i + j] = t >= 4294967295.0 ? 0xFFFFFFFFu : (uint32_t)t;
            }
            last_T = T;
        }
        cudaStream_t st = (cudaStream_t)stream;
        uint32_t *d_thr = nullptr;
        MF_CUDA(cudaMallocAsync((void **)&d_thr, thr.size() * sizeof(uint32_t), st));
        MF_CUDA(cudaMemcpyAsync(d_thr, thr.data(), thr.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        const int wpr = (side + 31) / 32;
        const size_t smem = (size_t)side * wpr * sizeof(uint32_t);
        const MetropolisArgs A{n_lattices, side, n_sweeps, d_spins, d_thr, seed, lattice_base, step0, d_n_up, d_bond_sum};
        const int threads = std::min(kMetropolisThreads, std::max(32, (side * wpr + 31) / 32 * 32));
        k_ising_metropolis<<<n_lattices, threads, smem, st>>>(A);
        const cudaError_t err = cudaGetLastError();
        MF_CUDA(cudaFreeAsync(d_thr, st));
        MF_CUDA(err);
    } catch (const std::exception &ex) {
        set_last_error(std::string("mfi_metropolis: ") + ex.what());
        return -1;
    }
    return 0;
}
