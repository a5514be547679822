// K9: Swendsen-Wang cluster updates on batches of L x L tori -- the MCMC reference of the Ising curve that stays
// usable near Tc (its autocorrelation time there is a few sweeps and almost flat in L, where K8's single-spin flips
// need ~L^2.17) and at odd sides (no colouring).
//
// Model: as K8, H = -1/2 sum_bonds sigma_i sigma_j (coupling 1/2, Tc = 1 / ln(1 + sqrt 2) on MF-Q's temperature axis).
// Site i = y L + x owns its right bond to ((x + 1) mod L, y) and its down bond to (x, (y + 1) mod L): 2N bonds, the
// two between the same pair of sites at L = 2 are distinct bonds.  One sweep:
//   1. a bond is active iff its spins are aligned and its Philox word is below thr = min(floor((1 - exp(-1/T)) 2^32),
//      2^32 - 1), computed on the host in double with the C library's exp (Fortuin-Kasteleyn, p = 1 - e^(-2 beta J));
//   2. clusters = connected components of the active bonds, each labelled by its SMALLEST flat site index;
//   3. the cluster with root r flips as a whole iff r's flip word has its top bit set;
//   4. n_up and the bond sum of the final spins.
// Every decision is an integer comparison of a Philox word, and every result a function of the canonical labels, so
// tests/swendsen_wang_ref.py (numpy + scipy's connected components) reproduces every bit.
//
// Mapping: one CTA per lattice for the whole launch; in shared memory the spins (bit-packed, flat: site i is bit i & 31
// of word i >> 5), one flip bit per site (meaningful at roots) and a uint16 union-find label per site (N <= 65536):
// 2N + N/4 bytes, 144 KB at 256^2.  A thread owns units of 8 sites (one byte of the packed arrays), so it stores its
// bytes without atomics.  Labelling is lock-free union-find: label[i] = i; for every active bond union(i, j) finds both
// roots (with path halving) and atomicCAS-links the LARGER root under the smaller, retrying when the CAS loses; then
// every site stores its root.  Links only ever point from a larger index to a smaller one, so a component's final root
// is its minimum index whatever the interleaving of the threads: the labels, and so the flips, are deterministic.
// The bond sum of the state after sweep k is counted in the bond pass of sweep k + 1 (it tests every bond's alignment
// anyway); one last bond pass without draws counts it after the final sweep.
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "../../include/mfmarl_batched.h"
#include "rng.cuh"
#include "engine.h"

namespace mfmarl {

constexpr uint32_t kClusterTag = 3u;          // counter word 3: MF-Q uses 0 and 1 there, K8 uses 2
constexpr int kClusterThreads = 1024;
constexpr int kClusterMaxSide = 256;          // uint16 labels: N <= 65536

struct ClusterArgs {
    int B, L, K;
    int8_t *spins;                 // [B][L][L] in/out
    const uint32_t *thr;           // [K][B]: bond activation thresholds
    uint32_t seed, lattice_base, step0;
    int32_t *n_up, *bond_sum;      // [K][B] out (or null)
};

// root of x, halving the path on the way (every write points a node at one of its ancestors: labels only decrease
// along a path, so no cycle can form and a concurrent link is never undone)
__device__ __forceinline__ int uf_find(volatile uint16_t *lab, int x) {
    int p = lab[x];
    while (p != x) {
        const int g = lab[p];
        if (g == p) return p;
        lab[x] = (uint16_t)g;
        x = g;
        p = lab[x];
    }
    return x;
}

// root of x without writes: the final flattening, where another thread's halving could overwrite a stored root
__device__ __forceinline__ int uf_root(volatile const uint16_t *lab, int x) {
    int p = lab[x];
    while (p != x) { x = p; p = lab[x]; }
    return x;
}

__device__ __forceinline__ void uf_union(volatile uint16_t *lab, int a, int b) {
    for (;;) {
        a = uf_find(lab, a);
        b = uf_find(lab, b);
        if (a == b) return;
        if (a < b) { const int t = a; a = b; b = t; }
        const unsigned short old = atomicCAS((unsigned short *)&lab[a], (unsigned short)a, (unsigned short)b);
        if (old == (unsigned short)a) return;
        a = old;                                          // a was linked meanwhile: go on from its new parent
    }
}

__global__ void __launch_bounds__(kClusterThreads) k_ising_swendsen_wang(const ClusterArgs A) {
    extern __shared__ uint32_t s_mem[];
    const int L = A.L, N = L * L, nwords = (N + 31) >> 5, nunits = (N + 7) >> 3;
    uint32_t *s_spin = s_mem;                                         // [nwords] bit i & 31 of word i >> 5 = site i
    uint8_t *s_spin8 = reinterpret_cast<uint8_t *>(s_mem);            // byte u = sites 8u .. 8u + 7
    uint8_t *s_flip8 = reinterpret_cast<uint8_t *>(s_mem + nwords);   // [nunits] flip bit of each root
    volatile uint16_t *lab = reinterpret_cast<volatile uint16_t *>(s_mem + 2 * nwords);   // [N]
    __shared__ int s_aligned, s_nup;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, nthr = blockDim.x;
    const uint2 key = make_uint2(A.seed, A.lattice_base + (uint32_t)b);

    if (tid == 0) { s_aligned = 0; s_nup = 0; }
    const int8_t *in = A.spins + (size_t)b * N;
    for (int u = tid; u < nunits; u += nthr) {                       // a thread packs its 8-site units
        uint32_t byte = 0u;
        for (int j = 0; j < 8 && u * 8 + j < N; j++) byte |= (in[u * 8 + j] != 0 ? 1u : 0u) << j;
        s_spin8[u] = (uint8_t)byte;
    }
    for (int i = tid; i < N; i += nthr) lab[i] = (uint16_t)i;
    __syncthreads();

    auto spin = [&](int i) { return (s_spin[i >> 5] >> (i & 31)) & 1u; };
    for (int k = 0; k <= A.K; k++) {
        // bonds of the current spins (those after sweep k - 1): count the aligned ones; in a sweep, union the active
        const bool draw = k < A.K;
        const uint32_t thr = draw ? A.thr[(size_t)k * A.B + b] : 0u;
        const uint32_t step = A.step0 + (uint32_t)k;
        int aligned = 0;
        for (int u = tid; u < nunits; u += nthr) {
            const int i0 = u * 8;
            int x = i0 % L;
#pragma unroll
            for (int q = 0; q < 4; q++) {                             // pair 4u + q: sites i0 + 2q, i0 + 2q + 1
                if (i0 + 2 * q >= N) break;
                uint4 r = make_uint4(0u, 0u, 0u, 0u);
                if (draw && thr != 0u)
                    r = philox4x32_10(make_uint4((uint32_t)(4 * u + q), step, 0u, kClusterTag), key);
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    const int i = i0 + 2 * q + h;
                    if (i >= N) break;
                    const int rt = x == L - 1 ? i + 1 - L : i + 1, dn = i + L >= N ? i + L - N : i + L;
                    const uint32_t si = spin(i);
                    const bool ar = si == spin(rt), ad = si == spin(dn);
                    aligned += (int)ar + (int)ad;
                    if (ar && (h ? r.z : r.x) < thr) uf_union(lab, i, rt);
                    if (ad && (h ? r.w : r.y) < thr) uf_union(lab, i, dn);
                    x = x == L - 1 ? 0 : x + 1;
                }
            }
        }
        aligned = __reduce_add_sync(0xFFFFFFFFu, aligned);
        if (lane == 0 && aligned) atomicAdd(&s_aligned, aligned);
        __syncthreads();
        // thread 0 reads and clears the count before the next barrier; the next adds come two barriers later
        if (tid == 0) {
            if (k > 0 && A.bond_sum) A.bond_sum[(size_t)(k - 1) * A.B + b] = 2 * s_aligned - 2 * N;
            s_aligned = 0;
        }
        if (!draw) break;

        // every site stores its root; the flip bits of the roots
        for (int u = tid; u < nunits; u += nthr) {
            const int i0 = u * 8;
            uint32_t fl = 0u;
#pragma unroll
            for (int g = 0; g < 2; g++) {                              // group 2u + g: sites i0 + 4g .. i0 + 4g + 3
                uint32_t roots = 0u;
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const int i = i0 + 4 * g + j;
                    if (i >= N) break;
                    const int r = uf_root(lab, i);
                    lab[i] = (uint16_t)r;
                    roots |= (r == i ? 1u : 0u) << j;
                }
                if (roots == 0u) continue;
                const uint4 r = philox4x32_10(make_uint4((uint32_t)(2 * u + g), step, 1u, kClusterTag), key);
                const uint32_t top = (r.x >> 31) | ((r.y >> 31) << 1) | ((r.z >> 31) << 2) | ((r.w >> 31) << 3);
                fl |= (top & roots) << (4 * g);
            }
            s_flip8[u] = (uint8_t)fl;
        }
        __syncthreads();

        // flip every site with its root; reset the labels for the next sweep (a thread reads only its own sites' labels)
        int nup = 0;
        for (int u = tid; u < nunits; u += nthr) {
            const int i0 = u * 8;
            uint32_t f = 0u;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int i = i0 + j;
                if (i >= N) break;
                const int r = lab[i];
                f |= ((uint32_t)(s_flip8[r >> 3] >> (r & 7)) & 1u) << j;
                lab[i] = (uint16_t)i;
            }
            const uint32_t nb = (uint32_t)s_spin8[u] ^ f;
            s_spin8[u] = (uint8_t)nb;
            nup += __popc(nb);
        }
        nup = __reduce_add_sync(0xFFFFFFFFu, nup);
        if (lane == 0 && nup) atomicAdd(&s_nup, nup);
        __syncthreads();
        if (tid == 0) {                                                // the next adds come two barriers later
            if (A.n_up) A.n_up[(size_t)k * A.B + b] = s_nup;
            s_nup = 0;
        }
    }
    int8_t *out = A.spins + (size_t)b * N;
    for (int u = tid; u < nunits; u += nthr) {
        const uint32_t byte = s_spin8[u];
        for (int j = 0; j < 8 && u * 8 + j < N; j++) out[u * 8 + j] = (int8_t)((byte >> j) & 1u);
    }
}

}  // namespace mfmarl

using namespace mfmarl;

extern "C" int mfi_swendsen_wang(int n_lattices, int side, int n_sweeps, int8_t *d_spins, const double *h_temperatures,
                                 unsigned seed, unsigned lattice_base, unsigned step0, int32_t *d_n_up,
                                 int32_t *d_bond_sum, void *stream) {
    try {
        if (n_lattices < 1 || n_sweeps < 1) throw Fatal("need at least one lattice and one sweep");
        if (side < 2 || side > kClusterMaxSide)
            throw Fatal("side must be in [2, 256] (the uint16 labels of a 256 x 256 lattice fill the shared memory), got " +
                        std::to_string(side));
        if (!d_spins || !h_temperatures) throw Fatal("null spins or temperatures");
        const size_t n = (size_t)n_sweeps * n_lattices;
        std::vector<uint32_t> thr(n);
        double last_T = 0.0;                          // neighbouring entries mostly repeat a temperature
        for (size_t i = 0; i < n; i++) {
            const double T = h_temperatures[i];
            if (!(T > 0.0) || !std::isfinite(T))
                throw Fatal("temperature " + std::to_string(T) + " at index " + std::to_string(i) + " is not finite and > 0");
            if (i > 0 && T == last_T) { thr[i] = thr[i - 1]; continue; }
            const double t = std::floor((1.0 - std::exp(-1.0 / T)) * 4294967296.0);
            thr[i] = t >= 4294967295.0 ? 0xFFFFFFFFu : (uint32_t)t;
            last_T = T;
        }
        const int N = side * side, nwords = (N + 31) / 32, nunits = (N + 7) / 8;
        const size_t smem = (size_t)nwords * 8 + (size_t)N * sizeof(uint16_t);
        const int threads = std::min(kClusterThreads, (nunits + 31) / 32 * 32);
        if (smem > 48 * 1024)
            MF_CUDA(cudaFuncSetAttribute(k_ising_swendsen_wang, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cudaStream_t st = (cudaStream_t)stream;
        uint32_t *d_thr = nullptr;
        MF_CUDA(cudaMallocAsync((void **)&d_thr, thr.size() * sizeof(uint32_t), st));
        MF_CUDA(cudaMemcpyAsync(d_thr, thr.data(), thr.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        const ClusterArgs A{n_lattices, side, n_sweeps, d_spins, d_thr, seed, lattice_base, step0, d_n_up, d_bond_sum};
        k_ising_swendsen_wang<<<n_lattices, threads, smem, st>>>(A);
        const cudaError_t err = cudaGetLastError();
        MF_CUDA(cudaFreeAsync(d_thr, st));
        MF_CUDA(err);
    } catch (const std::exception &ex) {
        set_last_error(std::string("mfi_swendsen_wang: ") + ex.what());
        return -1;
    }
    return 0;
}
