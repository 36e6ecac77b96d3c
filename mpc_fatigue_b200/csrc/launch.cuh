// launch.cuh — model policies, kernel wrappers and family dispatch shared by the kernels_*.cu files.
// sm_100a kernels of the batched dynamics + fatigue evaluator.
//
// Mapping: one thread per (scenario, node) unit; lanes of a warp hold 32 consecutive units so every
// global access to the SoA planes `[component][U]` is a fully coalesced 256-byte warp transaction.
// The Jacobian kernel adds the seed direction as blockIdx.y (warp-uniform), each thread carrying one
// forward-mode tangent in registers next to the primal.  FP64 pipe bound (SURVEY.md §8d); tensor cores
// are not applicable (6x6 spatial algebra per link, no dense contraction).
#pragma once
#include "kernels.cuh"

#include <atomic>
#include <type_traits>

#include "dyn.cuh"

namespace mpcf {

extern std::atomic<long> g_launches;

// ---------------------------------------------------------------------------------------------
// model policies
// ---------------------------------------------------------------------------------------------
template <int N, int L>
struct StaticModel {
    static constexpr int MAXN = N;
    static constexpr bool kStatic = true;
    static constexpr int kChain = L;  // length of each serial chain of the forest
    const StaticParams<N> &P;
    MPCF_DI int n() const { return N; }
    MPCF_DI int parent(int i) const { return (i % L == 0) ? -1 : i - 1; }
    MPCF_DI bool prismatic(int) const { return false; }
    MPCF_DI bool keep(int) const { return true; }
    MPCF_DI double Rp(int i, int k) const { return P.Rp[i][k]; }
    MPCF_DI double pp(int i, int k) const { return P.pp[i][k]; }
    MPCF_DI double mass(int i) const { return P.mass[i]; }
    MPCF_DI double mc(int i, int k) const { return P.mc[i][k]; }
    MPCF_DI double Io(int i, int k) const { return P.Io[i][k]; }
    MPCF_DI double arm(int i) const { return P.arm[i]; }
    MPCF_DI double fat(int i, int k) const { return P.fat[i][k]; }
    MPCF_DI double grav(int k) const { return P.grav[k]; }
    // Scheduling fence for fully unrolled link loops: `if (m.skip(i)) continue;` is never taken (fence0 == 0) but the
    // compiler cannot know, so every link's work stays in its own basic block and ptxas does not hoist later links' loads
    // and arithmetic over earlier ones (which multiplies the live registers: k_stage_derivs' stack frame 2.7 KB -> 0.1 KB).
    MPCF_DI bool skip(int i) const { return P.fence0 > i; }
};

template <int MAXN_>
struct GenericModel {
    static constexpr int MAXN = MAXN_;
    static constexpr bool kStatic = false;
    static constexpr int kChain = 0;
    int n_;
    const double *d;  // shared memory
    const int *ii;    // shared memory
    MPCF_HD int n() const { return n_; }
    MPCF_HD int parent(int i) const { return ii[i]; }
    MPCF_HD bool prismatic(int i) const { return ii[n_ + i] != 0; }
    MPCF_HD bool keep(int i) const { return ii[2 * n_ + i] != 0; }
    // depth of link i (roots: 0) and the offset of its row in the packed ancestor storage of the tree pipeline: entry (i, j), j an
    // ancestor of i or i itself, lives at rowptr(i) + depth(j)
    MPCF_HD int depth(int i) const { return ii[3 * n_ + i]; }
    MPCF_HD int rowptr(int i) const { return ii[4 * n_ + i]; }
    MPCF_HD double Rp(int i, int k) const { return d[9 * i + k]; }
    MPCF_HD double pp(int i, int k) const { return d[9 * n_ + 3 * i + k]; }
    MPCF_HD double mass(int i) const { return d[12 * n_ + i]; }
    MPCF_HD double mc(int i, int k) const { return d[13 * n_ + 3 * i + k]; }
    MPCF_HD double Io(int i, int k) const { return d[16 * n_ + 6 * i + k]; }
    MPCF_HD double arm(int i) const { return d[22 * n_ + i]; }
    MPCF_HD double fat(int i, int k) const { return d[23 * n_ + 4 * i + k]; }
    MPCF_HD double grav(int k) const { return d[27 * n_ + k]; }
    MPCF_HD bool skip(int) const { return false; }
};

// ---------------------------------------------------------------------------------------------
// kernel wrappers: Body::run<MP>(model, u, U, args...)
// ---------------------------------------------------------------------------------------------
constexpr int kThreads = 128;

template <int N, int L, class Body, class... Args>
__global__ void __launch_bounds__(kThreads) static_kernel(const __grid_constant__ StaticParams<N> P, long U, Args... args)
{
    const StaticModel<N, L> m{P};
    const long u = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (u < U) Body::run(m, u, U, args...);
}

// A body may ask for a register budget that lets several blocks of the run-time-topology kernel share an SM
// (`static constexpr int kGenericMinBlocks = 3;`): those kernels are latency bound, and for the ABA-based bodies twelve
// warps per SM with a few spills beat eight without (measured on the 37-joint tree: RK4 step 11.7 -> 9.4 ms).
template <class Body, class = void>
struct GenericMinBlocks {
    static constexpr int value = 0;  // 0 = no minimum (same as the one-argument __launch_bounds__)
};
template <class Body>
struct GenericMinBlocks<Body, decltype((void)Body::kGenericMinBlocks)> {
    static constexpr int value = Body::kGenericMinBlocks;
};

template <int MAXN, class Body, class... Args>
__global__ void __launch_bounds__(kThreads, GenericMinBlocks<Body>::value) generic_kernel(GenericBlob blob, long U, Args... args)
{
    extern __shared__ double smem[];
    const int n = blob.n;
    const int nd = 27 * n + 3;
    int *si = reinterpret_cast<int *>(smem + nd);
    for (int k = threadIdx.x; k < nd; k += blockDim.x) smem[k] = blob.dbl[k];
    for (int k = threadIdx.x; k < blob_ints(n); k += blockDim.x) si[k] = blob.ints[k];
    __syncthreads();
    const GenericModel<MAXN> m{n, smem, si};
    const long u = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (u < U) Body::run(m, u, U, args...);
}

// Bodies that only the run-time-topology families use (the static families have dedicated kernels for the same entry):
// no static_kernel instantiations, so they cost neither compile time nor binary size.
template <class Body, class... Args>
static cudaError_t dispatch_generic(const LaunchModel &m, long U, int grid_y, cudaStream_t s, Args... args)
{
    if (U <= 0) return cudaSuccess;
    dim3 grid((unsigned)((U + kThreads - 1) / kThreads), (unsigned)grid_y), block(kThreads);
    if (m.fam == FAM_GENERIC16) generic_kernel<16, Body, Args...><<<grid, block, blob_smem_bytes(m.n), s>>>(m.blob, U, args...);
    else if (m.fam == FAM_GENERIC64) generic_kernel<MPCF_MAX_DOF, Body, Args...><<<grid, block, blob_smem_bytes(m.n), s>>>(m.blob, U, args...);
    else return cudaErrorInvalidValue;
    g_launches.fetch_add(1);
    return cudaGetLastError();
}

template <class Body, class... Args>
static cudaError_t dispatch(const LaunchModel &m, long U, int grid_y, cudaStream_t s, Args... args)
{
    if (U <= 0) return cudaSuccess;
    dim3 grid((unsigned)((U + kThreads - 1) / kThreads), (unsigned)grid_y), block(kThreads);
    switch (m.fam) {
    case FAM_CHAIN3:
        static_kernel<3, 3, Body, Args...><<<grid, block, 0, s>>>(*static_cast<const StaticParams<3> *>(m.static_params), U, args...);
        break;
    case FAM_CHAIN6:
        static_kernel<6, 6, Body, Args...><<<grid, block, 0, s>>>(*static_cast<const StaticParams<6> *>(m.static_params), U, args...);
        break;
    case FAM_FOREST12x6:
        static_kernel<12, 6, Body, Args...><<<grid, block, 0, s>>>(*static_cast<const StaticParams<12> *>(m.static_params), U, args...);
        break;
    case FAM_CHAIN7:
        static_kernel<7, 7, Body, Args...><<<grid, block, 0, s>>>(*static_cast<const StaticParams<7> *>(m.static_params), U, args...);
        break;
    case FAM_FOREST14x7:
        static_kernel<14, 7, Body, Args...><<<grid, block, 0, s>>>(*static_cast<const StaticParams<14> *>(m.static_params), U, args...);
        break;
    case FAM_GENERIC16:
        generic_kernel<16, Body, Args...><<<grid, block, blob_smem_bytes(m.n), s>>>(m.blob, U, args...);
        break;
    default:
        generic_kernel<MPCF_MAX_DOF, Body, Args...><<<grid, block, blob_smem_bytes(m.n), s>>>(m.blob, U, args...);
        break;
    }
    g_launches.fetch_add(1);
    return cudaGetLastError();
}

// Static families run their dedicated kernels once per serial chain: f(L, chains, nchains) with the chain length L and the chain
// count as std::integral_constant (so forest-only kernels are instantiated for the forests alone) and chains = the parameter blocks
// of the m.n / L chains, chain c owning joints [c L, (c + 1) L).  Returns false without calling f for run-time-topology families.
template <class F>
static bool with_chains(const LaunchModel &m, F &&f)
{
    using std::integral_constant;
    const void *p = m.chain_params;
    switch (m.fam) {
    case FAM_CHAIN3: f(integral_constant<int, 3>{}, static_cast<const StaticParams<3> *>(p), integral_constant<int, 1>{}); return true;
    case FAM_CHAIN6: f(integral_constant<int, 6>{}, static_cast<const StaticParams<6> *>(p), integral_constant<int, 1>{}); return true;
    case FAM_FOREST12x6: f(integral_constant<int, 6>{}, static_cast<const StaticParams<6> *>(p), integral_constant<int, 2>{}); return true;
    case FAM_CHAIN7: f(integral_constant<int, 7>{}, static_cast<const StaticParams<7> *>(p), integral_constant<int, 1>{}); return true;
    case FAM_FOREST14x7: f(integral_constant<int, 7>{}, static_cast<const StaticParams<7> *>(p), integral_constant<int, 2>{}); return true;
    default: return false;
    }
}

// Raises Kernel's dynamic shared-memory limit to `bytes` once per device (function attributes are per device).  Every call site of
// a kernel asks for the same limit, so threads racing through the first call set the same value.
template <auto Kernel>
static cudaError_t raise_smem_limit(int bytes)
{
    static std::atomic<bool> done[64];
    int dev = 0;
    cudaGetDevice(&dev);
    const bool cached = dev >= 0 && dev < 64;
    if (cached && done[dev].load(std::memory_order_acquire)) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess && cached) done[dev].store(true, std::memory_order_release);
    return e;
}

}  // namespace mpcf
