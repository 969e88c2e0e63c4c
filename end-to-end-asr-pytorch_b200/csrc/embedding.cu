// K17: token embedding (nn.Embedding without padding_idx, src/lm.py:17 of the reference) forward and weight gradient.
//   forward   out[n, :] = W[ids[n], :]                       row gather, 16-byte vector loads when E % 4 == 0
//   backward  dW[v, :] (=|+=) sum over {n : ids[n] == v} of dY[n, :]
// The backward takes the ids already sorted (stable, so equal ids keep ascending position) together with the sort
// permutation.  One block per run of equal ids sums its rows in ascending sorted position with no atomics, so two
// runs give bit-identical gradients.  Id 0 is an ordinary row.  Ids outside [0, V) are never dereferenced: the
// forward writes a zero row for them and the backward skips them (the autograd wrapper rejects them beforehand).
#include <algorithm>

#include "common.cuh"
#include "../../include/b200asr.h"

namespace b200asr {

template <int VEC>
struct Vec;
template <>
struct Vec<4> {
    using T = float4;
    __device__ static T zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
    __device__ static void add(T& a, const T& b) { a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w; }
};
template <>
struct Vec<1> {
    using T = float;
    __device__ static T zero() { return 0.f; }
    __device__ static void add(T& a, const T& b) { a += b; }
};

template <int VEC>
__global__ void __launch_bounds__(256) embedding_fwd_kernel(const long long* __restrict__ ids, long long N,
                                                           const float* __restrict__ W, long long V, int E,
                                                           float* __restrict__ out) {
    using T = typename Vec<VEC>::T;
    const int ev = E / VEC;
    const long long total = N * ev;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long n = i / ev;
        const int c = (int)(i - n * ev);
        const long long id = __ldg(ids + n);
        T v = Vec<VEC>::zero();
        if (id >= 0 && id < V) v = __ldg(reinterpret_cast<const T*>(W + id * E) + c);
        reinterpret_cast<T*>(out + n * E)[c] = v;
    }
}

constexpr int EMB_BWD_THREADS = 128;

// grid (N, ceil(E / (VEC * 128))): block x = a sorted position; only the first position of each run of equal ids
// works.  The run is walked in chunks of 128 positions staged in shared memory, so the row loads of one chunk are
// independent of each other and of the run-length test.
template <int VEC>
__global__ void __launch_bounds__(EMB_BWD_THREADS) embedding_bwd_kernel(const long long* __restrict__ sorted_ids,
                                                                       const long long* __restrict__ order, long long N,
                                                                       const float* __restrict__ dY, long long V, int E,
                                                                       float* __restrict__ dW, int accumulate) {
    using T = typename Vec<VEC>::T;
    __shared__ long long rows[EMB_BWD_THREADS];
    const long long start = blockIdx.x;
    const long long id = sorted_ids[start];
    if (id < 0 || id >= V) return;
    if (start > 0 && sorted_ids[start - 1] == id) return;
    const int c = blockIdx.y * EMB_BWD_THREADS + threadIdx.x;       // vector column
    const bool active = c < E / VEC;
    T acc = Vec<VEC>::zero();
    for (long long base = start; base < N; base += EMB_BWD_THREADS) {
        const long long p = base + threadIdx.x;
        const bool same = p < N && sorted_ids[p] == id;
        if (same) rows[threadIdx.x] = order[p];
        // sorted: the positions of this run form a prefix of the chunk
        const int cnt = __syncthreads_count(same);
        if (active) {
#pragma unroll 4
            for (int j = 0; j < cnt; ++j) Vec<VEC>::add(acc, __ldg(reinterpret_cast<const T*>(dY + rows[j] * E) + c));
        }
        __syncthreads();
        if (cnt < EMB_BWD_THREADS) break;
    }
    if (!active) return;
    T* dst = reinterpret_cast<T*>(dW + id * E) + c;
    if (accumulate) {
        T old = *dst;
        Vec<VEC>::add(old, acc);
        *dst = old;
    } else {
        *dst = acc;
    }
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace b200asr

using namespace b200asr;

extern "C" int b200asr_embedding_fwd(const long long* ids, long long N, const float* W, long long V, int E, float* out,
                                     b200asr_stream stream) {
    B200_REQUIRE(N >= 0 && V > 0 && E > 0, "embedding_fwd: bad sizes (N=%lld V=%lld E=%d)", N, V, E);
    if (N == 0) return B200_OK;
    B200_REQUIRE(ids && W && out, "embedding_fwd: null pointer");
    const bool vec = E % 4 == 0 && aligned16(W) && aligned16(out);
    const long long work = N * (vec ? E / 4 : E);
    const int threads = 256;
    const long long blocks = std::min<long long>((work + threads - 1) / threads, (long long)sm_count() * 16);
    if (vec)
        embedding_fwd_kernel<4><<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(ids, N, W, V, E, out);
    else
        embedding_fwd_kernel<1><<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(ids, N, W, V, E, out);
    B200_LAUNCH_CHECK("embedding_fwd_kernel");
    return B200_OK;
}

extern "C" int b200asr_embedding_bwd(const long long* sorted_ids, const long long* order, long long N, const float* dY,
                                     long long V, int E, float* dW, int accumulate, b200asr_stream stream) {
    B200_REQUIRE(N >= 0 && V > 0 && E > 0, "embedding_bwd: bad sizes (N=%lld V=%lld E=%d)", N, V, E);
    B200_REQUIRE(N < (1LL << 31), "embedding_bwd: N=%lld exceeds the grid limit", N);
    B200_REQUIRE(dW, "embedding_bwd: null dW");
    cudaStream_t s = (cudaStream_t)stream;
    if (!accumulate) B200_CUDA(cudaMemsetAsync(dW, 0, (size_t)V * E * sizeof(float), s));   // rows that get no id
    if (N == 0) return B200_OK;
    B200_REQUIRE(sorted_ids && order && dY, "embedding_bwd: null pointer");
    const bool vec = E % 4 == 0 && aligned16(dY) && aligned16(dW);
    const int cols = vec ? E / 4 : E;
    dim3 grid((unsigned)N, (unsigned)((cols + EMB_BWD_THREADS - 1) / EMB_BWD_THREADS));
    if (vec)
        embedding_bwd_kernel<4><<<grid, EMB_BWD_THREADS, 0, s>>>(sorted_ids, order, N, dY, V, E, dW, accumulate);
    else
        embedding_bwd_kernel<1><<<grid, EMB_BWD_THREADS, 0, s>>>(sorted_ids, order, N, dY, V, E, dW, accumulate);
    B200_LAUNCH_CHECK("embedding_bwd_kernel");
    return B200_OK;
}
