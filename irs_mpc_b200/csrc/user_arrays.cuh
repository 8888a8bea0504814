// Read-only views of the arrays of a user-written system (user_system.py: CudaSourceDynamics(arrays=...)).
// Included only by the generated unit of a system that has arrays.  The values live in device memory, in an
// array set registered with irs_user_arrays_register (api.cu); load_params puts the set's fp64 and fp32 base
// pointers into SysParams, and UserSystem<R> points one view per array into the copy in R.  Elements are
// returned by value, so a body cannot write to an array; loads take the read-only data path (LDG.CONSTANT).
#pragma once
#include "common.cuh"

namespace irs {

template <typename T>
__device__ __forceinline__ const T* user_arrays(const SysParams& sp) {
    if constexpr (std::is_same<T, float>::value) return sp.arrays32;
    else return sp.arrays64;
}

// RANK dimensions of extents N0 x N1 x N2 (the missing ones 1), row-major: a[i] flat, a(i, j), a(i, j, k)
template <typename T, int RANK, int N0, int N1, int N2>
struct ArrayView {
    const T* __restrict__ data;
    __device__ __forceinline__ T operator[](int i) const { return __ldg(data + i); }
    template <int Q = RANK>
    __device__ __forceinline__ T operator()(int i, int j) const {
        static_assert(Q == 2, "a(i, j) indexes a two-dimensional array");
        return __ldg(data + i * N1 + j);
    }
    template <int Q = RANK>
    __device__ __forceinline__ T operator()(int i, int j, int k) const {
        static_assert(Q == 3, "a(i, j, k) indexes a three-dimensional array");
        return __ldg(data + (i * N1 + j) * N2 + k);
    }
};

}  // namespace irs
