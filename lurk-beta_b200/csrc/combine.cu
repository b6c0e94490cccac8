// N4 -- PolyEvalWitness::batch_diff_size (Arecibo spartan/mod.rs, the joint polynomial of batch_eval_reduce): the random linear
// combination of polynomials of different lengths, each zero-extended at the end to the output length,
//     out[i] = sum_{j : i < len_j} c_j P_j[i]      (i < out_len; zero where no P_j reaches).
// It turns the 2k evaluation claims of a (batched) Spartan proof into one polynomial, so each circuit of the cycle needs one PCS
// opening instead of 2k.
//
// One launch over out_len, grid-stride, 256-thread CTAs.  The pointer / length table and the Montgomery coefficients (up to 120
// polynomials = 2 x the batched sum-check's 60 instances, 5.8 KB) travel as a __grid_constant__ argument; the host sorts them by
// length, longest first, so element i walks a prefix of the table and stops at the first polynomial that does not reach it.
// 128-bit loads / stores of 32-byte elements.  HBM-bound: 32 (sum_j len_j + out_len) bytes for sum_j len_j products.
#include "common.cuh"
#include "sc_scratch.cuh"

#include <algorithm>
#include <numeric>
#include <vector>

namespace lurk {

constexpr int COMBINE_MAX_POLYS = 120;

template <class F>
struct CombineArgs {
    const F *poly[COMBINE_MAX_POLYS];
    size_t len[COMBINE_MAX_POLYS];     // non-increasing
    F coeff[COMBINE_MAX_POLYS];        // Montgomery
    int n;
};

template <class F>
__global__ void __launch_bounds__(256) poly_combine_kernel(const __grid_constant__ CombineArgs<F> a, F *__restrict__ out, size_t out_len) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < out_len; i += (size_t)gridDim.x * blockDim.x) {
        F acc = F::zero();
        for (int j = 0; j < a.n && i < a.len[j]; j++) acc += a.coeff[j] * load_fe<F>(a.poly[j] + i);
        store_fe(out + i, acc);
    }
}

template <class F>
static int poly_combine(int n, const void *const *d_polys, const size_t *lens, const uint8_t *coeffs, void *d_out, size_t out_len, int fmt,
                        cudaStream_t s) {
    CombineArgs<F> a;
    memset(&a, 0, sizeof a);
    std::vector<int> order(n);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return lens[x] > lens[y]; });
    for (int t = 0; t < n; t++) {
        const int j = order[t];
        if (!fe_in(coeffs + 32 * j, fmt, a.coeff[t])) { set_error("coefficient %d is not reduced", j); return LURK_ERR_RANGE; }
        a.poly[t] = static_cast<const F *>(d_polys[j]);
        a.len[t] = lens[j];
    }
    a.n = n;
    LURK_TRY(require_gpu());
    if (out_len == 0) return LURK_OK;
    poly_combine_kernel<F><<<sc_grid(out_len, 256), 256, 0, s>>>(a, static_cast<F *>(d_out), out_len);
    LURK_CUDA_TRY(cudaGetLastError());
    return LURK_OK;
}

}  // namespace lurk

using namespace lurk;

extern "C" {

int lurk_poly_combine_dev(int field_id, int n_polys, const void *const *d_polys, const size_t *lens, const uint8_t *coeffs, void *d_out,
                          size_t out_len, int fmt, void *stream) {
    if (n_polys < 1 || n_polys > COMBINE_MAX_POLYS) { set_error("1..%d polynomials, got %d", COMBINE_MAX_POLYS, n_polys); return LURK_ERR_ARG; }
    if (!d_polys || !lens || !coeffs || !d_out) { set_error("null argument"); return LURK_ERR_ARG; }
    if (fmt != LURK_FMT_CANONICAL && fmt != LURK_FMT_MONTGOMERY) { set_error("bad format %d", fmt); return LURK_ERR_ARG; }
    const uintptr_t o0 = reinterpret_cast<uintptr_t>(d_out), o1 = o0 + 32 * out_len;
    for (int j = 0; j < n_polys; j++) {
        if (lens[j] > out_len) { set_error("polynomial %d has %zu elements, more than the output's %zu", j, lens[j], out_len); return LURK_ERR_ARG; }
        if (!d_polys[j]) { set_error("polynomial %d is null", j); return LURK_ERR_ARG; }
        const uintptr_t p0 = reinterpret_cast<uintptr_t>(d_polys[j]), p1 = p0 + 32 * lens[j];
        if (p0 < o1 && o0 < p1) { set_error("polynomial %d overlaps the output", j); return LURK_ERR_ARG; }
    }
    return dispatch_field(field_id, [&](auto f) {
        return poly_combine<decltype(f)>(n_polys, d_polys, lens, coeffs, d_out, out_len, fmt, static_cast<cudaStream_t>(stream));
    });
}

}  // extern "C"
