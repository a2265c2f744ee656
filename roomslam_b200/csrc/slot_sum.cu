// The reduction that closes every split reduction in deterministic mode (common.cuh): per-split partials, stored by the
// CTAs of the split kernel into their own workspace slots, are added onto the output in ascending slot order.  One thread
// per output element, so the order of the additions is fixed whatever the grid.
#include "common.cuh"

namespace {

template <typename T>
struct SlotSums {
    rs::SlotSum<T> job[rs::kMaxSlotSums];
};

template <typename T>
__global__ void __launch_bounds__(256) slot_sum_kernel(const SlotSums<T> js, int n_parts, long long part_stride, int accumulate) {
    const rs::SlotSum<T>& j = js.job[blockIdx.y];
    const long long n = (long long)j.rows * j.cols;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        T* o = j.out + (e / j.cols) * j.ldo + e % j.cols;
        const T* src = j.parts + e;
        T v = accumulate ? *o : T(0);
        int s = 0;
        for (; s + 8 <= n_parts; s += 8) {     // eight loads in flight, added in slot order
            T t[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) t[k] = src[(s + k) * part_stride];
#pragma unroll
            for (int k = 0; k < 8; ++k) v += t[k];
        }
        for (; s < n_parts; ++s) v += src[s * part_stride];
        *o = v;
    }
}

// Do two outputs share an element?  Exact for equal leading dimensions (column blocks of one matrix), else by address range.
template <typename T>
bool overlap(const rs::SlotSum<T>& a, const rs::SlotSum<T>& b) {
    const long long d = b.out - a.out;
    if (d < 0) return overlap(b, a);
    if (a.ldo == b.ldo && a.cols <= a.ldo && b.cols <= b.ldo) {
        const long long q = d / a.ldo, m = d % a.ldo;         // b starts in row q, column m of a
        return (q < a.rows && m < a.cols) || (m + b.cols > a.ldo && q + 1 < a.rows);
    }
    return d < (a.rows - 1) * a.ldo + a.cols;
}

}  // namespace

namespace rs {

template <typename T>
int slot_sum(const SlotSum<T>* jobs, int n_jobs, int n_parts, long long part_stride, bool accumulate, cudaStream_t stream) {
    RS_REQUIRE(n_jobs >= 1 && n_jobs <= kMaxSlotSums && n_parts >= 1, "slot_sum: %d outputs, %d slots", n_jobs, n_parts);
    // outputs that overlap (callers may accumulate several tiles into the same elements) are summed one launch after another
    for (int i = 0; i < n_jobs; ++i)
        for (int k = i + 1; k < n_jobs; ++k) {
            if (overlap(jobs[i], jobs[k])) {
                for (int j = 0; j < n_jobs; ++j)
                    if (int rc = slot_sum(&jobs[j], 1, n_parts, part_stride, accumulate, stream)) return rc;
                return 0;
            }
        }
    SlotSums<T> js = {};
    long long most = 0;
    for (int i = 0; i < n_jobs; ++i) {
        js.job[i] = jobs[i];
        const long long n = (long long)jobs[i].rows * jobs[i].cols;
        if (n > most) most = n;
    }
    long long bx = (most + 255) / 256;
    if (bx > 1024) bx = 1024;
    if (bx < 1) bx = 1;
    slot_sum_kernel<T><<<dim3((unsigned)bx, n_jobs), 256, 0, stream>>>(js, n_parts, part_stride, accumulate ? 1 : 0);
    count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

template int slot_sum<float>(const SlotSum<float>*, int, int, long long, bool, cudaStream_t);
template int slot_sum<double>(const SlotSum<double>*, int, int, long long, bool, cudaStream_t);

}  // namespace rs
