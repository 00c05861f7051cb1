// Gather kernel of the device-resident result fetches (abg_fetch_batches_device, abg_fetch_all_device,
// abg_fetch_mixer_batches_device).  The result slots are channel-major ([G][nbmax*B] audio, [G][nbmax*B] I/Q,
// [nbmax][Gp] flags, [nbmax][n_mixers][2][B] mixer sums); callers want batch-major buffers ([n][C][B] ...).  The engine
// turns one fetch into a list of rectangular blocks and this kernel copies all of them in one launch: grid.y walks the
// blocks, grid.x the rows of a block, the threads of a CTA one row, 16 bytes per access when every address and pitch of
// the block allows it (audio rows of WAVE_BATCH floats do for WAVE_BATCH % 4 == 0), 4 or 1 bytes otherwise.
#include "abg_internal.h"

namespace {

template <typename T>
__device__ __forceinline__ void copy_row(const unsigned char* src, unsigned char* dst, int row_bytes) {
    const int n = row_bytes / (int)sizeof(T);
    T* d = reinterpret_cast<T*>(dst);
    if (src) {
        const T* s = reinterpret_cast<const T*>(src);
        for (int k = threadIdx.x; k < n; k += blockDim.x) d[k] = s[k];
    } else {
        T z;
        memset(&z, 0, sizeof(z));
        for (int k = threadIdx.x; k < n; k += blockDim.x) d[k] = z;
    }
}

__global__ void __launch_bounds__(256) abg_gather_results_kernel(const GatherList L) {
    const GatherCopy c = L.c[blockIdx.y];
    const unsigned long long align = reinterpret_cast<uintptr_t>(c.src) | reinterpret_cast<uintptr_t>(c.dst) |
                                     (unsigned long long)c.src_pitch | (unsigned long long)c.dst_pitch | (unsigned long long)c.row_bytes;
    for (int r = blockIdx.x; r < c.rows; r += gridDim.x) {
        const unsigned char* s = c.src ? c.src + (size_t)r * c.src_pitch : nullptr;
        unsigned char* d = c.dst + (size_t)r * c.dst_pitch;
        if ((align & 15) == 0)
            copy_row<uint4>(s, d, c.row_bytes);
        else if ((align & 3) == 0)
            copy_row<uint32_t>(s, d, c.row_bytes);
        else
            copy_row<unsigned char>(s, d, c.row_bytes);
    }
}

}  // namespace

cudaError_t abg_launch_gather(const GatherList& L, cudaStream_t s) {
    if (L.n <= 0) return cudaSuccess;
    // enough CTAs along x to keep every SM busy on a large block (one audio row per CTA iteration); small blocks (flags)
    // leave most of their CTAs idle, which costs one early exit each
    const int gx = L.max_rows < 1 ? 1 : (L.max_rows < 1024 ? L.max_rows : 1024);
    abg_gather_results_kernel<<<dim3(gx, L.n, 1), 256, 0, s>>>(L);
    return cudaGetLastError();
}
