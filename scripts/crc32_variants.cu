// crc32_variants.cu -- MEASUREMENT AID for scripts/bench_crc32.py: crc32_blocks_kernel's body (redux_crc.cuh) in
// other shapes -- replicas of the tables, threads per CTA, CTAs per SM, vectors loaded one trip ahead, two chains per
// lane -- so that the
// library's shape (CrcLib) is chosen by timing them against each other on the same bytes (DESIGN.md 3.11).
// bench_crc32.py compiles this file into a temporary directory with nvcc and loads it through ctypes; it is not part
// of the library.
#include <cuda_runtime.h>

#include <algorithm>

#include "../redux_b200/csrc/redux_crc.cuh"

using namespace rdx;

// name, replicas, threads, CTAs per SM, prefetch, two chains per lane
#define RDX_CRC_VARIANTS(X)                                                                                            \
    X(0, "r32_t1024_b1", 32, 1024, 1, false, false)                                                                    \
    X(1, "r32_t1024_b1_prefetch", 32, 1024, 1, true, false)                                                            \
    X(2, "r16_t1024_b2", 16, 1024, 2, false, false)                                                                    \
    X(3, "r16_t1024_b2_prefetch", 16, 1024, 2, true, false)                                                            \
    X(4, "r16_t512_b3", 16, 512, 3, false, false)                                                                      \
    X(5, "r16_t512_b3_prefetch", 16, 512, 3, true, false)                                                              \
    X(6, "r8_t1024_b2", 8, 1024, 2, false, false)                                                                      \
    X(7, "r8_t1024_b2_prefetch", 8, 1024, 2, true, false)                                                              \
    X(8, "r1_t1024_b2", 1, 1024, 2, false, false)                                                                      \
    X(9, "r32_t1024_b1_dual", 32, 1024, 1, false, true)                                                                \
    X(10, "r16_t512_b3_dual", 16, 512, 3, false, true)

#define RDX_CRC_KERNEL(id, name, R, T, B, PF, DU)                                                                      \
    __global__ void __launch_bounds__(T, B) crc_variant_##id(CrcJob j)                                                 \
    {                                                                                                                  \
        extern __shared__ uint32_t tab[];                                                                              \
        crc32_blocks_run<CrcShape<R, T, B, PF, DU>>(j, tab);                                                           \
    }
RDX_CRC_VARIANTS(RDX_CRC_KERNEL)

extern "C" {

int crc_variant_count(void)
{
    int n = 0;
#define RDX_COUNT(id, ...) ++n;
    RDX_CRC_VARIANTS(RDX_COUNT)
    return n;
}

const char *crc_variant_name(int v)
{
#define RDX_NAME(id, name, ...) if (v == id) return name;
    RDX_CRC_VARIANTS(RDX_NAME)
    return nullptr;
}

// Sets every variant's shared-memory limit; returns a cudaError_t.
int crc_variant_setup(void)
{
    cudaError_t e = cudaSuccess;
#define RDX_SETUP(id, name, R, T, B, PF, DU)                                                                           \
    if (e == cudaSuccess)                                                                                              \
        e = cudaFuncSetAttribute(crc_variant_##id, cudaFuncAttributeMaxDynamicSharedMemorySize,                        \
                                 (int)CrcShape<R, T, B, PF, DU>::kSmemBytes);
    RDX_CRC_VARIANTS(RDX_SETUP)
    return (int)e;
}

// Resident CTAs per SM of variant v (cudaOccupancyMaxActiveBlocksPerMultiprocessor).
int crc_variant_occupancy(int v)
{
    int n = -1;
#define RDX_OCC(id, name, R, T, B, PF, DU)                                                                             \
    if (v == id)                                                                                                      \
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, crc_variant_##id, T, CrcShape<R, T, B, PF, DU>::kSmemBytes);
    RDX_CRC_VARIANTS(RDX_OCC)
    return n;
}

// What crc_enqueue (redux_capi.cu) does, with variant v's kernel: zero d_crc, launch min(items, sms x B) CTAs.
int crc_variant_run(int v, const uint8_t *d_in, const uint64_t *d_off, uint64_t n_blocks, uint64_t max_len,
                    uint32_t *d_crc, void *stream, int sms)
{
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(d_crc, 0, n_blocks * sizeof(uint32_t), s);
    if (e != cudaSuccess || !max_len || !n_blocks) return (int)e;
    CrcJob j;
    j.in = d_in; j.in_off = d_off; j.lens = nullptr; j.crc = d_crc;
    j.n_blocks = n_blocks;
    j.piece = kCrcPiece;
    j.n_items = n_blocks * ((max_len + 30 + kCrcPiece - 1) / kCrcPiece);
#define RDX_RUN(id, name, R, T, B, PF, DU)                                                                             \
    if (v == id) {                                                                                                     \
        const uint64_t ctas = std::min<uint64_t>((j.n_items + T / 32 - 1) / (T / 32), (uint64_t)sms * B);              \
        crc_variant_##id<<<(uint32_t)ctas, T, CrcShape<R, T, B, PF, DU>::kSmemBytes, s>>>(j);                          \
    }
    RDX_CRC_VARIANTS(RDX_RUN)
    return (int)cudaGetLastError();
}

}  // extern "C"
