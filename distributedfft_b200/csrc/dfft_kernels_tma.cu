// dfft_kernels_tma.cu -- instantiations and host-side helpers of the TMA-pipelined pass kernels (fft_tma.cuh).
#include <cuda.h>

#include <mutex>

#include "dfft_kernels.cuh"
#include "fft_tma.cuh"

namespace dfft {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn()
{
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess) fn = (EncodeTiledFn)p;
        cudaGetLastError();
    });
    return fn;
}

bool tma_available() { return encode_fn() != nullptr; }

// 3-D tensor of complex elements: dim0 (fastest, contiguous) d0, dim1 d1 with stride s1, dim2 d2 with stride s2 (strides in complex
// elements); box (b0, b1, b2).  `map` points to 128 bytes, 64-byte aligned (a CUtensorMap).
int tma_encode_3d(void* map, void* base, int prec, long long d0, long long d1, long long d2, long long s1, long long s2, int b0, int b1, int b2)
{
    EncodeTiledFn fn = encode_fn();
    if (!fn) return -1;
    const size_t esz = prec == 0 ? 16 : 8;
    cuuint64_t dims[3] = {(cuuint64_t)d0 * 2, (cuuint64_t)d1, (cuuint64_t)d2};
    cuuint64_t strides[2] = {(cuuint64_t)s1 * esz, (cuuint64_t)s2 * esz};
    cuuint32_t box[3] = {(cuuint32_t)b0 * 2, (cuuint32_t)b1, (cuuint32_t)b2};
    cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = fn((CUtensorMap*)map, prec == 0 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, base, dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : (int)r;
}

template <class S, typename T, int C>
static cudaError_t launch_tma(int mode, const void* vargs, const void* map_in, const void* map_out, int sm_count, cudaStream_t st)
{
    const TmaArgs<T>& a = *reinterpret_cast<const TmaArgs<T>*>(vargs);
    using G_ = TmaGeom<S, T, C>;
    static CUtensorMap dummy{};
    const CUtensorMap& mi = map_in ? *reinterpret_cast<const CUtensorMap*>(map_in) : dummy;
    const CUtensorMap& mo = map_out ? *reinterpret_cast<const CUtensorMap*>(map_out) : dummy;
    if (a.ntiles <= 0) return cudaSuccess;
    long long grid = sm_count;
    if (grid > a.ntiles) grid = a.ntiles;
    cudaError_t e = cudaSuccess;
#define DFFT_TMA_LAUNCH(M)                                                                                                  \
    {                                                                                                                       \
        auto kern = fft_tma_pass_kernel<S, T, C, M>;                                                                        \
        static bool attr = false;                                                                                           \
        if (!attr) { e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)G_::SMEM); if (e != cudaSuccess) return e; attr = true; } \
        kern<<<(unsigned)grid, S::T * C, G_::SMEM, st>>>(a, mi, mo);                                                        \
    }
    switch (mode) {
        case TMA_Z: DFFT_TMA_LAUNCH(TMA_Z) break;
        case TMA_Y: DFFT_TMA_LAUNCH(TMA_Y) break;
        case TMA_XF: DFFT_TMA_LAUNCH(TMA_XF) break;
        case TMA_XB: DFFT_TMA_LAUNCH(TMA_XB) break;
        default: return cudaErrorInvalidValue;
    }
#undef DFFT_TMA_LAUNCH
    return cudaGetLastError();
}

template <class S, typename T, int C> static TmaEntry make_tma_entry(unsigned use)
{
    TmaEntry e{};
    e.use = use;
    e.N = S::N;
    e.prec = sizeof(T) == 8 ? 0 : 1;
    e.C = C;
    e.rows = TmaGeom<S, T, C>::ROWS;
    e.nstages = S::NSTAGES;
    for (int i = 0; i < S::NSTAGES; i++) e.rad[i] = S::rad(i);
    e.launch = launch_tma<S, T, C>;
    return e;
}

static std::vector<TmaEntry>& tma_table()
{
    static std::vector<TmaEntry> t;
    static std::once_flag once;
    std::call_once(once, [] {
        // tile = C lines of N points = 64 KB (48 KB for 768), S::T * C threads, one CTA per SM
        // which modes to use (measured per pass at N^3 on one B200, TMA vs register-staged ms):
        constexpr unsigned Z = 1u << TMA_Z, Y = 1u << TMA_Y, X = (1u << TMA_XF) | (1u << TMA_XB);
        t.push_back(make_tma_entry<Sched<512, 8, 8, 8, 8>, double, 8>(Y));               // Z .741/.697  Y .756/.781  X .781/.775
        t.push_back(make_tma_entry<Sched<1024, 8, 8, 8, 8, 2>, double, 4>(Y | X));       // Z 7.21/6.73  Y 7.59/9.23  X 8.30/8.49
        t.push_back(make_tma_entry<Sched<256, 8, 8, 8, 4>, double, 16>(Z | Y | X));      // Z .100/.120  Y .099/.113  X .103/.114
        t.push_back(make_tma_entry<Sched<768, 12, 4, 4, 4, 4, 3>, double, 4>(Y));        // Z 3.57/2.83  Y 3.56/3.87  X 3.79/3.53
        t.push_back(make_tma_entry<Sched<512, 16, 8, 8, 8>, float, 16>(Z | Y | X));      // Z .392/.454  Y .370/.523  X .380/.542
        t.push_back(make_tma_entry<Sched<1024, 16, 16, 8, 8>, float, 8>(Y | X));         // Z 3.48/2.99  Y 3.23/5.10  X 3.95/4.39
        t.push_back(make_tma_entry<Sched<768, 12, 4, 4, 4, 4, 3>, float, 8>(Y | X));     // Z 1.87/1.74  Y 1.78/1.92  X 1.90/2.01
    });
    return t;
}

const TmaEntry* find_tma_entry(int N, int prec)
{
    const char* env = getenv("DFFT_TMA");
    if (env && atoi(env) == 0) return nullptr;
    if (getenv("DFFT_GENERIC") && atoi(getenv("DFFT_GENERIC")) != 0) return nullptr;
    if (!tma_available()) return nullptr;
    // DFFT_TMA=2: a copy of every entry with all modes on.  One copy per entry, built once: a plan keeps the pointers of all
    // three axes (and of other plans) alive, so they must not share one slot.
    static std::vector<TmaEntry> forced;
    static std::once_flag once;
    std::call_once(once, [] {
        forced = tma_table();
        for (TmaEntry& e : forced) e.use = 0xf;
    });
    const std::vector<TmaEntry>& t = env && atoi(env) == 2 ? forced : tma_table();
    for (const TmaEntry& e : t)
        if (e.N == N && e.prec == prec) return &e;
    return nullptr;
}

}  // namespace dfft
