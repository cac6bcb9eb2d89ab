// dfft_kernels_inst.cuh -- launcher template + size-table macros, included by the per-precision
// instantiation units.
#pragma once
#include <atomic>
#include <type_traits>
#include "dfft_kernels.cuh"

namespace dfft {

template <class S, typename T, int C, int MI, int MO, bool TW, bool CI, bool CO, int MINB, bool PP, bool EPI = false>
cudaError_t launch_pass(const void* vargs, int sm_count, cudaStream_t st)
{
    const TileArgs<T>& a = *reinterpret_cast<const TileArgs<T>*>(vargs);
    auto kern = fft_tile_kernel<S, T, C, MI, MO, TW, CI, CO, MINB, PP, false, EPI>;
    constexpr size_t smem = TileSmem<S, T, C, PP>::bytes(CI || CO);
    static std::atomic<int> occ_cache[64];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    int occ = occ_cache[dev & 63].load();
    if (occ == 0) {
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, S::T * C, smem);
        if (e != cudaSuccess) return e;
        if (occ < 1) return cudaErrorLaunchOutOfResources;
        occ_cache[dev & 63].store(occ);
    }
    if (a.ntiles <= 0) return cudaSuccess;
    if (a.max_ctas_per_sm > 0 && occ > a.max_ctas_per_sm) occ = a.max_ctas_per_sm;
    long long grid = (long long)sm_count * occ;
    if (grid > a.ntiles) grid = a.ntiles;
    kern<<<(unsigned)grid, S::T * C, smem, st>>>(a);
    return cudaGetLastError();
}

// dynamic shared memory one CTA may use on sm_100 (cudaDevAttrMaxSharedMemoryPerBlockOptin: 227 KB)
constexpr size_t DFFT_MAX_SMEM = 227 * 1024;
// shared memory of a kernel running several TileOp roles: one exchange buffer (the largest) + every role's own part
template <class A, class... More> constexpr size_t roles_smem()
{
    size_t exch = A::SM::exch_bytes, aux = A::aux_bytes;
    ((exch = More::SM::exch_bytes > exch ? More::SM::exch_bytes : exch), ...);
    ((aux += More::aux_bytes), ...);
    return exch + aux;
}

template <class OpA, class OpB, typename T, int MINB>
cudaError_t launch_fused(const void* va, const void* vb, const FusedCtl* ctl, int sm_count, cudaStream_t st)
{
    const TileArgs<T>& a = *reinterpret_cast<const TileArgs<T>*>(va);
    const TileArgs<T>& b = *reinterpret_cast<const TileArgs<T>*>(vb);
    auto kern = fft_fused2_kernel<OpA, OpB, T, MINB>;
    constexpr size_t smem = roles_smem<OpA, OpB>();
    static std::atomic<int> occ_cache[64];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    int occ = occ_cache[dev & 63].load();
    if (occ == 0) {
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, OpA::NT, smem);
        if (e != cudaSuccess) return e;
        if (occ < 1) return cudaErrorLaunchOutOfResources;
        occ_cache[dev & 63].store(occ);
    }
    if (ctl->planes <= 0) return cudaSuccess;
    const long long total = ctl->planes * ((long long)ctl->GA + ctl->GB);
    if (total >= (1ll << 31)) return cudaErrorInvalidConfiguration;   // the kernel decodes tickets in 32 bits
    long long grid = (long long)sm_count * occ;
    if (grid > total) grid = total;
    FusedCtl c = *ctl;
    if (c.lag <= 0) c.lag = (int)((grid + c.GA + c.GB - 1) / ((long long)c.GA + c.GB)) + 1;   // role A stays one in-flight window ahead
    kern<<<(unsigned)grid, OpA::NT, smem, st>>>(a, b, c);
    return cudaGetLastError();
}

template <class OpA, class OpB, typename T, int MINB>
cudaError_t launch_fused_yx(const void* va, const void* vb, const YxCtl* ctl, int sm_count, cudaStream_t st)
{
    const TileArgs<T>& a = *reinterpret_cast<const TileArgs<T>*>(va);
    const TileArgs<T>& b = *reinterpret_cast<const TileArgs<T>*>(vb);
    auto kern = fft_fused_yx_kernel<OpA, OpB, T, MINB>;
    constexpr size_t smem = roles_smem<OpA, OpB>();
    static std::atomic<int> occ_cache[64];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    int occ = occ_cache[dev & 63].load();
    if (occ == 0) {
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, OpA::NT, smem);
        if (e != cudaSuccess) return e;
        if (occ < 1) return cudaErrorLaunchOutOfResources;
        occ_cache[dev & 63].store(occ);
    }
    const long long total = (long long)ctl->TA + ctl->TB;
    if (total <= 0) return cudaSuccess;
    long long grid = (long long)sm_count * occ;
    if (grid > total) grid = total;
    kern<<<(unsigned)grid, OpA::NT, smem, st>>>(a, b, *ctl);
    return cudaGetLastError();
}

template <class OpA, class OpB, class OpC, typename T, int MINB>
cudaError_t launch_fused3(const void* va, const void* vb, const void* vc, const Fused3Ctl* ctl, int sm_count, cudaStream_t st)
{
    const TileArgs<T>& a = *reinterpret_cast<const TileArgs<T>*>(va);
    const TileArgs<T>& b = *reinterpret_cast<const TileArgs<T>*>(vb);
    const TileArgs<T>& c = *reinterpret_cast<const TileArgs<T>*>(vc);
    auto kern = fft_fused3_kernel<OpA, OpB, OpC, T, MINB>;
    constexpr size_t smem = roles_smem<OpA, OpB, OpC>();
    static std::atomic<int> occ_cache[64];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    int occ = occ_cache[dev & 63].load();
    if (occ == 0) {
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, OpA::NT, smem);
        if (e != cudaSuccess) return e;
        if (occ < 1) return cudaErrorLaunchOutOfResources;
        occ_cache[dev & 63].store(occ);
    }
    if (ctl->planes <= 0) return cudaSuccess;
    const long long total = ctl->planes * ((long long)ctl->GA + ctl->GB) + ctl->rows * (long long)ctl->GX;
    if (total >= (1ll << 31)) return cudaErrorInvalidConfiguration;   // the kernel decodes tickets in 32 bits
    long long grid = (long long)sm_count * occ;
    if (grid > total) grid = total;
    Fused3Ctl f = *ctl;
    if (f.lag <= 0) f.lag = (int)((grid + f.GA + f.GBk - 1) / ((long long)f.GA + f.GBk)) + 1;
    kern<<<(unsigned)grid, OpA::NT, smem, st>>>(a, b, c, f);
    return cudaGetLastError();
}

template <class S> void fill_rad(int& n, int* rad)
{
    n = S::NSTAGES;
    for (int i = 0; i < S::NSTAGES; i++) rad[i] = S::rad(i);
}

// One kernel configuration: schedule, lines per tile, twiddles in registers, min CTAs/SM, ping-pong exchange buffer
template <class S_, int C_, bool TW_, int MB_, bool PP_> struct Cfg {
    using S = S_;
    static constexpr int C = C_, MB = MB_;
    static constexpr bool TW = TW_, PP = PP_;
};

// Z: contiguous pass.  Y: strided pass on local memory (t0 axis-1, backward unpack).  X: the t3 passes (strided on one
// side, contiguous on the other).  PEER: the Y pass with the chunked store (pack / peer receive buffers over NVLink),
// which wants >= 128-byte row segments; must use Y's schedule (it shares the twiddle table).
// FH bit 0: the fused t0 kernels carry L2 eviction hints (first role: streamed input evict_first, intermediate evict_last;
// second role: intermediate and output evict_first); FH bit 1: the contiguous role of the fused kernels synchronises per
// line (named barriers) instead of per CTA -- experiments, see DESIGN.md
template <typename T, class Z, class Y, class X = Y, class PEER = Y, int FH = 0>
SizeEntry make_entry(int variant = 0)
{
    using ZS = typename Z::S;
    using SS = typename Y::S;
    using XS = typename X::S;
    static_assert(std::is_same<typename PEER::S, SS>::value, "the peer-store configuration shares the Y schedule");
    SizeEntry e{};
    e.N = ZS::N;
    e.variant = variant;
    e.prec = sizeof(T) == 8 ? 0 : 1;
    e.z_C = Z::C;
    e.s_C = Y::C;
    e.p_C = PEER::C;
    e.x_C = X::C;
    fill_rad<ZS>(e.z_nstages, e.z_rad);
    fill_rad<SS>(e.s_nstages, e.s_rad);
    fill_rad<XS>(e.x_nstages, e.x_rad);
    e.launch[PK_Z] = launch_pass<ZS, T, Z::C, MAP_T, MAP_T, Z::TW, false, false, Z::MB, Z::PP>;
    e.launch[PK_Y] = launch_pass<SS, T, Y::C, MAP_C, MAP_C, Y::TW, false, false, Y::MB, Y::PP>;
    e.launch[PK_Y_CO] = launch_pass<SS, T, PEER::C, MAP_C, MAP_C, PEER::TW, false, true, PEER::MB, PEER::PP>;
    e.launch[PK_Y_CI] = launch_pass<SS, T, Y::C, MAP_C, MAP_C, Y::TW, true, false, Y::MB, Y::PP>;
    e.launch[PK_XF] = launch_pass<XS, T, X::C, MAP_C, MAP_T, X::TW, false, false, X::MB, X::PP>;
    e.launch[PK_XB] = launch_pass<XS, T, X::C, MAP_T, MAP_C, X::TW, false, false, X::MB, X::PP>;
    e.launch[PK_XB_CO] = launch_pass<XS, T, X::C, MAP_T, MAP_C, X::TW, false, true, X::MB, X::PP>;
    e.launch[PK_XF_TW] = launch_pass<XS, T, X::C, MAP_C, MAP_T, X::TW, false, false, X::MB, X::PP, true>;
    // fused two-pass kernels: the contiguous role is re-tiled so that both roles fill the same CTA
    constexpr int NT = SS::T * Y::C, NTP = SS::T * PEER::C;
    static_assert(NT % ZS::T == 0 && NTP % ZS::T == 0, "strided CTA size must be a multiple of the contiguous line's thread count");
    e.f_zC = NT / ZS::T;
    e.f_zCp = NTP / ZS::T;
    constexpr int H1 = (FH & 1) ? 1 : 0, H2 = (FH & 1) ? 2 : 0;
    constexpr bool ZL = (FH & 2) != 0 && ZS::T % 32 == 0 && NT / ZS::T <= 15;
    constexpr bool ZLp = (FH & 2) != 0 && ZS::T % 32 == 0 && NTP / ZS::T <= 15;
    // first-role flavour (intermediate written with evict_last) and second-role flavour (everything evict_first)
    using OZ = TileOp<ZS, T, NT / ZS::T, MAP_T, MAP_T, false, false, false, false, false, H1, H2, false, ZL>;
    using OZ2 = TileOp<ZS, T, NT / ZS::T, MAP_T, MAP_T, false, false, false, false, false, H1, H1, false, ZL>;
    using OZp = TileOp<ZS, T, NTP / ZS::T, MAP_T, MAP_T, false, false, false, false, false, H1, H2, false, ZLp>;
    using OY = TileOp<SS, T, Y::C, MAP_C, MAP_C, false, false, false, false, false, H1, H2>;
    using OY2 = TileOp<SS, T, Y::C, MAP_C, MAP_C, false, false, false, false, false, H1, H1>;
    using OYco = TileOp<SS, T, PEER::C, MAP_C, MAP_C, false, false, true, false, false, H1, 0>;
    using OYci = TileOp<SS, T, Y::C, MAP_C, MAP_C, false, true, false, false, false, H1, H2>;
    // a multi-role kernel whose roles together need more shared memory than one CTA may have cannot launch: it gets no
    // launcher (nullptr), and plans of this length run the passes as separate kernels instead
    if constexpr (roles_smem<OZ, OY2>() <= DFFT_MAX_SMEM) e.fused[FK_ZY] = launch_fused<OZ, OY2, T, Y::MB>;
    if constexpr (roles_smem<OZp, OYco>() <= DFFT_MAX_SMEM) e.fused[FK_ZY_CO] = launch_fused<OZp, OYco, T, PEER::MB>;
    if constexpr (roles_smem<OY, OZ2>() <= DFFT_MAX_SMEM) e.fused[FK_YZ] = launch_fused<OY, OZ2, T, Y::MB>;
    if constexpr (roles_smem<OYci, OZ2>() <= DFFT_MAX_SMEM) e.fused[FK_YZ_CI] = launch_fused<OYci, OZ2, T, Y::MB>;
    // whole forward transform of a device in one kernel: needs the X role to fill the peer-store CTA shape
    e.fused3 = nullptr;
    e.fused_yx = nullptr;
    if constexpr (XS::T * X::C == NTP) {
        using OX = TileOp<XS, T, X::C, MAP_C, MAP_T, false, false, false, false>;
        if constexpr (roles_smem<OZp, OYco, OX>() <= DFFT_MAX_SMEM)
            e.fused3 = launch_fused3<OZp, OYco, OX, T, (PEER::MB < X::MB ? PEER::MB : X::MB)>;
        if constexpr (roles_smem<OYco, OX>() <= DFFT_MAX_SMEM)
            e.fused_yx = launch_fused_yx<OYco, OX, T, (PEER::MB < X::MB ? PEER::MB : X::MB)>;
    }
    return e;
}

}  // namespace dfft
