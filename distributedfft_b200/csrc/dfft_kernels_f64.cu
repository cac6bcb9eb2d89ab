// fp64 instantiations.  Per-length choices come from kbench sweeps on B200 (profiles/kbench*.log):
// small CTAs (finer barriers) win for the contiguous pass, 128-byte row segments (C = 8 complex
// doubles) for the strided ones.
#include "dfft_kernels_inst.cuh"
namespace dfft {
void register_f64(std::vector<SizeEntry>& v)
{
    using T = double;
    v.push_back(make_entry<T, Cfg<Sched<4, 2, 2, 2>, 64, false, 4, true>, Cfg<Sched<4, 2, 2, 2>, 32, false, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<8, 4, 4, 2>, 64, false, 4, true>, Cfg<Sched<8, 4, 4, 2>, 32, false, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<16, 4, 4, 4>, 32, false, 4, true>, Cfg<Sched<16, 4, 4, 4>, 32, false, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<32, 8, 8, 4>, 32, false, 4, true>, Cfg<Sched<32, 8, 8, 4>, 32, false, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<64, 8, 8, 8>, 16, true, 4, true>, Cfg<Sched<64, 8, 8, 8>, 16, true, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<128, 16, 16, 8>, 16, false, 4, true>, Cfg<Sched<128, 16, 16, 8>, 16, false, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<256, 16, 16, 16>, 8, false, 4, true>, Cfg<Sched<256, 16, 16, 16>, 8, false, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<512, 8, 8, 8, 8>, 2, true, 4, true>, Cfg<Sched<512, 16, 8, 8, 8>, 8, false, 2, false>>());
    // 1024 (kbench5): contiguous R=8 with register twiddles 6.66 ms vs 7.73; X pass C=8 8.34 vs 8.58; 128-byte rows for peer stores
    v.push_back(make_entry<T, Cfg<Sched<1024, 8, 8, 8, 8, 2>, 1, true, 4, true>, Cfg<Sched<1024, 16, 16, 8, 8>, 4, false, 2, false>,
                           Cfg<Sched<1024, 16, 16, 8, 8>, 8, false, 1, false>, Cfg<Sched<1024, 16, 16, 8, 8>, 8, false, 1, false>>());
    v.push_back(make_entry<T, Cfg<Sched<2048, 16, 16, 16, 8>, 1, false, 4, false>, Cfg<Sched<2048, 16, 16, 16, 8>, 4, false, 1, false>>());
    v.push_back(make_entry<T, Cfg<Sched<4096, 16, 16, 16, 16>, 1, false, 2, false>, Cfg<Sched<4096, 16, 16, 16, 16>, 2, false, 1, false>>());
#ifdef DFFT_EXPERIMENTS   // build with -DDFFT_EXPERIMENTS (python -m distributedfft_b200.build --experiments): alternate tunings selected
                          // at run time with DFFT_VARIANT=n; every instantiation of the default tables runs against an fp64 reference
                          // in tests/test_gpu_parity.py / test_gpu_multi.py (cases: tests/kernel_matrix.py, completeness checked on
                          // the CPU by tests/test_kernel_matrix_complete.py)
    // experiments for the fused t0 kernel (DFFT_VARIANT=1|2, not used by default): the strided role reads its tile from L2,
    // not HBM, so narrow tiles (64- / 32-byte rows) cost no DRAM efficiency there and allow 3-5 smaller CTAs per SM
    // (finer-grained phases; the fused kernel's top stall is the CTA barrier, profiles/r1_ncu_full_fused_t0_512.txt)
    v.push_back(make_entry<T, Cfg<Sched<512, 8, 8, 8, 8>, 2, true, 4, true>, Cfg<Sched<512, 8, 8, 8, 8>, 4, false, 3, false>>(1));
    v.push_back(make_entry<T, Cfg<Sched<512, 8, 8, 8, 8>, 2, true, 4, true>, Cfg<Sched<512, 8, 8, 8, 8>, 2, false, 5, false>>(2));
    // DFFT_VARIANT=3|4: the default / the 3-CTA shapes with L2 eviction hints in the fused kernels (streamed data evict_first,
    // the Z->Y intermediate evict_last: the lag sweep says the intermediate survives only a few planes otherwise)
    using Y512 = Cfg<Sched<512, 16, 8, 8, 8>, 8, false, 2, false>;
    using Y512n = Cfg<Sched<512, 8, 8, 8, 8>, 4, false, 3, false>;
    v.push_back(make_entry<T, Cfg<Sched<512, 8, 8, 8, 8>, 2, true, 4, true>, Y512, Y512, Y512, 1>(3));
    v.push_back(make_entry<T, Cfg<Sched<512, 8, 8, 8, 8>, 2, true, 4, true>, Y512n, Y512n, Y512n, 1>(4));
    // DFFT_VARIANT=6|7|8: the contiguous role of the fused kernels synchronises per line (2 warps) instead of per CTA:
    // default shapes, 3-CTA shapes, 3-CTA shapes + L2 hints
    v.push_back(make_entry<T, Cfg<Sched<512, 8, 8, 8, 8>, 2, true, 4, true>, Y512, Y512, Y512, 2>(6));
    v.push_back(make_entry<T, Cfg<Sched<512, 8, 8, 8, 8>, 2, true, 4, true>, Y512n, Y512n, Y512n, 2>(7));
    v.push_back(make_entry<T, Cfg<Sched<512, 8, 8, 8, 8>, 2, true, 4, true>, Y512n, Y512n, Y512n, 3>(8));
#endif
    using Y512d = Cfg<Sched<512, 16, 8, 8, 8>, 8, false, 2, false>;
    // DFFT_VARIANT=5: 256-byte rows for the peer (NVLink) stores only; local passes keep the default shapes
    v.push_back(make_entry<T, Cfg<Sched<512, 8, 8, 8, 8>, 2, true, 4, true>, Y512d, Y512d, Cfg<Sched<512, 16, 8, 8, 8>, 16, false, 1, false>>(5));
    // mixed radix
    // 768 (kbench5): 24 points/thread (8.8.4.3, three exchanges instead of four): Z 2.83 vs 3.45 ms, Y 3.87 vs 4.28, X 3.52 vs 4.19
    v.push_back(make_entry<T, Cfg<Sched<768, 24, 8, 8, 4, 3>, 4, false, 2, false>, Cfg<Sched<768, 24, 8, 8, 4, 3>, 4, false, 2, false>>());
    v.push_back(make_entry<T, Cfg<Sched<384, 12, 4, 4, 4, 3, 2>, 4, false, 4, true>, Cfg<Sched<384, 12, 4, 4, 4, 3, 2>, 8, false, 2, false>>());
    v.push_back(make_entry<T, Cfg<Sched<192, 12, 4, 4, 4, 3>, 8, false, 4, true>, Cfg<Sched<192, 12, 4, 4, 4, 3>, 8, false, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<96, 12, 4, 4, 3, 2>, 16, false, 4, true>, Cfg<Sched<96, 12, 4, 4, 3, 2>, 16, false, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<48, 12, 4, 4, 3>, 32, false, 4, true>, Cfg<Sched<48, 12, 4, 4, 3>, 32, false, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<24, 6, 3, 2, 2, 2>, 32, false, 4, true>, Cfg<Sched<24, 6, 3, 2, 2, 2>, 32, false, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<12, 6, 3, 2, 2>, 64, false, 4, true>, Cfg<Sched<12, 6, 3, 2, 2>, 32, false, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<6, 6, 3, 2>, 64, false, 4, true>, Cfg<Sched<6, 6, 3, 2>, 32, false, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<9, 3, 3, 3>, 32, false, 4, true>, Cfg<Sched<9, 3, 3, 3>, 32, false, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<10, 10, 5, 2>, 64, false, 4, true>, Cfg<Sched<10, 10, 5, 2>, 32, false, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<100, 10, 5, 5, 2, 2>, 16, false, 4, true>, Cfg<Sched<100, 10, 5, 5, 2, 2>, 16, false, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<125, 5, 5, 5, 5>, 8, false, 4, true>, Cfg<Sched<125, 5, 5, 5, 5>, 8, false, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<49, 7, 7, 7>, 16, false, 4, true>, Cfg<Sched<49, 7, 7, 7>, 16, false, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<243, 9, 3, 3, 3, 3, 3>, 8, false, 4, true>, Cfg<Sched<243, 9, 3, 3, 3, 3, 3>, 8, false, 4, true>>());
    v.push_back(make_entry<T, Cfg<Sched<1000, 10, 5, 5, 5, 2, 2, 2>, 2, false, 4, true>, Cfg<Sched<1000, 10, 5, 5, 5, 2, 2, 2>, 4, false, 2, false>>());
}
}  // namespace dfft
