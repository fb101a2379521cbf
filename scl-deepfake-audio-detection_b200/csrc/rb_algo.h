// rb_algo.h -- which operators each algo of the reference's dispatcher (asvspoof_2019_augall_3.py:377-439) runs:
// 1 LnL, 2 ISD, 3 SSI, 4 LnL>ISD>SSI, 5 LnL>ISD, 6 LnL>SSI, 7 ISD>SSI, 8 LnL+ISD; any other value none.
// The one C++ definition, shared by device code, nvcc host code and the g++-compiled planner; plans.ALGO_USES_* is the
// Python one. The order the operators run in is rb_process's.
#pragma once

#ifdef __CUDACC__
#define RB_ALGO_HD __host__ __device__
#else
#define RB_ALGO_HD
#endif

namespace rb {

RB_ALGO_HD constexpr bool algo_uses_lnl(int algo) { return algo == 1 || algo == 4 || algo == 5 || algo == 6 || algo == 8; }
RB_ALGO_HD constexpr bool algo_uses_isd(int algo) { return algo == 2 || algo == 4 || algo == 5 || algo == 7 || algo == 8; }
RB_ALGO_HD constexpr bool algo_uses_ssi(int algo) { return algo == 3 || algo == 4 || algo == 6 || algo == 7; }

}  // namespace rb

#undef RB_ALGO_HD
