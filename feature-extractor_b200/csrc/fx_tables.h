// fx_tables.h -- host-side table builders shared by fx_engine.cu (see fx_tables.cu)
#pragma once
#include "fx_kernels.cuh"
#include <vector>

namespace fx {
void build_twiddles (int N, std::vector<float2>& tw2, std::vector<float2>& tw1f);
void build_lag_tables (int N, double sample_rate, std::vector<short>& her_tab);
void build_exact_ratio_table (int N, double sample_rate, std::vector<double>& ex_tab, std::vector<int>& ex_off);
}
