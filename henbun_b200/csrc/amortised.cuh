// The network layout of the amortised model (BASELINE config 4) shared by its fp32 (amortised.cu) and fp64 (amortised64.cu)
// entry points: which configs are valid and where each layer's weight and bias sit in the packed parameter vector.
#pragma once
#include "../../include/henbun_b200.h"
#include <stddef.h>

namespace hb {

bool amortised_valid(const hb_amortised_config& c);
// offsets of w_l [nodes[l], nodes[l + 1]] and b_l [nodes[l + 1]] from `start`; returns the end
size_t amortised_net_params(const int* nodes, int n, size_t start, size_t* w_off, size_t* b_off);

}  // namespace hb
