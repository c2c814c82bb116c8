// Explicit instantiation of the tensor-core FPN kernel for V = 22 joints, single-term bf16 operands.
#include "fpn_tc_launch.h"
#ifndef CISTGCN_EMU
template int cg::launch_fpn_tc_impl<22, true>(const cg::FpnTcArgs&, void*);
#endif
