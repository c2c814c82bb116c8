// Explicit instantiation of the FPN-chain kernel for V = 18 joints.
#include "fpn_launch.h"
template int cg::launch_fpn_impl<18>(const cg::FpnArgs&, void*);
