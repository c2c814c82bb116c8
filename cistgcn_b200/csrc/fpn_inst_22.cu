// Explicit instantiation of the FPN-chain kernel for V = 22 joints.
#include "fpn_launch.h"
template int cg::launch_fpn_impl<22>(const cg::FpnArgs&, void*);
