"""bk200: B200-native Newton-Krylov corrector for BifurcationKit-style pseudo-arclength
continuation.  The directory name carries a dot (bifurcationkit.jl_b200), so import it through
``__graft_entry__.load_package()`` (registers it as the module ``bk200``).

Contents: csrc/ (CUDA kernels + C ABI -> libbk200.so), lib.py (ctypes binding), core.py (mirror of
the reference's AbstractLinearSolver / AbstractBorderedLinearSolver / AbstractEigenSolver surfaces),
palc.py (host-side Newton / newton_palc / continuation loop driving the device kernels).
"""
from . import lib
from .lib import (BK200Error, BK_CHAN, BK_SH2D, BK_SH3D, BK_CGL2D, BK_POTRAP_CGL2D, BK_COMPLEX, BK_PC_NONE, BK_PC_SH_DCT,
                  BK_PC_CHAN_TRIDIAG, BK_PC_CGL_DST, BK_PC_POTRAP_CIRC, BK_SPARSE, BK_PC_JACOBI, BK_SPARSE_CSR, BK_SPARSE_CSC, build)
from .core import (Context, DeviceVec, Jacobian, ComplexJacobian, GMRESB200, ComplexGMRESB200, BorderingBLSB200, MatrixFreeBLSB200, ShiftInvertB200,
                   bls_map, bls_map_block, make_opts, hessenberg_eig, sparse_pattern_args)
from . import palc
from . import segments
from . import floquet
from . import events
from . import deflation
from . import codim2
