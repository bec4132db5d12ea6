"""cuddhelmholtz_b200 — B200 (sm_100a) implementation of CuDDHelmholtz's solve path behind the reference's
own operator interface. The compute lives in csrc/ (CUDA + C ABI, include/cuddh_b200.h); this package is the
Python host mirror used by tests/ and bench.py."""
from .api import (CGS2, MGS, Basis, Comm, DDH, DDHDist, DDHPreconditioner, DDHTransfer, DiagInvFaceMassMatrix, DiagInvMassMatrix, FaceLinearFunctional, FaceMassMatrix, FaceSpace, GaussLegendre,  # noqa: F401
                  GaussLobatto, H1Space, Helmholtz, HelmholtzSlab, LinearFunctional, MassMatrix, Mesh2D, Operator, QuadratureRule, StiffnessMatrix, axpby, copy,
                  dist, dot, fill, gmres, gmres_batch, get_option, launch_count, norm, scal, set_option)
from .capi import CuddhError, load  # noqa: F401
