"""lrvb_b200 -- B200-native (sm_100a CUDA) implementation of the data-parallel hot path of
rgiordan/LinearResponseVariationalBayes.py: logistic-GLMM ELBO, gradient, sparse Hessian, HVP,
CG and LRVB covariances, behind the reference's Python API.

Import as ``import lrvb_b200 as vb`` (the repo-root shim ``lrvb_b200.py`` loads this directory,
whose on-disk name contains a dot, as the package ``lrvb_b200``).
"""
from .Parameters import (ScalarParam, VectorParam, ArrayParam, constrain, unconstrain,  # noqa: F401
                         convert_vector_to_free_hessian, set_free_offset, set_vector_offset,
                         get_free_offset, get_vector_offset, free_to_vector_jac_offset,
                         free_to_vector_hess_offset)
from .ParameterDictionary import ModelParamsDict  # noqa: F401
from .MatrixParameters import (PosDefMatrixParam, PosDefMatrixParamVector,  # noqa: F401
                               PosDefMatrixParamArray)
from .NormalParams import (UVNParam, UVNParamVector, UVNParamArray, MVNParam,  # noqa: F401
                           UVNMomentParamArray, MVNArray)
from .GammaParams import GammaParam  # noqa: F401
from .DirichletParams import DirichletParamArray  # noqa: F401
from .WishartParams import WishartParam  # noqa: F401
from .SimplexParams import SimplexParam  # noqa: F401
from . import MatrixParameters  # noqa: F401
from . import SimplexParams  # noqa: F401
from . import ExponentialFamilies  # noqa: F401
from . import Modeling  # noqa: F401
from . import SparseObjectives  # noqa: F401
from . import ConjugateGradient  # noqa: F401
from . import ModelSensitivity  # noqa: F401
from . import OptimizationUtils  # noqa: F401
from . import GLMM  # noqa: F401
from .SparseObjectives import (Objective, Logger, Timer, make_index_param,  # noqa: F401
                               get_sparse_sub_matrix, get_sparse_sub_hessian, pack_csr_matrix,
                               unpack_csr_matrix, json_pack_csr_matrix,
                               json_unpack_csr_matrix, safe_matmul)
from .ConjugateGradient import ConjugateGradientSolver  # noqa: F401
from .ModelSensitivity import (LinearResponseCovariances, ArrowheadCovariance,  # noqa: F401
                               WeightSensitivityLinearApproximation)
from .GLMM import (LogisticGLMM, GLMMPrior, DeviceCSR, Prediction, ApproximateLOO, ApproximateLOGO,  # noqa: F401
                   ApproximateMaxInfluence, DropResult)

__version__ = "0.1.0"
