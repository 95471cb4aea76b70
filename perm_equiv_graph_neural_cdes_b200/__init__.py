"""B200-native (sm_100a) hot path of hits-mli/perm-equiv-graph-neural-cdes.

The package holds only what the path needs: the CUDA kernels + C-ABI (``csrc/``, built into
``libpegncde.so``) and the host-side mirror of the reference's vector-field / solve interface.
Importing it fails loudly when the CUDA extension has not been built -- there is no CPU fallback.
"""
from ._lib import LIB_PATH, PegControl, PegDims, PegError, lib  # noqa: F401

lib()  # raise ImportError right here if libpegncde.so is missing

from .control import CubicInterpolation, LinearInterpolation, PackedControl, backward_hermite_coefficients, build_control, pack_control  # noqa: E402,F401
from .control import SparseControl, SparsePattern, build_sparse_control, pack_sparse_control, sparse_pattern  # noqa: E402,F401
from .models import MLP, GraphNeuralCDE, PGTGraphNeuralCDE, TGBGraphNeuralCDE  # noqa: E402,F401
from .solve import (ConstantStepSize, ODETerm, PIDController, SaveAt, Solution, Tsit5, clip_to_end, constant_step_table,  # noqa: E402,F401
                    dense_weights, diffeqsolve, tsit5_step)  # noqa: E402,F401
from .vector_field import (CDEWrapperVectorField, ConvEquivFusionDirectedLayer, ConvEquivFusionLayer, ConvLayer,  # noqa: E402,F401
                           GNODEVectorField, GraphVectorField, PermEquivDirGraphVectorField, PermEquivGraphVectorField)  # noqa: E402,F401

__version__ = "0.1.0"
