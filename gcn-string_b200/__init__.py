"""gcn_string_b200 — B200-native GeneralGNN hot path (see DESIGN.md).

Sub-modules: ``params`` (hyper-parameters + flat parameter layout), ``synthetic``
(E. coli-shaped graph generator), ``_lib`` (ctypes binding of the C-ABI CUDA library),
``data`` / ``layers`` / ``models`` / ``optimizers`` / ``losses`` (the Spektral/Keras
call surface the reference script uses), ``shards`` (packed device-ready ingest format),
``evaluate`` (the reference's evaluation pass and ROC metrics), ``contact`` (contact maps and pair graphs from CA
coordinates on the device), ``distributed`` (graph sharding + gradient
all-reduce).  Importing the package does not load CUDA; the first native call does and
raises if ``libgcnstring_b200.so`` is missing — there is no CPU fallback.
"""
from .params import GNNConfig, block_specs, init_params, n_state, n_trainable, named_slices  # noqa: F401

from .data import Dataset, DisjointLoader, Graph, SparseAdjacency  # noqa: F401,E402
from .layers import GeneralConv, GlobalAttnSumPool, GlobalAvgPool, GlobalSumPool, MLP  # noqa: F401,E402
from .losses import BinaryCrossentropy, CategoricalCrossentropy, binary_accuracy, categorical_accuracy  # noqa: F401,E402
from .losses import Huber, MeanAbsoluteError, MeanSquaredError, mean_absolute_error, mean_squared_error  # noqa: F401,E402
from .models import GeneralGNN, GradientTape  # noqa: F401,E402
from . import optimizers  # noqa: F401,E402
from . import shards  # noqa: F401,E402
from . import contact  # noqa: F401,E402
from .evaluate import auc, evaluate, roc_auc, roc_curve  # noqa: F401,E402

__version__ = "0.1.0"
