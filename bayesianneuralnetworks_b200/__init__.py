"""bayesianneuralnetworks_b200 — the variational hot path of pytorch_bayesian
(Mirko-Nava/BayesianNeuralNetworks) on B200: hand-written sm_100a kernels behind a C ABI
(include/bnn_b200.h, libbnn_b200.so) and this source-compatible mirror of pytorch_bayesian.nn /
.prune / .utils.  There is no CPU or PyTorch fallback for the hot path: modules may be built on the
CPU, but forward, KL, `.sampled` and pruning need a compute-capability-10.x device."""
from . import nn, optim, prune, utils
from .functional import set_conv_output_format
from .runtime import (advance_rng_step, graph_safe_rng, injected_eps, manual_seed, mc_batching, precision_name,
                      set_mc_batching, set_precision, set_sample_partition)

__version__ = '0.0.4+b200'

__all__ = ['nn', 'optim', 'prune', 'utils', '__version__', 'manual_seed', 'set_precision', 'precision_name',
           'set_mc_batching', 'mc_batching', 'set_sample_partition', 'injected_eps', 'graph_safe_rng',
           'advance_rng_step', 'set_conv_output_format']
