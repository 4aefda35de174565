"""Source-compatible surface of pytorch_bayesian.nn for the variational hot path
(pytorch_bayesian/nn/__init__.py:7-35).  Every name of the reference's `__all__` is present, so
`sys.modules['pytorch_bayesian.nn'] = bayesianneuralnetworks_b200.nn` is a total alias; the classes outside SURVEY §8's
scope (MC-dropout, evidential regression) are plain torch (nn/other.py)."""
from .container import BayesianModule, BayesianNetworkModule, register_rowwise_module
from .variational import WeightNormal
from .layers import (BayesianLinear, NormalLinear, BayesianConvNd, NormalConvNd, NormalConv1d, NormalConv2d,
                     NormalConv3d, NormalConvTransposeNd, NormalConvTranspose1d, NormalConvTranspose2d,
                     NormalConvTranspose3d)
from .flipout import (FlipoutNormalLinear, FlipOutNormalConvNd, FlipOutNormalConv1d, FlipOutNormalConv2d,
                      FlipOutNormalConv3d, FlipOutNormalConvTransposeNd, FlipOutNormalConvTranspose1d,
                      FlipOutNormalConvTranspose2d, FlipOutNormalConvTranspose3d)
from .mvn import WeightMultivariateNormal, MultivariateNormalLinear
from .loss import KLDivergence, Entropy
from .elbo import MCSamples, mc_mean_loss
from .other import (NormalInverseGaussianLinear, MCDropoutLinear, MCDropoutConvNd, MCDropoutConv1d, MCDropoutConv2d,
                    MCDropoutConv3d, NormalInverseGaussianLoss, NormalInverseGaussianUncertainty)

__all__ = [
    'BayesianModule', 'BayesianNetworkModule', 'WeightNormal', 'BayesianLinear', 'NormalLinear',
    'BayesianConvNd', 'NormalConvNd', 'NormalConv1d', 'NormalConv2d', 'NormalConv3d', 'FlipoutNormalLinear',
    'FlipOutNormalConvNd', 'FlipOutNormalConv1d', 'FlipOutNormalConv2d', 'FlipOutNormalConv3d', 'WeightMultivariateNormal',
    'MultivariateNormalLinear', 'KLDivergence', 'Entropy', 'MCSamples', 'mc_mean_loss',
    'NormalInverseGaussianLinear', 'MCDropoutLinear', 'MCDropoutConvNd', 'MCDropoutConv1d', 'MCDropoutConv2d',
    'MCDropoutConv3d', 'NormalInverseGaussianLoss', 'NormalInverseGaussianUncertainty',
    'NormalConvTransposeNd', 'NormalConvTranspose1d', 'NormalConvTranspose2d', 'NormalConvTranspose3d',
    'FlipOutNormalConvTransposeNd', 'FlipOutNormalConvTranspose1d', 'FlipOutNormalConvTranspose2d',
    'FlipOutNormalConvTranspose3d',
]
