"""Exact GP model with the reference's API (/root/reference/denoising_model/GPModel.py:4-13):
``ExactGPModel(train_x, train_y, likelihood)`` with a constant mean and ScaleKernel(RBF) prior whose
dense covariance is built by the gpblur CUDA kernel and is differentiable (hand-written backward,
``gpblur_covariance_backward``): the model trains with ``gpcompat.ExactMarginalLogLikelihood`` exactly as a
gpytorch exact GP does.  (Imported nowhere in the reference; kept for API completeness.)"""
from . import gpcompat as gp


class ExactGPModel(gp.ExactGP):
    def __init__(self, train_x, train_y, likelihood):
        super().__init__(train_x, train_y, likelihood)
        self.mean_module = gp.ConstantMean()
        self.covar_module = gp.ScaleKernel(gp.RBFKernel())

    def forward(self, x):
        return gp.MultivariateNormal(self.mean_module(x), self.covar_module(x))
