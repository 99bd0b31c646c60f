from fine_grained_gaussian_process_forcasting_b200.gpcompat import (  # noqa: F401
    Kernel, ScaleKernel, RBFKernel, MaternKernel, RQKernel)
