"""gpb200 -- host-side mirror of the GaussianProcesses.jl GP / GPE / Kernel / predict_f surface
over libgpb200.so (the B200-native exact-GP hot path).  See DESIGN.md / INTEGRATION.md."""
from .capi import Engine, FitcEngine, LocalGroupEngine, PosDefException, load_library, declared_symbols, LIB_PATH
from .kernels import (Kernel, SEIso, SEArd, SE, Mat12Iso, Mat32Iso, Mat52Iso, Mat12Ard, Mat32Ard, Mat52Ard, Matern,
                      RQIso, RQArd, RQ, Periodic, LinIso, LinArd, Poly, Noise, Const, SumKernel, ProdKernel, Masked,
                      FixedKernel, fix, flatten)
from .means import Mean, MeanZero, MeanConst, MeanLin
from .gpe import GPE, GP, ElasticGPE
from .sparse import FITC, DTC, SoR
from .likelihoods import Likelihood, BernLik, BinLik, ExpLik, GaussLik, PoisLik, StuTLik
from .gpa import GPA
from . import dist
