"""mcmc.jl_b200 -- host-side mirror of MCMC.jl's model x sampler x runner interface over libmcmcgpu.so.

The reference is a Julia package (dingliumath/MCMC.jl); no Julia toolchain exists in this image, so
the host side above the C ABI is written in Python with the reference's names, argument meaning and
error behaviour, and the Julia glue a maintainer would add is kept in julia/GPUMC.jl and
INTEGRATION.md.  Everything that computes goes through the CUDA library: there is no CPU path here.

    m = model("logistic", X=X, Y=Y, vars=np.zeros(d), gradient=True)      # likmodel.jl:72-143
    chain = run(m * HMC(2, 0.1) * SerialMC(1000, 10000))                   # MCMC.jl:87, runners.jl:7-11
    batch = run(m * HMCDA(len=0.02) * GPUMC(steps=400, burnin=200, nchains=10000))
    ess(batch), acceptance(chain), var(chain, vtype="bm")                 # src/stats
"""
from .api import (EmpMCTuner, GPUMC, HMC, HMCDA, MALA, NUTS, MCMCChain, MCMCChainBatch, MCMCLikelihoodModel, MCMCTask,
                  RAM, RWM, SerialMC, SeqMC, SerialTempMC, acceptance, actime, describe, linearZv, quadraticZv, ess, mean, mean_rb, model, prun, resume, run, std, var,
                  default_context, set_default_device, shard_rows, init_row_sharding, broadcast_unique_id)
from ._capi import MCMCGPUError, LIB_PATH

__all__ = ["model", "MCMCLikelihoodModel", "RWM", "RAM", "MALA", "HMC", "HMCDA", "NUTS", "EmpMCTuner", "SerialMC", "GPUMC", "SeqMC", "SerialTempMC",
           "MCMCTask", "MCMCChain", "MCMCChainBatch", "run", "prun", "resume", "mean", "mean_rb", "var", "std", "ess", "actime",
           "acceptance", "describe", "linearZv", "quadraticZv", "MCMCGPUError", "LIB_PATH", "default_context", "set_default_device", "shard_rows", "init_row_sharding",
           "broadcast_unique_id"]
