# GPUMC.jl -- the Julia-side glue a maintainer of MCMC.jl would add to plug libmcmcgpu.so in as a runner.
#
# Written against include/mcmcgpu.h in the dialect the package itself uses (Julia 0.2: `immutable`,
# `Union(...)`, `Array(T, n)`).  No Julia toolchain exists in the build image, so this file has never been
# executed here; mcmc.jl_b200/_capi.py makes exactly the same calls with the same column-major buffers
# through ctypes and is what the test-suite drives.
#
# Where it hooks in (reference file:line):
#   * include("runners/GPUMC.jl") next to the other runners          src/MCMC.jl:100-103
#   * run(t::MCMCTask) gets a GPUMC branch                            src/runners/runners.jl:7-11
#   * run(t::Array{MCMCTask}) gets a GPUMC branch                     src/runners/runners.jl:17-32
#   * models carry a family tag + data (GPUFamily) besides closures   src/modellers/likmodel.jl:20-58

export GPUMC, gpumodel

const libmcmcgpu = "libmcmcgpu"

immutable GPUMC <: MCMCRunner
  burnin::Int
  thinning::Int
  len::Int
  r::Range
  nchains::Int
  seed::Uint64
  storegradients::Bool

  function GPUMC(steps::Range{Int}, nchains::Int, seed::Integer, storegradients::Bool)
    burnin = first(steps)-1
    thinning = steps.step
    len = last(steps)
    @assert burnin >= 0 "Burnin rounds ($burnin) should be >= 0"
    @assert len > burnin "Total MCMC length ($len) should be > to burnin ($burnin)"
    @assert thinning >= 1 "Thinning ($thinning) should be >= 1"
    @assert nchains >= 1
    new(burnin, thinning, len, steps, nchains, uint64(seed), storegradients)
  end
end
GPUMC(; steps::Int=100, burnin::Int=0, thinning::Int=1, nchains::Int=1, seed::Integer=0, storegradients::Bool=true) =
  GPUMC((burnin+1):thinning:steps, nchains, seed, storegradients)

# family tag + data attached to a model built by gpumodel(...)
immutable GPUFamily
  family::Int32            # MCMCGPU_FAM_*
  X::Matrix{Float64}       # N x d column-major (Julia native), or 0 x 0
  y::Vector{Float64}
  hyper::Vector{Float64}
end
const gpufamilies = ObjectIdDict()   # MCMCLikelihoodModel -> GPUFamily

# e.g. gpumodel(:logistic, X, Y, zeros(nbeta)) == the model of examples/logistic_regression.jl:16-22,
# with the usual CPU closures kept (so SerialMC still works on it) plus the family tag for GPUMC
function gpumodel(family::Symbol, X::Matrix{Float64}, y::Vector{Float64}, init::Vector{Float64}; hyper=Float64[], cpumodel=nothing)
  code = [:normal=>0, :normal_dsl=>1, :linear=>2, :logistic=>3, :probit=>4, :ou=>5][family]
  m = cpumodel == nothing ? model(v -> error("CPU closure not supplied"), init=init) : cpumodel
  gpufamilies[m] = GPUFamily(int32(code), X, y, hyper)
  m
end

check(rc::Int32) = rc == 0 || error(bytestring(ccall((:mcmcgpu_last_error, libmcmcgpu), Ptr{Uint8}, ())))

type SamplerCfg   # mirrors mcmcgpu_sampler_cfg field for field
  kind::Int32; nleaps::Int32; scale::Float64
  rate::Float64; len::Float64; shrinkage::Float64; t0::Float64; step::Float64
  max_leaps::Int64; tuner_on::Int32; adapt_step::Int32; max_step::Int32
  target_path::Float64; target_rate::Float64
end
type RunnerCfg    # mirrors mcmcgpu_runner_cfg
  first::Int64; step::Int64; last::Int64; nchains::Int64; chain_offset::Int64; seed::Uint64
  init_per_chain::Int32; store_grad::Int32; store_logtarget::Int32; engine::Int32; store_rb::Int32
  stream_stats::Int32; stream_batchlen::Int32
end

tunercfg(t) = isa(t, EmpMCTuner) ? (int32(1), int32(t.adaptStep), int32(t.maxStep), t.targetPath, t.targetRate) :
                                   (int32(0), int32(0), int32(0), 0., 0.)
samplercfg(s::RWM)   = SamplerCfg(0, 0, s.scale, 0., 0., 0., 0., 0., 0, 0, 0, 0, 0., 0.)
samplercfg(s::MALA)  = SamplerCfg(1, 0, s.driftStep, 0., 0., 0., 0., 0., 0, tunercfg(s.tuner)...)
samplercfg(s::HMC)   = SamplerCfg(2, s.nLeaps, s.leapStep, 0., 0., 0., 0., 0., 0, tunercfg(s.tuner)...)
samplercfg(s::HMCDA) = SamplerCfg(3, 0, 0., s.rate, s.len, s.shrinkage, s.t0, s.step, 0, 0, 0, 0, 0., 0.)
samplercfg(s::RAM)   = SamplerCfg(4, 0, s.scale, s.rate, 0., 0., 0., 0., 0, 0, 0, 0, 0., 0.)
# NUTS: nleaps = maxdoublings; rate / shrinkage / t0 / step = the dual averaging (include/mcmcgpu.h, MCMCGPU_NUTS)
samplercfg(s::NUTS)  = SamplerCfg(5, s.maxdoublings, 0., s.rate, 0., s.shrinkage, s.t0, s.step, 0, 0, 0, 0, 0., 0.)

# NUTS's diagonal metric on a run handle (mcmcgpu_run_create), before its first execute.  The NUTS type carries
#   invmetric::Union(Nothing, Array{Float64})   # d, or d x nchains; nothing = the identity
#   adaptmetric::Bool; initbuffer::Int; termbuffer::Int; window::Int   # Stan's windows, defaults 75 / 50 / 25
#   metric::Symbol                              # :diag, or :dense with invmetric d x d / d x d x nchains (nothing = I)
#   transition::Symbol                          # :slice (default), or :multinomial (Stan's transition)
function nuts_metric!(run::Ptr{Void}, s::NUTS)
  if s.transition == :multinomial
    check(ccall((:mcmcgpu_run_set_nuts_transition, libmcmcgpu), Int32, (Ptr{Void}, Int32), run, 1))
  end
  if s.metric == :dense
    check(ccall((:mcmcgpu_run_set_dense_metric, libmcmcgpu), Int32, (Ptr{Void}, Ptr{Float64}, Int32),
                run, s.invmetric == nothing ? C_NULL : s.invmetric, s.invmetric != nothing && ndims(s.invmetric) == 3 ? 1 : 0))
  elseif s.invmetric != nothing
    check(ccall((:mcmcgpu_run_set_metric, libmcmcgpu), Int32, (Ptr{Void}, Ptr{Float64}, Int32),
                run, s.invmetric, ndims(s.invmetric) == 2 ? 1 : 0))
  end
  if s.adaptmetric
    check(ccall((:mcmcgpu_run_set_metric_adaptation, libmcmcgpu), Int32, (Ptr{Void}, Int64, Int64, Int64),
                run, s.initbuffer, s.termbuffer, s.window))
  end
end
# the d x nchains inverse metric of a run (after execute: the adapted one)
function nuts_metric(run::Ptr{Void}, d::Int, nchains::Int)
  out = Array(Float64, d, nchains)
  check(ccall((:mcmcgpu_run_get_metric, libmcmcgpu), Int32, (Ptr{Void}, Ptr{Float64}), run, out))
  out
end
# the d x d x nchains dense inverse metric of a run with metric = :dense
function nuts_dense_metric(run::Ptr{Void}, d::Int, nchains::Int)
  out = Array(Float64, d, d, nchains)
  check(ccall((:mcmcgpu_run_get_dense_metric, libmcmcgpu), Int32, (Ptr{Void}, Ptr{Float64}), run, out))
  out
end

# multinomial NUTS: the accept_stat, energy and divergence flag of every kept step, S x nchains each
function nuts_stats(run::Ptr{Void}, S::Int, nchains::Int)
  acc, energy, div = Array(Float64, S, nchains), Array(Float64, S, nchains), Array(UInt8, S, nchains)
  check(ccall((:mcmcgpu_run_fetch_nuts_stats, libmcmcgpu), Int32, (Ptr{Void}, Ptr{Float64}, Ptr{Float64}, Ptr{UInt8}),
              run, acc, energy, div))
  acc, energy, div .!= 0
end

function run_gpumc(t::MCMCTask)
  tic()
  m, r = t.model, t.runner
  fam = gpufamilies[m]
  ctx = Array(Ptr{Void}, 1); mdl = Array(Ptr{Void}, 1)
  check(ccall((:mcmcgpu_init, libmcmcgpu), Int32, (Int32, Ptr{Ptr{Void}}), -1, ctx))
  N = length(fam.y)
  check(ccall((:mcmcgpu_model_create, libmcmcgpu), Int32,
              (Ptr{Void}, Int32, Int64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int32, Int32, Ptr{Ptr{Void}}),
              ctx[1], fam.family, N, m.size, fam.X, fam.y, fam.hyper, length(fam.hyper), 0, mdl))
  S = length(r.r); C = r.nchains; d = m.size
  samples = Array(Float64, d, S, C); grads = Array(Float64, d, S, C)
  accept = Array(Uint8, S, C); logtarget = Array(Float64, S, C)
  scfg = samplercfg(t.sampler)
  rcfg = RunnerCfg(first(r.r), r.r.step, last(r.r), C, 0, r.seed, 0, r.storegradients, 1, 0, 0, 0, 0)
  info = Array(Float64, 5)
  rc = ccall((:mcmcgpu_run_chains, libmcmcgpu), Int32,
             (Ptr{Void}, Ptr{SamplerCfg}, Ptr{RunnerCfg}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
              Ptr{Float64}, Ptr{Float64}, Ptr{Uint8}, Ptr{Float64}, Ptr{Void}),
             mdl[1], &scfg, &rcfg, m.init, m.scale, C_NULL, C_NULL, samples, grads, accept, logtarget, info)
  rc == -2 && error("Initial values out of model support, try other values")   # RWM.jl:55 etc.
  check(rc)
  ccall((:mcmcgpu_model_destroy, libmcmcgpu), Int32, (Ptr{Void},), mdl[1])
  ccall((:mcmcgpu_destroy, libmcmcgpu), Int32, (Ptr{Void},), ctx[1])
  rt = toq()

  cn = ASCIIString[ "pars.$i" for i in 1:d ]                                   # SerialMC.jl:70-79 (default pmap)
  chains = Array(MCMCChain, C)
  for c in 1:C                                                                 # SerialMC.jl:84
    diags = {"step" => collect(r.r), "accept" => bool(accept[:, c])}
    chains[c] = MCMCChain(r.r, DataFrame(samples[:, :, c]', cn), DataFrame(grads[:, :, c]', cn), diags, t, rt)
  end
  C == 1 ? chains[1] : chains
end

# dispatch: the two lines to add to src/runners/runners.jl
#   run(t::MCMCTask):           elseif isa(t.runner, GPUMC); run_gpumc(t)
#   run(t::Array{MCMCTask}):    elseif isa(lastrunner, GPUMC); map(run_gpumc, t)
