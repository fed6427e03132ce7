# SubspaceInferenceB200.jl — thin `ccall` shim over libssi.so (include/ssi.h).
#
# Keeps the reference's Julia-visible signatures for the accelerated path:
#   subspace_construction(model, cost, data, opt; T, c, M, print_freq)      src/subspace_construction.jl:26
#   sub_inference(in_model, data, W_swa, P; σ_z, σ_m, σ_p, itr, M, alg, backend)   src/space_inference.jl:82-84
#   subspace_inference(model, cost, data, opt; ...)                         src/space_inference.jl:33-35
#   inference = sub_inference, alg=:mh ≡ :rwmh                              README.md:153-154
# Everything numeric goes through the C ABI; there is no CUDA.jl code generation and no CPU
# fallback.  NOT EXECUTED in the build container (no Julia toolchain there): the same ABI is
# exercised by the Python ctypes mirror in subspaceinference.jl_b200/ and by tests/.
module SubspaceInferenceB200

using Flux
using Flux: Data.DataLoader

export subspace_construction, subspace_inference, sub_inference, inference, predictive,
       auto_encoder_subspace, auto_inference, autoencoder_inference

const libssi = get(ENV, "LIBSSI", joinpath(@__DIR__, "..", "lib", "libssi.so"))

const TERM_LL, TERM_PRIOR_W, TERM_PRIOR_Z = UInt32(1), UInt32(2), UInt32(4)

# ---- plumbing ------------------------------------------------------------------------------
# Ctx(0): one device.  Ctx([0, 1, ..., 7]): ONE context over several devices (ssi_ctx_create_multi) -- this single Julia
# process then drives all of them: W_swa, P, X, Y are replicated, the batched calls shard their samples / chains, every
# device lands its slice in the host arrays.  No MPI.jl / NCCL.jl is needed on the Julia side.
mutable struct Ctx
    h::Ptr{Cvoid}
    function Ctx(device::Union{Integer, AbstractVector{<:Integer}} = 0)
        out = Ref{Ptr{Cvoid}}(C_NULL)
        rc = device isa Integer ?
            ccall((:ssi_ctx_create, libssi), Cint, (Cint, Ref{Ptr{Cvoid}}), device, out) :
            ccall((:ssi_ctx_create_multi, libssi), Cint, (Ptr{Int32}, Int32, Ref{Ptr{Cvoid}}), Int32.(device), length(device), out)
        rc == 0 || throw(unsafe_string(ccall((:ssi_last_error, libssi), Cstring, (Ptr{Cvoid},), C_NULL)))
        c = new(out[])
        finalizer(x -> ccall((:ssi_ctx_destroy, libssi), Cint, (Ptr{Cvoid},), x.h), c)
        return c
    end
end

# the reference throws Strings (src/space_inference.jl:42,103,162); so does the shim
check(ctx::Ctx, rc) = rc == 0 ? nothing :
    throw(unsafe_string(ccall((:ssi_last_error, libssi), Cstring, (Ptr{Cvoid},), ctx.h)))

act_code(f) = f === identity ? 0 : f === relu ? 1 : f === tanh ? 2 : f === σ ? 3 :
    throw("Error: activation is not supported on the device path")

function describe(model::Chain)
    all(l -> l isa Dense, model.layers) || throw("Error: density function is not avaliable for this model")
    dims = Int32[size(model.layers[1].W, 2); [size(l.W, 1) for l in model.layers]...]
    acts = Int32[act_code(l.σ) for l in model.layers]
    return dims, acts
end

# same as the reference's extract_params (src/libs.jl:19-22): Flux.destructure order
flat_params(model) = Float32.(first(Flux.destructure(model)))

function set_problem!(ctx::Ctx, model::Chain, data, W_swa, P)
    dims, acts = describe(model)
    check(ctx, ccall((:ssi_set_model, libssi), Cint, (Ptr{Cvoid}, Cint, Ptr{Int32}, Ptr{Int32}),
                     ctx.h, length(acts), dims, acts))
    X = Matrix{Float32}(data.data[1]); Y = Matrix{Float32}(data.data[2])        # split_data, src/libs.jl:75-77
    check(ctx, ccall((:ssi_set_data, libssi), Cint, (Ptr{Cvoid}, Ptr{Float32}, Ptr{Float32}, Int64),
                     ctx.h, X, Y, size(X, 2)))
    Wf = Vector{Float32}(W_swa); Pf = Matrix{Float32}(P)                          # Float64 -> Float32 (documented, SURVEY Q7)
    check(ctx, ccall((:ssi_set_subspace, libssi), Cint, (Ptr{Cvoid}, Ptr{Float32}, Ptr{Float32}, Int64, Int32),
                     ctx.h, Wf, Pf, length(Wf), size(Pf, 2)))
end

"""density(z) batched: one log-probability per column of Z (M×B).  Replaces the closure at
src/space_inference.jl:90-95."""
function logpost_batch(ctx::Ctx, Z::AbstractMatrix; σ_m = 1.0, σ_p = 1.0, σ_z = 1.0, mask = TERM_LL)
    Zf = Matrix{Float32}(Z); lp = Vector{Float64}(undef, size(Zf, 2))
    check(ctx, ccall((:ssi_logpost_batch, libssi), Cint,
                     (Ptr{Cvoid}, Ptr{Float32}, Int64, Float64, Float64, Float64, UInt32, Ptr{Float64}, Ptr{Float64}),
                     ctx.h, Zf, size(Zf, 2), σ_m, σ_p, σ_z, mask, lp, C_NULL))
    return lp
end

# ssi_hmc_params_t (include/ssi.h): passed by reference, inv_metric a host pointer (C_NULL = identity)
struct HmcParams
    step_size::Float64
    n_leapfrog::Int32
    n_adapts::Int64
    target_accept::Float64
    inv_metric::Ptr{Float64}
end

# alg = :static_hmc: fixed-length HMC (AdvancedHMC's StaticTrajectory, Turing's HMC(ε, n_leapfrog)) with per-chain dual averaging
# of ε over the first n_adapts transitions; the warm-up samples stay in the trace.  Not :hmc, which in the reference is NUTS with
# Stan's windowed adaptation and stays host-side.
function check_hmc(M, n_leapfrog, step_size, n_adapts, target_accept, inv_metric)
    n_leapfrog >= 1 || throw(ArgumentError("n_leapfrog must be >= 1"))
    (isfinite(step_size) && step_size > 0) || throw(ArgumentError("step_size must be positive and finite"))
    n_adapts >= 0 || throw(ArgumentError("n_adapts must be >= 0"))
    0 < target_accept < 1 || throw(ArgumentError("target_accept must be in (0, 1)"))
    inv_metric === nothing || (length(inv_metric) == M && all(x -> isfinite(x) && x > 0, inv_metric)) ||
        throw(ArgumentError("inv_metric must hold M positive finite values"))
end

function run_static_hmc(ctx::Ctx, M, n_chains, itr, seed, σ_z, σ_m, σ_p, prior_mask, n_leapfrog, step_size, n_adapts,
                        target_accept, inv_metric)
    zt = Array{Float32}(undef, M, n_chains, itr); lp = Matrix{Float64}(undef, n_chains, itr)
    minv = inv_metric === nothing ? nothing : Vector{Float64}(inv_metric)
    GC.@preserve minv begin
        hp = Ref(HmcParams(step_size, n_leapfrog, n_adapts, target_accept, minv === nothing ? C_NULL : pointer(minv)))
        check(ctx, ccall((:ssi_hmc_run, libssi), Cint,
                         (Ptr{Cvoid}, Int64, Int64, UInt64, Int64, Int64, Ref{HmcParams}, Float64, Float64, Float64, UInt32,
                          Ptr{Float32}, Ptr{Float64}, Ptr{Float32}, Ptr{Float64}, Ptr{UInt8}, Ptr{Float64}),
                         ctx.h, n_chains, itr, seed, 0, 0, hp, σ_z, σ_m, σ_p, prior_mask, C_NULL, C_NULL, zt, lp, C_NULL, C_NULL))
    end
    return zt, lp
end

# ---- public API ---------------------------------------------------------------------------------
# l_pi_grad(theta) = (density(theta), gradient(density, theta))  (src/space_inference.jl:107), batched over the columns of Z:
# what AdvancedHMC's Hamiltonian(metric, density, l_pi_grad) (:146) needs, one reverse pass instead of ForwardDiff's M forward passes.
function logpost_grad(ctx::Ctx, Z::AbstractMatrix; σ_m = 1.0, σ_p = 1.0, σ_z = 1.0, mask = TERM_LL)
    B = size(Z, 2); lp = Vector{Float64}(undef, B); g = Matrix{Float64}(undef, size(Z, 1), B)
    check(ctx, ccall((:ssi_logpost_grad_batch, libssi), Cint,
                     (Ptr{Cvoid}, Ptr{Float32}, Int64, Float64, Float64, Float64, UInt32, Ptr{Float64}, Ptr{Float64}),
                     ctx.h, Float32.(Z), B, σ_m, σ_p, σ_z, mask, lp, g))
    return lp, g
end

# device_train = true keeps the mini-batch step itself on the device (ssi_train_*; cost must be mse(model(x), y), opt Descent or
# ADAM): snapshots then go device-to-device into the SWA recurrence.  Mini-batches are contiguous windows of the data set
# (a DataLoader without shuffle); pass index vectors to ssi_train_step for a shuffled one.
function subspace_construction(model, cost, data, opt; T = 10, c = 1, M = 3, print_freq = 1,
                               ctx::Ctx = Ctx(), device_train::Bool = false)
    training_loss = 0.0
    ps = Flux.params(model)
    n = length(flat_params(model))
    check(ctx, ccall((:ssi_swa_begin, libssi), Cint, (Ptr{Cvoid}, Int64, Int64), ctx.h, n, max(1, div(T, c) * length(data))))
    if device_train
        # the device step walks contiguous windows of the data set: a shuffled loader would silently train on other batches
        data.shuffle && throw("Error: device_train needs a DataLoader without shuffle (pass index vectors to ssi_train_step otherwise)")
        dims, acts = describe(model)
        check(ctx, ccall((:ssi_set_model, libssi), Cint, (Ptr{Cvoid}, Cint, Ptr{Int32}, Ptr{Int32}), ctx.h, length(acts), dims, acts))
        X = Matrix{Float32}(data.data[1]); Y = Matrix{Float32}(data.data[2]); N = size(X, 2)
        check(ctx, ccall((:ssi_set_data, libssi), Cint, (Ptr{Cvoid}, Ptr{Float32}, Ptr{Float32}, Int64), ctx.h, X, Y, N))
        kind, β = opt isa Flux.ADAM ? (Int32(1), opt.beta) : (Int32(0), (0.9, 0.999))
        check(ctx, ccall((:ssi_train_begin, libssi), Cint, (Ptr{Cvoid}, Ptr{Float32}, Int32, Float64, Float64, Float64),
                         ctx.h, flat_params(model), kind, opt.eta, β[1], β[2]))
        loss = Ref{Float64}(0.0)
        for i in 1:T
            for j0 in 0:data.batchsize:(N - 1)
                check(ctx, ccall((:ssi_train_step, libssi), Cint, (Ptr{Cvoid}, Ptr{Int64}, Int64, Int64, Ptr{Float64}),
                                 ctx.h, C_NULL, j0, min(data.batchsize, N - j0), loss))             # was :39-43
                mod(i, c) == 0 && check(ctx, ccall((:ssi_train_snapshot, libssi), Cint, (Ptr{Cvoid}, Float64), ctx.h, i / c))
            end
            ((mod(i, print_freq) == 0) || (i == T)) && println("Traing loss: ", loss[], " Epoch: ", i)
        end
        W = Vector{Float32}(undef, n)
        check(ctx, ccall((:ssi_train_get_weights, libssi), Cint, (Ptr{Cvoid}, Ptr{Float32}), ctx.h, W))
        Flux.loadparams!(model, Flux.params(Flux.destructure(model)[2](W)))
        check(ctx, ccall((:ssi_train_end, libssi), Cint, (Ptr{Cvoid},), ctx.h))
        T = 0
    end
    for i in 1:T
        for d in data
            gs = gradient(ps) do                                  # the SGD step stays in Flux/Zygote (:39-43)
                training_loss = cost(model, d...)
                return training_loss
            end
            Flux.update!(opt, ps, gs)
            if mod(i, c) == 0
                W = flat_params(model)
                check(ctx, ccall((:ssi_swa_push, libssi), Cint, (Ptr{Cvoid}, Ptr{Float32}, Float64), ctx.h, W, i / c))  # n = i/c (:46)
            end
        end
        if (mod(i, print_freq) == 0) || (i == T)
            println("Traing loss: ", training_loss, " Epoch: ", i)
        end
    end
    W_swa = Vector{Float32}(undef, n); P = Matrix{Float32}(undef, n, M)
    check(ctx, ccall((:ssi_swa_finish, libssi), Cint, (Ptr{Cvoid}, Int32, Ptr{Float32}, Ptr{Float32}, Ptr{Float64}, Int32),
                     ctx.h, M, W_swa, P, C_NULL, 0))
    return W_swa, P
end

function sub_inference(in_model, data, W_swa, P; σ_z = 1.0, σ_m = 1.0, σ_p = 1.0, itr = 100, M = 3,
                       alg = :rwmh, backend = :forwarddiff,
                       n_chains = 1, seed = rand(UInt64), prior_mask = TERM_LL, ctx::Ctx = Ctx(),
                       n_leapfrog = 10, step_size = 0.1, n_adapts = div(itr, 2), target_accept = 0.8, inv_metric = nothing)
    # :rwmh / :mh (:113-116), :mala (:117-120) and :static_hmc run on the device; :hmc / :nuts / :advi stay in the reference and
    # can take logpost_grad below as their l_pi_grad (:107)
    (alg == :rwmh || alg == :mh || alg == :mala || alg == :static_hmc) || throw("$alg is not available")            # :162
    alg == :static_hmc && check_hmc(M, n_leapfrog, step_size, n_adapts, target_accept, inv_metric)
    size(P, 2) == M || throw(DimensionMismatch("P has $(size(P, 2)) columns but M = $M"))
    set_problem!(ctx, in_model, data, W_swa, P)
    if alg == :static_hmc
        zt, lp = run_static_hmc(ctx, M, n_chains, itr, seed, σ_z, σ_m, σ_p, prior_mask, n_leapfrog, step_size, n_adapts,
                                target_accept, inv_metric)
    else
        zt = Array{Float32}(undef, M, n_chains, itr); lp = Matrix{Float64}(undef, n_chains, itr)
        check(ctx, ccall((alg == :mala ? :ssi_mala_run : :ssi_mh_run, libssi), Cint,
                         (Ptr{Cvoid}, Int64, Int64, UInt64, Int64, Float64, Float64, Float64, UInt32,
                          Ptr{Float32}, Ptr{Float32}, Ptr{Float64}, Ptr{UInt8}),
                         ctx.h, n_chains, itr, seed, 0, σ_z, σ_m, σ_p, prior_mask, C_NULL, zt, lp, C_NULL))
    end
    if n_chains == 1
        # map(z -> W_swa + P*z.params, chm), map(z -> z.lp, chm)   (:125)
        Wout = Matrix{Float32}(undef, length(W_swa), itr)
        Z = Matrix{Float32}(zt[:, 1, :])
        check(ctx, ccall((:ssi_project, libssi), Cint, (Ptr{Cvoid}, Ptr{Float32}, Int64, Ptr{Float32}), ctx.h, Z, itr, Wout))
        return [Wout[:, t] for t in 1:itr], vec(lp[1, :])
    end
    return zt, lp
end

const inference = sub_inference

# Checkpoint / resume (SURVEY 5; the docs save and reload around sampling, docs/src/nn_example.md:158,168): the chains of the
# last run are resumable from (seed, step, z).  `chain_state` returns their final (z, lp); `continue_chains` draws steps
# step_offset .. step_offset + itr - 1 of the same Philox streams -- bit-identical to an uninterrupted run.
function chain_state(ctx::Ctx, M::Integer, n_chains::Integer)
    z = Matrix{Float32}(undef, M, n_chains); lp = Vector{Float64}(undef, n_chains)
    check(ctx, ccall((:ssi_mh_get_state, libssi), Cint, (Ptr{Cvoid}, Ptr{Float32}, Ptr{Float64}), ctx.h, z, lp))
    return z, lp
end
function continue_chains(ctx::Ctx, z_state::AbstractMatrix, step_offset::Integer, itr::Integer; σ_z = 1.0, σ_m = 1.0, σ_p = 1.0,
                         alg = :rwmh, seed, chain_offset = 0, prior_mask = TERM_LL)
    M, C = size(z_state)
    zt = Array{Float32}(undef, M, C, itr); lp = Matrix{Float64}(undef, C, itr)
    check(ctx, ccall((:ssi_mh_run_from, libssi), Cint,
                     (Ptr{Cvoid}, Int32, Int64, Int64, UInt64, Int64, Int64, Float64, Float64, Float64, UInt32,
                      Ptr{Float32}, Ptr{Float32}, Ptr{Float64}, Ptr{UInt8}),
                     ctx.h, alg == :mala ? 1 : 0, C, itr, seed, chain_offset, step_offset, σ_z, σ_m, σ_p, prior_mask,
                     Matrix{Float32}(z_state), zt, lp, C_NULL))
    return zt, lp
end

# ---- non-linear subspace operator: new_W = W_swa + decoder(z)  (src/space_inference.jl:238-318) ---------------------------------
# auto_encoder_subspace keeps the reference's code (src/subspace_construction.jl:93-143) except that the moment recurrence
# runs on the device; the auto-encoder itself is trained by Flux as in the reference.
function auto_encoder_subspace(model, cost, data, opt, encoder, decoder; T = 10, c = 1, M = 3, print_freq = 1, ctx::Ctx = Ctx())
    training_loss = 0.0
    ps = Flux.params(model)
    n = length(flat_params(model))
    check(ctx, ccall((:ssi_swa_begin, libssi), Cint, (Ptr{Cvoid}, Int64, Int64), ctx.h, n, max(1, div(T, c) * length(data))))
    for i in 1:T
        for d in data
            gs = gradient(ps) do
                training_loss = cost(model, d...)
                return training_loss
            end
            Flux.update!(opt, ps, gs)
            mod(i, c) == 0 && check(ctx, ccall((:ssi_swa_push, libssi), Cint, (Ptr{Cvoid}, Ptr{Float32}, Float64), ctx.h, flat_params(model), i / c))
        end
        ((mod(i, print_freq) == 0) || (i == T)) && println("Traing loss: ", training_loss, " Epoch: ", i)
    end
    K = ccall((:ssi_swa_columns, libssi), Int64, (Ptr{Cvoid},), ctx.h)
    W_swa = Vector{Float32}(undef, n); re_weight = Matrix{Float32}(undef, n, K)
    check(ctx, ccall((:ssi_swa_mean, libssi), Cint, (Ptr{Cvoid}, Ptr{Float32}), ctx.h, W_swa))
    check(ctx, ccall((:ssi_swa_deviations, libssi), Cint, (Ptr{Cvoid}, Ptr{Float32}), ctx.h, re_weight))
    sae = Chain(encoder, decoder)
    autoloss(X) = Flux.mse(sae(X), X)                     # the reference's `+ sum(sqnorm, autops)` line never contributes (:130-131)
    Flux.train!(autoloss, Flux.params(sae), DataLoader(re_weight, batchsize = 5, shuffle = true), ADAM())
    return W_swa, decoder
end

function auto_inference(m, data, decoder, W_swa; σ_z = 1.0, σ_m = 1.0, σ_p = 1.0, itr = 100, M = 3, alg = :hmc,
                        backend = :forwarddiff, n_chains = 1, seed = rand(UInt64), prior_mask = TERM_LL, ctx::Ctx = Ctx(),
                        n_leapfrog = 10, step_size = 0.1, n_adapts = div(itr, 2), target_accept = 0.8, inv_metric = nothing)
    # :316; :hmc/:nuts/:advi stay host-side
    (alg == :rwmh || alg == :mh || alg == :mala || alg == :static_hmc) || throw("$alg is not available")
    alg == :static_hmc && check_hmc(M, n_leapfrog, step_size, n_adapts, target_accept, inv_metric)
    dims, acts = describe(m)
    check(ctx, ccall((:ssi_set_model, libssi), Cint, (Ptr{Cvoid}, Cint, Ptr{Int32}, Ptr{Int32}), ctx.h, length(acts), dims, acts))
    X = Matrix{Float32}(data.data[1]); Y = Matrix{Float32}(data.data[2])
    check(ctx, ccall((:ssi_set_data, libssi), Cint, (Ptr{Cvoid}, Ptr{Float32}, Ptr{Float32}, Int64), ctx.h, X, Y, size(X, 2)))
    ddims, dacts = describe(decoder)
    check(ctx, ccall((:ssi_set_decoder, libssi), Cint, (Ptr{Cvoid}, Ptr{Float32}, Int32, Ptr{Int32}, Ptr{Int32}, Ptr{Float32}),
                     ctx.h, Float32.(W_swa), length(dacts), ddims, dacts, flat_params(decoder)))
    if alg == :static_hmc
        zt, lp = run_static_hmc(ctx, M, n_chains, itr, seed, σ_z, σ_m, σ_p, prior_mask, n_leapfrog, step_size, n_adapts,
                                target_accept, inv_metric)
    else
        zt = Array{Float32}(undef, M, n_chains, itr); lp = Matrix{Float64}(undef, n_chains, itr)
        check(ctx, ccall((alg == :mala ? :ssi_mala_run : :ssi_mh_run, libssi), Cint,
                         (Ptr{Cvoid}, Int64, Int64, UInt64, Int64, Float64, Float64, Float64, UInt32,
                          Ptr{Float32}, Ptr{Float32}, Ptr{Float64}, Ptr{UInt8}),
                         ctx.h, n_chains, itr, seed, 0, σ_z, σ_m, σ_p, prior_mask, C_NULL, zt, lp, C_NULL))
    end
    n_chains == 1 || return zt, lp
    Wout = Matrix{Float32}(undef, length(W_swa), itr)          # map(z -> W_swa + decoder(z.params), chm)  (:277)
    check(ctx, ccall((:ssi_project, libssi), Cint, (Ptr{Cvoid}, Ptr{Float32}, Int64, Ptr{Float32}), ctx.h, Matrix{Float32}(zt[:, 1, :]), itr, Wout))
    return [Wout[:, t] for t in 1:itr], vec(lp[1, :])
end

function autoencoder_inference(model, cost, data, opt, encoder, decoder; σ_z = 1.0, σ_m = 1.0, σ_p = 1.0, itr = 1000, T = 25, c = 1,
                               M = 20, print_freq = 1, alg = :hmc, backend = :forwarddiff, kw...)
    ctx = Ctx()
    W_swa, decoder = auto_encoder_subspace(model, cost, data, opt, encoder, decoder; T = T, c = c, M = M, print_freq = print_freq, ctx = ctx)
    return auto_inference(model, data, decoder, W_swa; σ_z = σ_z, σ_m = σ_m, σ_p = σ_p, itr = itr, M = M, alg = alg,
                          backend = backend, ctx = ctx, kw...)
end

# The sweep of docs/src/nn_example.md:207-216 + src/plotting.jl:8-9 on the device: trajectories[:, :, i] = re(W_swa + P z_i)(inp),
# their mean and (corrected) std over the samples.  Z is M x B (subspace samples), inp is in0 x Ng.
function predictive(in_model, W_swa, P, Z::AbstractMatrix, inp::AbstractMatrix; ctx::Ctx = Ctx(), trajectories::Bool = true)
    dims, acts = describe(in_model)
    check(ctx, ccall((:ssi_set_model, libssi), Cint, (Ptr{Cvoid}, Cint, Ptr{Int32}, Ptr{Int32}), ctx.h, length(acts), dims, acts))
    check(ctx, ccall((:ssi_set_subspace, libssi), Cint, (Ptr{Cvoid}, Ptr{Float32}, Ptr{Float32}, Int64, Int32),
                     ctx.h, Float32.(W_swa), Float32.(P), length(W_swa), size(P, 2)))
    O, Ng, B = Int(dims[end]), size(inp, 2), size(Z, 2)
    traj = trajectories ? Array{Float32}(undef, O, Ng, B) : nothing
    μ = Matrix{Float64}(undef, O, Ng); σ = Matrix{Float64}(undef, O, Ng)
    check(ctx, ccall((:ssi_predict_batch, libssi), Cint,
                     (Ptr{Cvoid}, Ptr{Float32}, Int64, Ptr{Float32}, Int64, Ptr{Float32}, Ptr{Float64}, Ptr{Float64}),
                     ctx.h, Float32.(Z), B, Float32.(inp), Ng, trajectories ? traj : C_NULL, μ, σ))
    return traj, μ, σ
end

function subspace_inference(model, cost, data, opt; σ_z = 1.0, σ_m = 1.0, σ_p = 1.0, itr = 1000, T = 25, c = 1,
                            M = 20, print_freq = 1, alg = :rwmh, backend = :forwarddiff, method = :subspace, kw...)
    method == :subspace || throw("Error: No method found")                        # :42 (diffusion_subspace is outside the device path)
    ctx = Ctx()
    W_swa, P = subspace_construction(model, cost, data, opt; T = T, c = c, M = M, print_freq = print_freq, ctx = ctx)
    chn, lp = sub_inference(model, data, W_swa, P; σ_z = σ_z, σ_m = σ_m, σ_p = σ_p, itr = itr, M = M, alg = alg,
                            backend = backend, ctx = ctx, kw...)
    return chn, lp, W_swa
end

end # module
