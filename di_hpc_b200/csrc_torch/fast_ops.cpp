// fast_ops.cpp -- the autograd layer of hpc_rll.rl_utils in C++ (round 2).
//
// Round 1 bound the C ABI with ctypes underneath Python `torch.autograd.Function`s; measured on B200 that host path
// cost ~50 us per forward+backward (argument checks, torch.empty, ctypes marshalling, Python autograd bookkeeping),
// i.e. more than the kernels of the small ops (q_nstep_td: 0.25 ms of kernels per 4.2 M samples; PPO, C51), and it
// held the module-level GAE step at 0.268 ms against 0.2526 ms for the raw ABI (VERDICT r1 item 3).  Here the same
// logic -- checks, output allocation, save-for-backward, the C-ABI call on PyTorch's current stream -- is one C++
// `torch::autograd::Function` per op, and the nn.Modules of di_hpc_b200/rl_utils call straight into it.
// The Python `*Function` classes stay (same names as /root/reference/hpc_rll/rl_utils/*.py) as the ctypes-bound
// twins and are tested against these.
//
// Semantics, argument order and error behaviour follow di_hpc_b200/rl_utils/*.py one to one; nothing here computes.
#include "common.h"

namespace hpcrl {
namespace {

using torch::autograd::AutogradContext;
using torch::autograd::Function;
using torch::autograd::variable_list;
using OptTensor = c10::optional<Tensor>;

inline Tensor opt_f32(const OptTensor& t, const char* name) {
    return (t.has_value() && t->defined()) ? f32(*t, name) : Tensor();
}

// ------------------------------------------------------------------------------------------------ GAE
struct GaeFn : public Function<GaeFn> {
    static Tensor forward(AutogradContext* ctx, const Tensor& value_, const Tensor& reward_, double gamma,
                          double lambda) {
        const Tensor value = f32(value_, "value"), reward = f32(reward_, "reward");
        TORCH_CHECK_VALUE(reward.dim() == 2, "reward must be (T, B)");
        const int64_t T = reward.size(0), B = reward.size(1);
        TORCH_CHECK_VALUE(value.dim() == 2 && value.size(0) == T + 1 && value.size(1) == B, "value must be (T+1, B)=(",
                          T + 1, ", ", B, "), got ", value.sizes());
        c10::cuda::CUDAGuard guard(reward.device());
        Tensor adv = torch::empty_like(reward);
        ck(hpc_rll_gae_forward(fp(value), fp(reward), fpm(adv), T, B, gamma, lambda, cur_stream()), "hpc_rll_gae_forward");
        ctx->saved_data["gamma"] = gamma;
        ctx->saved_data["lambda"] = lambda;
        return adv;
    }
    static variable_list backward(AutogradContext* ctx, variable_list grads) {
        const Tensor g = f32(grads[0], "grad_adv");
        const int64_t T = g.size(0), B = g.size(1);
        c10::cuda::CUDAGuard guard(g.device());
        Tensor gv = torch::empty({T + 1, B}, g.options()), gr = torch::empty({T, B}, g.options());
        ck(hpc_rll_gae_backward(fp(g), fpm(gv), fpm(gr), T, B, ctx->saved_data["gamma"].toDouble(),
                                ctx->saved_data["lambda"].toDouble(), cur_stream()),
           "hpc_rll_gae_backward");
        return {gv, gr, Tensor(), Tensor()};
    }
};

// ------------------------------------------------------------------------------------------------ TD(lambda)
struct TdLambdaFn : public Function<TdLambdaFn> {
    static Tensor forward(AutogradContext* ctx, const Tensor& value_, const Tensor& reward_, const OptTensor& weight_,
                          double gamma, double lambda, int64_t global_B) {
        const Tensor value = f32(value_, "value"), reward = f32(reward_, "reward");
        TORCH_CHECK_VALUE(reward.dim() == 2, "reward must be (T, B)");
        const int64_t T = reward.size(0), B = reward.size(1);
        TORCH_CHECK_VALUE(value.dim() == 2 && value.size(0) == T + 1 && value.size(1) == B, "value must be (T+1, B)=(",
                          T + 1, ", ", B, "), got ", value.sizes());
        Tensor weight = opt_f32(weight_, "weight");
        if (weight.defined()) {
            // the reference documents weight as (B,) (rl_utils/td.py:172) though its kernel indexes (T,B)
            // (td_lambda_kernel.h:24): broadcast the documented form
            if (weight.dim() == 1) weight = weight.unsqueeze(0).expand({T, B}).contiguous();
            TORCH_CHECK_VALUE(weight.dim() == 2 && weight.size(0) == T && weight.size(1) == B,
                              "weight must be (T, B) or (B,), got ", weight.sizes());
        }
        c10::cuda::CUDAGuard guard(reward.device());
        Tensor loss = torch::empty({1}, reward.options()), grad_buf = torch::empty_like(reward);
        Tensor ws = workspace(HPC_RLL_OP_TD_LAMBDA, T, B, 0, reward);
        ck(hpc_rll_td_lambda_forward(fp(value), fp(reward), fp(weight), fpm(loss), fpm(grad_buf), T, B, gamma, lambda,
                                     global_B, ws.data_ptr(), ws.numel(), cur_stream()),
           "hpc_rll_td_lambda_forward");
        ctx->save_for_backward({grad_buf});
        return loss;
    }
    static variable_list backward(AutogradContext* ctx, variable_list grads) {
        const Tensor grad_buf = ctx->get_saved_variables()[0];
        const int64_t T = grad_buf.size(0), B = grad_buf.size(1);
        c10::cuda::CUDAGuard guard(grad_buf.device());
        const Tensor g = gscalar(grads[0], grad_buf);
        Tensor gv = torch::empty({T + 1, B}, grad_buf.options());
        ck(hpc_rll_td_lambda_backward(fp(g), fp(grad_buf), fpm(gv), T, B, cur_stream()), "hpc_rll_td_lambda_backward");
        return {gv, Tensor(), Tensor(), Tensor(), Tensor(), Tensor()};
    }
};

// ------------------------------------------------------------------------------------------------ V-trace
struct VtraceFn : public Function<VtraceFn> {
    static variable_list forward(AutogradContext* ctx, const Tensor& target_, const Tensor& behaviour_,
                                 const Tensor& action_, const Tensor& value_, const Tensor& reward_,
                                 const OptTensor& weight_, double gamma, double lambda, double rho_clip, double c_clip,
                                 double rho_pg_clip, int64_t global_B) {
        const Tensor target = f32(target_, "target_output"), behaviour = f32(behaviour_, "behaviour_output");
        const Tensor action = i64(action_, "action"), value = f32(value_, "value"), reward = f32(reward_, "reward");
        TORCH_CHECK_VALUE(target.dim() == 3, "target_output must be (T, B, N)");
        const int64_t T = target.size(0), B = target.size(1), N = target.size(2);
        TORCH_CHECK_VALUE(behaviour.sizes() == target.sizes() && action.dim() == 2 && action.size(0) == T &&
                              action.size(1) == B && reward.sizes() == action.sizes() && value.dim() == 2 &&
                              value.size(0) == T + 1 && value.size(1) == B,
                          "vtrace: inconsistent shapes");
        const Tensor weight = opt_f32(weight_, "weight");
        TORCH_CHECK_VALUE(!weight.defined() || weight.sizes() == reward.sizes(), "weight must be (T, B)");
        c10::cuda::CUDAGuard guard(reward.device());
        Tensor losses = torch::empty({3}, reward.options());
        Tensor pg_coef = torch::empty_like(reward), gv_buf = torch::empty_like(reward);
        Tensor ws = workspace(HPC_RLL_OP_VTRACE, T, B, N, reward);
        ck(hpc_rll_vtrace_forward(fp(target), fp(behaviour), ip(action), fp(value), fp(reward), fp(weight), fpm(losses),
                                  fpm(pg_coef), fpm(gv_buf), T, B, N, gamma, lambda, rho_clip, c_clip, rho_pg_clip,
                                  global_B, ws.data_ptr(), ws.numel(), cur_stream()),
           "hpc_rll_vtrace_forward");
        ctx->save_for_backward({target, action, weight, pg_coef, gv_buf});
        ctx->saved_data["global_B"] = global_B;
        return {losses.slice(0, 0, 1), losses.slice(0, 1, 2), losses.slice(0, 2, 3)};
    }
    static variable_list backward(AutogradContext* ctx, variable_list grads) {
        const auto sv = ctx->get_saved_variables();
        const Tensor &target = sv[0], &action = sv[1], &weight = sv[2], &pg_coef = sv[3], &gv_buf = sv[4];
        const int64_t T = target.size(0), B = target.size(1), N = target.size(2);
        c10::cuda::CUDAGuard guard(pg_coef.device());
        const Tensor g0 = gscalar(grads[0], pg_coef), g1 = gscalar(grads[1], pg_coef), g2 = gscalar(grads[2], pg_coef);
        Tensor gt = torch::empty_like(target), gv = torch::empty({T + 1, B}, pg_coef.options());
        ck(hpc_rll_vtrace_backward(fp(g0), fp(g1), fp(g2), fp(target), ip(action), fp(weight), fp(pg_coef), fp(gv_buf),
                                   fpm(gt), fpm(gv), T, B, N, ctx->saved_data["global_B"].toInt(), cur_stream()),
           "hpc_rll_vtrace_backward");
        variable_list out(12);
        out[0] = gt;
        out[3] = gv;
        return out;
    }
};

// ------------------------------------------------------------------------------------------------ UPGO
struct UpgoFn : public Function<UpgoFn> {
    static Tensor forward(AutogradContext* ctx, const Tensor& target_, const Tensor& rho_, const Tensor& action_,
                          const Tensor& reward_, const Tensor& value_, int64_t global_B) {
        const Tensor target = f32(target_, "target_output"), rho = f32(rho_, "rhos"), action = i64(action_, "action");
        const Tensor reward = f32(reward_, "rewards"), value = f32(value_, "bootstrap_values");
        TORCH_CHECK_VALUE(target.dim() == 3, "target_output must be (T, B, N)");
        const int64_t T = target.size(0), B = target.size(1), N = target.size(2);
        TORCH_CHECK_VALUE(rho.dim() == 2 && rho.size(0) == T && rho.size(1) == B && action.sizes() == rho.sizes() &&
                              reward.sizes() == rho.sizes() && value.dim() == 2 && value.size(0) == T + 1 &&
                              value.size(1) == B,
                          "upgo: inconsistent shapes");
        c10::cuda::CUDAGuard guard(reward.device());
        Tensor loss = torch::empty({1}, reward.options()), coef = torch::empty_like(reward);
        Tensor ws = workspace(HPC_RLL_OP_UPGO, T, B, N, reward);
        ck(hpc_rll_upgo_forward(fp(target), fp(rho), ip(action), fp(reward), fp(value), fpm(loss), fpm(coef), T, B, N,
                                global_B, ws.data_ptr(), ws.numel(), cur_stream()),
           "hpc_rll_upgo_forward");
        ctx->save_for_backward({target, action, coef});
        return loss;
    }
    static variable_list backward(AutogradContext* ctx, variable_list grads) {
        const auto sv = ctx->get_saved_variables();
        const Tensor &target = sv[0], &action = sv[1], &coef = sv[2];
        const int64_t T = target.size(0), B = target.size(1), N = target.size(2);
        c10::cuda::CUDAGuard guard(coef.device());
        const Tensor g = gscalar(grads[0], coef);
        Tensor gt = torch::empty_like(target);
        ck(hpc_rll_upgo_backward(fp(g), fp(target), ip(action), fp(coef), fpm(gt), T, B, N, cur_stream()),
           "hpc_rll_upgo_backward");
        variable_list out(6);
        out[0] = gt;
        return out;
    }
};

// ------------------------------------------------------------------------------------------------ PPO
struct PpoFn : public Function<PpoFn> {
    static variable_list forward(AutogradContext* ctx, const Tensor& logits_new_, const Tensor& logits_old_,
                                 const Tensor& action_, const Tensor& value_new_, const Tensor& value_old_,
                                 const Tensor& adv_, const Tensor& return__, const OptTensor& weight_, double clip_ratio,
                                 bool use_value_clip, double dual_clip, int64_t global_B, const OptTensor& adv_stats_) {
        const Tensor ln = f32(logits_new_, "logits_new"), lo = f32(logits_old_, "logits_old");
        const Tensor action = i64(action_, "action"), vn = f32(value_new_, "value_new"), vo = f32(value_old_, "value_old");
        const Tensor adv = f32(adv_, "adv"), ret = f32(return__, "return_");
        TORCH_CHECK_VALUE(ln.dim() == 2, "logits_new must be (B, N)");
        const int64_t B = ln.size(0), N = ln.size(1);
        auto is_b = [B](const Tensor& t) { return t.dim() == 1 && t.size(0) == B; };
        TORCH_CHECK_VALUE(lo.sizes() == ln.sizes() && is_b(action) && is_b(vn) && is_b(vo) && is_b(adv) && is_b(ret),
                          "ppo: inconsistent shapes");
        const Tensor weight = opt_f32(weight_, "weight");
        TORCH_CHECK_VALUE(!weight.defined() || is_b(weight), "weight must be (B,)");
        const Tensor stats = opt_f32(adv_stats_, "adv_stats");
        TORCH_CHECK_VALUE(!stats.defined() || (stats.dim() == 1 && stats.size(0) == 2),
                          "adv_stats must be (2,) = [mean, std + 1e-8]");
        c10::cuda::CUDAGuard guard(adv.device());
        Tensor out = torch::empty({5}, adv.options());
        Tensor pol_coef = torch::empty({B}, adv.options()), val_coef = torch::empty({B}, adv.options());
        Tensor ws = workspace(HPC_RLL_OP_PPO, 0, B, N, adv);
        if (stats.defined())
            ck(hpc_rll_ppo_forward_norm(fp(ln), fp(lo), ip(action), fp(vn), fp(vo), fp(adv), fp(ret), fp(weight),
                                        fp(stats), fpm(out), fpm(pol_coef), fpm(val_coef), B, N, clip_ratio,
                                        use_value_clip ? 1 : 0, dual_clip, global_B, ws.data_ptr(), ws.numel(),
                                        cur_stream()),
               "hpc_rll_ppo_forward_norm");
        else
            ck(hpc_rll_ppo_forward(fp(ln), fp(lo), ip(action), fp(vn), fp(vo), fp(adv), fp(ret), fp(weight), fpm(out),
                                   fpm(pol_coef), fpm(val_coef), B, N, clip_ratio, use_value_clip ? 1 : 0, dual_clip,
                                   global_B, ws.data_ptr(), ws.numel(), cur_stream()),
               "hpc_rll_ppo_forward");
        ctx->save_for_backward({ln, action, weight, pol_coef, val_coef});
        ctx->saved_data["global_B"] = global_B;
        Tensor info = out.slice(0, 3, 5);
        ctx->mark_non_differentiable({info});
        return {out.slice(0, 0, 1), out.slice(0, 1, 2), out.slice(0, 2, 3), info};
    }
    static variable_list backward(AutogradContext* ctx, variable_list grads) {
        const auto sv = ctx->get_saved_variables();
        const Tensor &ln = sv[0], &action = sv[1], &weight = sv[2], &pol_coef = sv[3], &val_coef = sv[4];
        const int64_t B = ln.size(0), N = ln.size(1);
        c10::cuda::CUDAGuard guard(pol_coef.device());
        const Tensor g0 = gscalar(grads[0], pol_coef), g1 = gscalar(grads[1], pol_coef), g2 = gscalar(grads[2], pol_coef);
        Tensor gl = torch::empty_like(ln), gv = torch::empty({B}, pol_coef.options());
        ck(hpc_rll_ppo_backward(fp(g0), fp(g1), fp(g2), fp(ln), ip(action), fp(weight), fp(pol_coef), fp(val_coef),
                                fpm(gl), fpm(gv), B, N, ctx->saved_data["global_B"].toInt(), cur_stream()),
           "hpc_rll_ppo_backward");
        variable_list out(13);
        out[0] = gl;
        out[3] = gv;
        return out;
    }
};

// ------------------------------------------------------------------------------------------------ n-step family
struct NStepArgs {
    Tensor action, next_n_action, reward, done, weight;
    int64_t T;
};

// shared argument normalisation (di_hpc_b200/rl_utils/td.py:_nstep_common)
NStepArgs nstep_common(const Tensor& action_, const Tensor& next_n_action_, const Tensor& reward_, const Tensor& done_,
                       const OptTensor& weight_, int64_t B) {
    NStepArgs a;
    a.action = i64(action_, "action");
    a.next_n_action = i64(next_n_action_, "next_n_action");
    a.reward = f32(reward_, "reward");
    // the reference kernels read `done` as float* (src/rl_utils/q_nstep_td.cu:39); accept bool too
    a.done = f32(done_.scalar_type() == torch::kFloat32 ? done_ : done_.to(torch::kFloat32), "done");
    auto is_b = [B](const Tensor& t) { return t.dim() == 1 && t.size(0) == B; };
    TORCH_CHECK_VALUE(is_b(a.action) && is_b(a.next_n_action) && is_b(a.done) && a.reward.dim() == 2 &&
                          a.reward.size(1) == B,
                      "n-step td: inconsistent shapes (B=", B, ")");
    a.weight = opt_f32(weight_, "weight");
    TORCH_CHECK_VALUE(!a.weight.defined() || is_b(a.weight), "weight must be (B,)");
    a.T = a.reward.size(0);
    return a;
}

Tensor opt_vec_b(const OptTensor& t, const char* name, int64_t B) {
    Tensor v = opt_f32(t, name);
    TORCH_CHECK_VALUE(!v.defined() || (v.dim() == 1 && v.size(0) == B), name, " must be (B,)");
    return v;
}

struct QNStepFn : public Function<QNStepFn> {
    static variable_list forward(AutogradContext* ctx, const Tensor& q_, const Tensor& nq_, const Tensor& action_,
                                 const Tensor& naction_, const Tensor& reward_, const Tensor& done_,
                                 const OptTensor& weight_, double gamma, bool rescale, int64_t global_B) {
        const Tensor q = f32(q_, "q"), nq = f32(nq_, "next_n_q");
        TORCH_CHECK_VALUE(q.dim() == 2, "q must be (B, N)");
        const int64_t B = q.size(0), N = q.size(1);
        TORCH_CHECK_VALUE(nq.sizes() == q.sizes(), "next_n_q must match q");
        const NStepArgs a = nstep_common(action_, naction_, reward_, done_, weight_, B);
        c10::cuda::CUDAGuard guard(q.device());
        Tensor loss = torch::empty({1}, q.options()), td = torch::empty({B}, q.options()), gb = torch::empty({B}, q.options());
        Tensor ws = workspace(HPC_RLL_OP_Q_NSTEP_TD, a.T, B, N, q);
        ck(hpc_rll_q_nstep_td_forward(fp(q), fp(nq), ip(a.action), ip(a.next_n_action), fp(a.reward), fp(a.done),
                                      fp(a.weight), fpm(loss), fpm(td), fpm(gb), a.T, B, N, gamma, rescale ? 1 : 0,
                                      global_B, ws.data_ptr(), ws.numel(), cur_stream()),
           "hpc_rll_q_nstep_td_forward");
        ctx->save_for_backward({gb, a.action});
        ctx->saved_data["N"] = N;
        ctx->mark_non_differentiable({td});
        return {loss, td};
    }
    static variable_list backward(AutogradContext* ctx, variable_list grads) {
        const auto sv = ctx->get_saved_variables();
        const Tensor &gb = sv[0], &action = sv[1];
        const int64_t B = gb.size(0), N = ctx->saved_data["N"].toInt();
        c10::cuda::CUDAGuard guard(gb.device());
        const Tensor g = gscalar(grads[0], gb);
        Tensor gq = torch::empty({B, N}, gb.options());
        ck(hpc_rll_q_nstep_td_backward(fp(g), fp(gb), ip(action), fpm(gq), B, N, cur_stream()),
           "hpc_rll_q_nstep_td_backward");
        variable_list out(10);
        out[0] = gq;
        return out;
    }
};

struct DistNStepFn : public Function<DistNStepFn> {
    static variable_list forward(AutogradContext* ctx, const Tensor& dist_, const Tensor& ndist_, const Tensor& action_,
                                 const Tensor& naction_, const Tensor& reward_, const Tensor& done_,
                                 const OptTensor& weight_, double gamma, double v_min, double v_max, int64_t global_B) {
        const Tensor dist = f32(dist_, "dist"), ndist = f32(ndist_, "next_n_dist");
        TORCH_CHECK_VALUE(dist.dim() == 3, "dist must be (B, N, n_atom)");
        const int64_t B = dist.size(0), N = dist.size(1), n_atom = dist.size(2);
        TORCH_CHECK_VALUE(ndist.sizes() == dist.sizes(), "next_n_dist must match dist");
        const NStepArgs a = nstep_common(action_, naction_, reward_, done_, weight_, B);
        c10::cuda::CUDAGuard guard(dist.device());
        Tensor loss = torch::empty({1}, dist.options()), td = torch::empty({B}, dist.options());
        Tensor gb = torch::empty({B, n_atom}, dist.options());
        Tensor ws = workspace(HPC_RLL_OP_DIST_NSTEP_TD, a.T, B, N, dist);
        ck(hpc_rll_dist_nstep_td_forward(fp(dist), fp(ndist), ip(a.action), ip(a.next_n_action), fp(a.reward),
                                         fp(a.done), fp(a.weight), fpm(loss), fpm(td), fpm(gb), a.T, B, N, n_atom, gamma,
                                         v_min, v_max, global_B, ws.data_ptr(), ws.numel(), cur_stream()),
           "hpc_rll_dist_nstep_td_forward");
        ctx->save_for_backward({gb, a.action});
        ctx->saved_data["N"] = N;
        ctx->mark_non_differentiable({td});
        return {loss, td};
    }
    static variable_list backward(AutogradContext* ctx, variable_list grads) {
        const auto sv = ctx->get_saved_variables();
        const Tensor &gb = sv[0], &action = sv[1];
        const int64_t B = gb.size(0), n_atom = gb.size(1), N = ctx->saved_data["N"].toInt();
        c10::cuda::CUDAGuard guard(gb.device());
        const Tensor g = gscalar(grads[0], gb);
        Tensor gd = torch::empty({B, N, n_atom}, gb.options());
        ck(hpc_rll_dist_nstep_td_backward(fp(g), fp(gb), ip(action), fpm(gd), B, N, n_atom, cur_stream()),
           "hpc_rll_dist_nstep_td_backward");
        variable_list out(11);
        out[0] = gd;
        return out;
    }
};

struct QrdqnFn : public Function<QrdqnFn> {
    static variable_list forward(AutogradContext* ctx, const Tensor& q_, const Tensor& nq_, const Tensor& action_,
                                 const Tensor& naction_, const Tensor& reward_, const Tensor& done_,
                                 const OptTensor& weight_, const OptTensor& value_gamma_, double gamma,
                                 int64_t global_B) {
        const Tensor q = f32(q_, "q"), nq = f32(nq_, "next_n_q");
        TORCH_CHECK_VALUE(q.dim() == 3, "q must be (B, N, tau)");
        const int64_t B = q.size(0), N = q.size(1), tau = q.size(2);
        TORCH_CHECK_VALUE(nq.sizes() == q.sizes(), "next_n_q must match q");
        const NStepArgs a = nstep_common(action_, naction_, reward_, done_, weight_, B);
        const Tensor vg = opt_vec_b(value_gamma_, "value_gamma", B);
        c10::cuda::CUDAGuard guard(q.device());
        Tensor loss = torch::empty({1}, q.options()), td = torch::empty({B}, q.options());
        Tensor gb = torch::empty({B, tau}, q.options());
        Tensor ws = workspace(HPC_RLL_OP_QRDQN_NSTEP_TD, a.T, B, N, q);
        ck(hpc_rll_qrdqn_nstep_td_forward(fp(q), fp(nq), ip(a.action), ip(a.next_n_action), fp(a.reward), fp(a.done),
                                          fp(a.weight), fp(vg), fpm(loss), fpm(td), fpm(gb), tau, a.T, B, N, gamma,
                                          global_B, ws.data_ptr(), ws.numel(), cur_stream()),
           "hpc_rll_qrdqn_nstep_td_forward");
        ctx->save_for_backward({gb, a.action});
        ctx->saved_data["N"] = N;
        ctx->mark_non_differentiable({td});
        return {loss, td};
    }
    static variable_list backward(AutogradContext* ctx, variable_list grads) {
        const auto sv = ctx->get_saved_variables();
        const Tensor &gb = sv[0], &action = sv[1];
        const int64_t B = gb.size(0), tau = gb.size(1), N = ctx->saved_data["N"].toInt();
        c10::cuda::CUDAGuard guard(gb.device());
        const Tensor g = gscalar(grads[0], gb);
        Tensor gq = torch::empty({B, N, tau}, gb.options());
        ck(hpc_rll_qrdqn_nstep_td_backward(fp(g), fp(gb), ip(action), fpm(gq), tau, B, N, cur_stream()),
           "hpc_rll_qrdqn_nstep_td_backward");
        variable_list out(10);
        out[0] = gq;
        return out;
    }
};

struct IqnFn : public Function<IqnFn> {
    static variable_list forward(AutogradContext* ctx, const Tensor& q_, const Tensor& nq_, const Tensor& action_,
                                 const Tensor& naction_, const Tensor& reward_, const Tensor& done_,
                                 const Tensor& replay_quantiles_, const OptTensor& weight_,
                                 const OptTensor& value_gamma_, double gamma, double kappa, int64_t global_B) {
        const Tensor q = f32(q_, "q"), nq = f32(nq_, "next_n_q"), rq = f32(replay_quantiles_, "replay_quantiles");
        TORCH_CHECK_VALUE(q.dim() == 3, "q must be (tau, B, N)");
        const int64_t tau = q.size(0), B = q.size(1), N = q.size(2);
        TORCH_CHECK_VALUE(nq.dim() == 3 && nq.size(1) == B && nq.size(2) == N, "next_n_q must be (tau', B, N)");
        const int64_t tau_p = nq.size(0);
        TORCH_CHECK_VALUE(rq.numel() == tau * B, "replay_quantiles must hold tau*B values");
        const NStepArgs a = nstep_common(action_, naction_, reward_, done_, weight_, B);
        const Tensor vg = opt_vec_b(value_gamma_, "value_gamma", B);
        c10::cuda::CUDAGuard guard(q.device());
        Tensor loss = torch::empty({1}, q.options()), td = torch::empty({B}, q.options());
        Tensor gb = torch::empty({tau, B}, q.options());
        Tensor ws = workspace(HPC_RLL_OP_IQN_NSTEP_TD, a.T, B, N, q);
        ck(hpc_rll_iqn_nstep_td_forward(fp(q), fp(nq), ip(a.action), ip(a.next_n_action), fp(a.reward), fp(a.done),
                                        fp(rq), fp(a.weight), fp(vg), fpm(loss), fpm(td), fpm(gb), tau, tau_p, a.T, B, N,
                                        gamma, kappa, global_B, ws.data_ptr(), ws.numel(), cur_stream()),
           "hpc_rll_iqn_nstep_td_forward");
        ctx->save_for_backward({gb, a.action});
        ctx->saved_data["N"] = N;
        ctx->mark_non_differentiable({td});
        return {loss, td};
    }
    static variable_list backward(AutogradContext* ctx, variable_list grads) {
        const auto sv = ctx->get_saved_variables();
        const Tensor &gb = sv[0], &action = sv[1];
        const int64_t tau = gb.size(0), B = gb.size(1), N = ctx->saved_data["N"].toInt();
        c10::cuda::CUDAGuard guard(gb.device());
        const Tensor g = gscalar(grads[0], gb);
        Tensor gq = torch::empty({tau, B, N}, gb.options());
        ck(hpc_rll_iqn_nstep_td_backward(fp(g), fp(gb), ip(action), fpm(gq), tau, B, N, cur_stream()),
           "hpc_rll_iqn_nstep_td_backward");
        variable_list out(12);
        out[0] = gq;
        return out;
    }
};

// ------------------------------------------------------------------------------------------------ P2P all-reduce
// all-reduce(SUM) of <= 16 loss scalars over NVLink peer memory (csrc/p2p.cu); gradient = identity.  `bufs_addr` is the
// address of the host array of `world` device pointers held by di_hpc_b200.sharding.P2PScalarAllReduce.
struct P2PAllReduceFn : public Function<P2PAllReduceFn> {
    static Tensor forward(AutogradContext*, const Tensor& x, int64_t bufs_addr, int64_t rank, int64_t world) {
        TORCH_CHECK(x.is_cuda() && x.numel() >= 1 && x.numel() <= 16, "p2p all-reduce takes 1..16 CUDA scalars");
        c10::cuda::CUDAGuard guard(x.device());
        Tensor y = x.detach().to(torch::kFloat32).contiguous().clone();
        ck(hpc_rll_allreduce_scalars_p2p(y.data_ptr<float>(), static_cast<int>(y.numel()),
                                         reinterpret_cast<void* const*>(bufs_addr), static_cast<int>(rank),
                                         static_cast<int>(world), cur_stream()),
           "hpc_rll_allreduce_scalars_p2p");
        return y;
    }
    static variable_list backward(AutogradContext*, variable_list grads) {
        return {grads[0], Tensor(), Tensor(), Tensor()};
    }
};

// ------------------------------------------------------------------------------------------------ ScatterConnection
// x (B,M,N) fp32, location (B,M,2) int64 (y, x) -> out (B,N,H,W), always a fresh tensor; backward needs only location
struct ScatterConnectionFn : public Function<ScatterConnectionFn> {
    static Tensor forward(AutogradContext* ctx, const Tensor& x_, const Tensor& location_, int64_t H, int64_t W,
                          int64_t mode) {
        const Tensor x = f32(x_, "x"), loc = i64(location_, "location");
        TORCH_CHECK_VALUE(x.dim() == 3, "x must be (B, M, N), got ", x.sizes());
        const int64_t B = x.size(0), M = x.size(1), N = x.size(2);
        TORCH_CHECK_VALUE(loc.dim() == 3 && loc.size(0) == B && loc.size(1) == M && loc.size(2) == 2,
                          "location must be (B, M, 2)=(", B, ", ", M, ", 2), got ", loc.sizes());
        TORCH_CHECK(loc.device() == x.device(), "x and location must live on one CUDA device");
        TORCH_CHECK_VALUE(H >= 0 && W >= 0, "H and W must be non-negative");
        c10::cuda::CUDAGuard guard(x.device());
        Tensor out = torch::empty({B, N, H, W}, x.options());
        ck(hpc_rll_scatter_connection_forward(fp(x), ip(loc), fpm(out), B, M, N, H, W, static_cast<int>(mode),
                                              cur_stream()),
           "hpc_rll_scatter_connection_forward");
        ctx->save_for_backward({loc});
        ctx->saved_data["N"] = N;
        return out;
    }
    static variable_list backward(AutogradContext* ctx, variable_list grads) {
        const Tensor loc = ctx->get_saved_variables()[0];
        const Tensor g = f32(grads[0], "grad_out");
        const int64_t B = loc.size(0), M = loc.size(1), N = ctx->saved_data["N"].toInt(), H = g.size(2), W = g.size(3);
        c10::cuda::CUDAGuard guard(g.device());
        Tensor gx = torch::empty({B, M, N}, g.options());
        ck(hpc_rll_scatter_connection_backward(fp(g), ip(loc), fpm(gx), B, M, N, H, W, cur_stream()),
           "hpc_rll_scatter_connection_backward");
        return {gx, Tensor(), Tensor(), Tensor(), Tensor()};
    }
};

}  // namespace

// the ops of hpc_rll.torch_utils.network, in the extension's `_network` submodule (keeps the names of the top-level
// module -- what `hpc_rl_utils` re-exports -- exactly the reference's rl_utils set plus the rl_utils fast ops)
void register_fast_network_ops(pybind11::module& net) {
    net.def("scatter_connection",
            [](const Tensor& x, const Tensor& loc, int64_t H, int64_t W, int64_t mode) {
                return ScatterConnectionFn::apply(x, loc, H, W, mode);
            },
            "ScatterConnection forward (mode 0 cover, 1 add) with autograd -- C++ twin of ScatterConnectionFunction");
}

void register_fast_ops(pybind11::module& m) {
    m.def("allreduce_scalars_p2p",
          [](const Tensor& x, int64_t bufs_addr, int64_t rank, int64_t world) {
              return P2PAllReduceFn::apply(x, bufs_addr, rank, world);
          },
          "all-reduce(SUM) of <= 16 scalars over NVLink peer memory, differentiable (identity gradient)");
    namespace py = pybind11;
    m.def("gae", [](const Tensor& v, const Tensor& r, double g, double l) { return GaeFn::apply(v, r, g, l); },
          "GAE forward with autograd (adjoint) -- C++ twin of GAEFunction");
    m.def("td_lambda",
          [](const Tensor& v, const Tensor& r, const OptTensor& w, double g, double l, int64_t gb) {
              return TdLambdaFn::apply(v, r, w, g, l, gb);
          },
          "TD(lambda) loss with autograd");
    m.def("vtrace",
          [](const Tensor& t, const Tensor& b, const Tensor& a, const Tensor& v, const Tensor& r, const OptTensor& w,
             double g, double l, double rho, double c, double rho_pg, int64_t gb) {
              return VtraceFn::apply(t, b, a, v, r, w, g, l, rho, c, rho_pg, gb);
          },
          "V-trace losses (policy, value, entropy) with autograd");
    m.def("upgo",
          [](const Tensor& t, const Tensor& rho, const Tensor& a, const Tensor& r, const Tensor& v, int64_t gb) {
              return UpgoFn::apply(t, rho, a, r, v, gb);
          },
          "UPGO loss with autograd");
    m.def("ppo",
          [](const Tensor& ln, const Tensor& lo, const Tensor& a, const Tensor& vn, const Tensor& vo, const Tensor& adv,
             const Tensor& ret, const OptTensor& w, double clip, bool vclip, double dual, int64_t gb,
             const OptTensor& stats) { return PpoFn::apply(ln, lo, a, vn, vo, adv, ret, w, clip, vclip, dual, gb, stats); },
          "PPO losses + info (approx_kl, clipfrac as a 2-element device tensor) with autograd");
    m.def("q_nstep_td",
          [](const Tensor& q, const Tensor& nq, const Tensor& a, const Tensor& na, const Tensor& r, const Tensor& d,
             const OptTensor& w, double g, bool rescale, int64_t gb) {
              return QNStepFn::apply(q, nq, a, na, r, d, w, g, rescale, gb);
          },
          "q n-step TD error (optionally with value rescaling) with autograd");
    m.def("dist_nstep_td",
          [](const Tensor& q, const Tensor& nq, const Tensor& a, const Tensor& na, const Tensor& r, const Tensor& d,
             const OptTensor& w, double g, double vmin, double vmax, int64_t gb) {
              return DistNStepFn::apply(q, nq, a, na, r, d, w, g, vmin, vmax, gb);
          },
          "C51 n-step TD error with autograd");
    m.def("qrdqn_nstep_td",
          [](const Tensor& q, const Tensor& nq, const Tensor& a, const Tensor& na, const Tensor& r, const Tensor& d,
             const OptTensor& w, const OptTensor& vg, double g, int64_t gb) {
              return QrdqnFn::apply(q, nq, a, na, r, d, w, vg, g, gb);
          },
          "QR-DQN n-step TD error with autograd");
    m.def("iqn_nstep_td",
          [](const Tensor& q, const Tensor& nq, const Tensor& a, const Tensor& na, const Tensor& r, const Tensor& d,
             const Tensor& rq, const OptTensor& w, const OptTensor& vg, double g, double k, int64_t gb) {
              return IqnFn::apply(q, nq, a, na, r, d, rq, w, vg, g, k, gb);
          },
          "IQN n-step TD error with autograd");
}

}  // namespace hpcrl
