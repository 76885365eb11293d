"""Thin torch-tensor wrappers over the policy C ABI (include/marllb_b200_policy.h).

Tensors are float32, CUDA, contiguous; torch only owns the memory and the stream.
"""
from __future__ import annotations

import ctypes as C

import torch

from .. import _lib
from .._lib import check

ACT_NONE, ACT_RELU, ACT_ABS = 0, 1, 2
_bound = False


def _L():
    global _bound
    L = _lib.load()
    if not _bound:
        vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float
        sig = {
            "mlb_gemm": [vp, i64, i64, i64, vp, i64, i64, i64, vp, i64, i64, vp, i64, i32, i32, i32, i32, f32, i32, vp],
            "mlb_linear_tc_supported": [i32, i32, i32, i64, i64, i64],
            "mlb_gemm_tc_supported": [vp, i64, i64, vp, i64, i64, vp, i64, i32, i32, i32],
            "mlb_gemm_tc": [vp, i64, i64, vp, i64, i64, vp, i64, vp, i32, i32, i32, f32, i32, vp],
            "mlb_linear_tc": [vp, i64, vp, i64, vp, vp, i64, i32, i32, i32, i32, vp],
            "mlb_gru_gates_forward": [vp, vp, vp, vp, vp, i32, i32, vp],
            "mlb_gru_gates_backward": [vp, vp, vp, vp, vp, vp, vp, i32, i32, vp],
            "mlb_relu_backward": [vp, vp, vp, i64, vp],
            "mlb_abs_backward": [vp, vp, vp, i64, vp],
            "mlb_colsum": [vp, vp, i32, i32, i64, f32, vp],
            "mlb_axpby": [f32, vp, f32, vp, i64, vp],
            "mlb_sumsq": [vp, i64, vp, vp],
            "mlb_scale": [vp, i64, vp, f32, vp],
            "mlb_adam": [vp, vp, vp, vp, i64, f32, f32, f32, f32, i32, vp],
            "mlb_adam_dev": [vp, vp, vp, vp, i64, f32, f32, f32, f32, vp, vp, vp],
            "mlb_egreedy_select": [vp, vp, vp, f32, vp, vp, i32, i32, vp],
            "mlb_row_max": [vp, vp, vp, i32, i32, vp],
            "mlb_onehot_action": [vp, i32, i32, i32, C.c_uint8, C.c_uint8, vp, vp],
            "mlb_mixer_forward": [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp],
            "mlb_mixer_backward": [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp],
            "mlb_tanh_gaussian_forward": [vp, vp, vp, f32, f32, f32, f32, vp, vp, vp, i32, i32, vp],
            "mlb_tanh_gaussian_backward": [vp, vp, vp, f32, f32, f32, vp, vp, vp, vp, i32, i32, vp],
            "mlb_abs_forward": [vp, vp, i64, vp],
            "mlb_qmix_td_loss": [vp, vp, vp, vp, vp, f32, vp, vp, vp, i32, i32, vp],
            "mlb_sac_q_target": [vp, vp, vp, vp, vp, vp, f32, vp, i32, vp],
            "mlb_mse_loss": [vp, vp, vp, vp, i32, vp],
            "mlb_sac_policy_loss": [vp, vp, vp, vp, vp, vp, vp, vp, i32, vp],
            "mlb_sac_alpha_loss": [vp, vp, f32, vp, vp, i32, vp],
            "mlb_exp_scalar": [vp, vp, vp],
            "mlb_softmax_forward": [vp, vp, i64, i32, vp],
            "mlb_softmax_backward": [vp, vp, vp, i64, i32, vp],
            "mlb_concat_onehot": [vp, vp, vp, i64, i32, i32, i32, vp],
            "mlb_categorical": [vp, vp, vp, vp, vp, vp, i64, i32, vp],
            "mlb_logprob_backward": [vp, vp, vp, vp, i64, i32, i32, vp],
            "mlb_scatter_class": [vp, vp, vp, i64, i32, vp],
            "mlb_td_lambda_targets": [vp, vp, vp, f32, f32, i32, i32, vp],
            "mlb_weighted_sum_forward": [vp, vp, vp, i32, i32, vp],
            "mlb_weighted_sum_backward": [vp, vp, vp, vp, vp, i32, i32, vp],
            "mlb_reward_normalize": [vp, vp, f32, i32, i32, vp],
            "mlb_dsac_q_target": [vp, vp, vp, vp, vp, f32, vp, i32, vp],
            "mlb_gru_seq_forward": [vp] * 8 + [i32] * 3 + [vp],
            "mlb_gru_seq_backward": [vp] * 8 + [i32] * 3 + [vp],
            "mlb_replay_push": [vp] * 13 + [i32] * 5 + [vp],
            "mlb_replay_gather": [vp] * 13 + [i32] * 4 + [vp],
            "mlb_set_workspace_slot": [i32],
            "mlb_get_workspace_slot": [],
            "mlb_reserve_workspace_slots": [i32],
        }
        for name, args in sig.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = C.c_int, args
        _bound = True
    return L


POLICY_EXPORTS = ["mlb_gemm", "mlb_linear_tc_supported", "mlb_linear_tc", "mlb_gemm_tc_supported", "mlb_gemm_tc", "mlb_gru_gates_forward", "mlb_gru_gates_backward", "mlb_relu_backward",
                  "mlb_abs_backward", "mlb_colsum", "mlb_axpby", "mlb_sumsq", "mlb_scale", "mlb_adam", "mlb_adam_dev",
                  "mlb_egreedy_select", "mlb_onehot_action", "mlb_row_max", "mlb_mixer_forward", "mlb_mixer_backward",
                  "mlb_tanh_gaussian_forward", "mlb_tanh_gaussian_backward", "mlb_abs_forward",
                  "mlb_qmix_td_loss", "mlb_sac_q_target", "mlb_mse_loss", "mlb_sac_policy_loss",
                  "mlb_sac_alpha_loss", "mlb_exp_scalar",
                  "mlb_softmax_forward", "mlb_softmax_backward", "mlb_concat_onehot", "mlb_categorical",
                  "mlb_logprob_backward", "mlb_scatter_class", "mlb_td_lambda_targets", "mlb_reward_normalize",
                  "mlb_dsac_q_target", "mlb_weighted_sum_forward", "mlb_weighted_sum_backward",
                  "mlb_replay_push", "mlb_replay_gather", "mlb_gru_seq_forward", "mlb_gru_seq_backward",
                  "mlb_set_workspace_slot", "mlb_get_workspace_slot", "mlb_reserve_workspace_slots"]


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


LAUNCHES = 0   # kernels launched through this module (every op fetches the stream once per launch)


class side_branch:
    """`with side_branch(stream):` -- issue the enclosed ops on `stream`, concurrently with what the caller goes on to
    issue on its own stream, with their own split-K workspace (mlb_set_workspace_slot).  The caller forks before
    (stream.wait_stream(current)) and joins after (current.wait_stream(stream)); under stream capture both become
    graph edges, so the two chains are parallel branches of the CUDA graph."""

    def __init__(self, stream, slot=1):
        self.stream, self.slot = stream, slot

    def __enter__(self):
        L = _L()
        self._prev = L.mlb_get_workspace_slot()
        check(L.mlb_set_workspace_slot(self.slot))
        self._ctx = torch.cuda.stream(self.stream)
        self._ctx.__enter__()
        return self

    def __exit__(self, *exc):
        self._ctx.__exit__(*exc)
        _L().mlb_set_workspace_slot(self._prev)
        return False


def reserve_workspace_slots(n):
    """Slots 1 .. n-1 get the capacity slot 0 has reached (call after an eager single-stream warm-up; nothing can be
    allocated once a stream capture is running)."""
    check(_L().mlb_reserve_workspace_slots(n))


def _st():
    global LAUNCHES
    LAUNCHES += 1
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _chk(t):
    assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous(), "float32 contiguous CUDA tensor required"
    return t


TC_MIN_M = 512   # below this the tile launch overhead beats the FFMA kernel's


def linear_tc(x, W, b=None, act=ACT_NONE, out=None):
    """y = act(x W^T + b) on the tensor cores (tcgen05, 3xTF32).  x [M,K] with unit inner stride
    (rows may be strided, e.g. one agent's slice of [E, A, obs]); W [N,K] contiguous."""
    assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
    _chk(W)
    M, K = x.shape
    N = W.shape[0]
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32, device=x.device)
    check(_L().mlb_linear_tc(_p(x), x.stride(0), _p(W), K, _p(b), _p(out), out.stride(0), M, N, K, act, _st()))
    return out


def linear(x, W, b=None, act=ACT_NONE, out=None):
    """y = act(x W^T + b).  x [M,K] or [G,M,K]; W [N,K] or [G,N,K]; b [N] / [G,N] (nn.Linear layout).
    Large-M 2-D calls go to the tensor-core kernel, the rest to the FFMA GEMM."""
    if (x.dim() == 2 and W.dim() == 2 and x.shape[0] >= TC_MIN_M and x.stride(1) == 1 and x.stride(0) % 4 == 0
            and W.is_contiguous() and x.shape[1] % 4 == 0 and x.data_ptr() % 16 == 0 and W.data_ptr() % 16 == 0
            and (b is None or b.dim() == 1) and (out is None or out.stride(1) == 1)):
        return linear_tc(x, W, b, act, out)
    _chk(x), _chk(W)
    batched = x.dim() == 3
    G = x.shape[0] if batched else 1
    M, K = x.shape[-2], x.shape[-1]
    N = W.shape[-2]
    assert W.shape[-1] == K
    if out is None:
        out = torch.empty((G, M, N) if batched else (M, N), dtype=torch.float32, device=x.device)
    check(_L().mlb_gemm(_p(x), M * K if batched else 0, K, 1,
                        _p(W), N * K if (batched and W.dim() == 3) else 0, 1, K,
                        _p(out), M * N, N, _p(b), N if (b is not None and b.dim() == 2) else 0,
                        M, N, K, G, 0.0, act, _st()))
    return out


def gemm_tc(A, B, out=None, bias=None, beta=0.0, act=ACT_NONE, trans_a=False, trans_b=False):
    """C = act(beta * C + op(A) op(B) + bias) on the tensor cores (mlb_gemm_tc; tests and benchmarks call it directly,
    the layers reach it through mlb_gemm's own dispatch).  A [M,K] (or [K,M] with trans_a), B [K,N] (or [N,K] with
    trans_b = the nn.Linear weight layout), both contiguous."""
    _chk(A), _chk(B)
    M, K = (A.shape[1], A.shape[0]) if trans_a else A.shape
    N = B.shape[0] if trans_b else B.shape[1]
    if out is None:
        out = torch.zeros((M, N), dtype=torch.float32, device=A.device)
    a_rs, a_cs = (1, M) if trans_a else (K, 1)
    b_rs, b_cs = (1, K) if trans_b else (N, 1)
    check(_L().mlb_gemm_tc(_p(A), a_rs, a_cs, _p(B), b_rs, b_cs, _p(out), out.stride(0), _p(bias), M, N, K, beta, act, _st()))
    return out


def matmul_nn(dy, W, out=None, beta=0.0):
    """dx = dy W  (input gradient of nn.Linear).  dy [.,M,N], W [.,N,K] -> [.,M,K]."""
    _chk(dy), _chk(W)
    batched = dy.dim() == 3
    G = dy.shape[0] if batched else 1
    M, N = dy.shape[-2], dy.shape[-1]
    K = W.shape[-1]
    if out is None:
        out = torch.empty((G, M, K) if batched else (M, K), dtype=torch.float32, device=dy.device)
    check(_L().mlb_gemm(_p(dy), M * N if batched else 0, N, 1,
                        _p(W), N * K if (batched and W.dim() == 3) else 0, K, 1,
                        _p(out), M * K, K, None, 0, M, K, N, G, beta, ACT_NONE, _st()))
    return out


def matmul_tn(dy, x, out=None, beta=0.0):
    """dW (+)= dy^T x  (weight gradient of nn.Linear).  dy [.,M,N], x [.,M,K] -> [.,N,K]."""
    _chk(dy), _chk(x)
    batched = dy.dim() == 3
    G = dy.shape[0] if batched else 1
    M, N = dy.shape[-2], dy.shape[-1]
    K = x.shape[-1]
    if out is None:
        out = torch.zeros((G, N, K) if batched else (N, K), dtype=torch.float32, device=dy.device)
        beta = 0.0
    check(_L().mlb_gemm(_p(dy), M * N if batched else 0, 1, N,       # A(n, m) = dy[m][n]
                        _p(x), M * K if batched else 0, K, 1,        # B(m, k) = x[m][k]
                        _p(out), N * K, K, None, 0, N, K, M, G, beta, ACT_NONE, _st()))
    return out


def colsum(dy, out=None, beta=0.0):
    """db (+)= sum over rows.  dy [M,N] (2-D only)."""
    _chk(dy)
    M, N = dy.shape
    if out is None:
        out = torch.empty(N, dtype=torch.float32, device=dy.device)
        beta = 0.0
    check(_L().mlb_colsum(_p(dy), _p(out), M, N, N, beta, _st()))
    return out


def gru_gates_forward(gi, gh, h, save_gates=False):
    M, H = h.shape[-2] * (h.shape[0] if h.dim() == 3 else 1), h.shape[-1]
    h_new = torch.empty_like(h)
    gates = torch.empty_like(gi) if save_gates else None
    check(_L().mlb_gru_gates_forward(_p(_chk(gi)), _p(_chk(gh)), _p(_chk(h)), _p(h_new), _p(gates), M, H, _st()))
    return h_new, gates


def gru_gates_backward(dh_new, gates, h, gh):
    M, H = h.shape[-2] * (h.shape[0] if h.dim() == 3 else 1), h.shape[-1]
    dgi, dgh, dh = torch.empty_like(gates), torch.empty_like(gates), torch.empty_like(h)
    check(_L().mlb_gru_gates_backward(_p(_chk(dh_new)), _p(gates), _p(h), _p(gh), _p(dgi), _p(dgh), _p(dh), M, H, _st()))
    return dgi, dgh, dh


def gru_seq_supported(H):
    return 3 * H <= 1024 and (3 * H * H + 4 * H + 12 * H + 12 * H) * 4 <= 227 * 1024


def gru_seq_forward(gi_all, W_hh, b_hh, h0, save=True):
    """gi_all [T,B,3H] -> hs [T,B,H] (+ hprev, ghs, gates for the backward pass) in one launch."""
    T, B, H3 = gi_all.shape
    H = H3 // 3
    f = dict(dtype=torch.float32, device=gi_all.device)
    hs = torch.empty((T, B, H), **f)
    hprev = torch.empty((T, B, H), **f) if save else None
    ghs = torch.empty((T, B, H3), **f) if save else None
    gates = torch.empty((T, B, H3), **f) if save else None
    check(_L().mlb_gru_seq_forward(_p(_chk(gi_all)), _p(_chk(W_hh)), _p(_chk(b_hh)), _p(_chk(h0)), _p(hs), _p(hprev), _p(ghs),
                                   _p(gates), T, B, H, _st()))
    return hs, hprev, ghs, gates


def gru_seq_backward(dhs, gates, hprev, ghs, W_hh):
    T, B, H = dhs.shape
    dgi = torch.empty_like(gates)
    dgh = torch.empty_like(gates)
    dh0 = torch.empty((B, H), dtype=torch.float32, device=dhs.device)
    check(_L().mlb_gru_seq_backward(_p(_chk(dhs)), _p(_chk(gates)), _p(_chk(hprev)), _p(_chk(ghs)), _p(_chk(W_hh)), _p(dgi), _p(dgh),
                                    _p(dh0), T, B, H, _st()))
    return dgi, dgh, dh0


def relu_backward(y, dy):
    dx = torch.empty_like(dy)
    check(_L().mlb_relu_backward(_p(_chk(y)), _p(_chk(dy)), _p(dx), y.numel(), _st()))
    return dx


def abs_backward(pre, dy):
    dx = torch.empty_like(dy)
    check(_L().mlb_abs_backward(_p(_chk(pre)), _p(_chk(dy)), _p(dx), pre.numel(), _st()))
    return dx


def axpby(a, x, b, y):
    """y = a*x + b*y in place."""
    check(_L().mlb_axpby(a, _p(_chk(x)), b, _p(_chk(y)), x.numel(), _st()))
    return y


def clip_grad_norm_(grads, max_norm):
    """torch.nn.utils.clip_grad_norm_ over a list of gradient tensors; returns the total norm tensor."""
    acc = torch.zeros(1, dtype=torch.float64, device=grads[0].device)
    for g in grads:
        check(_L().mlb_sumsq(_p(_chk(g)), g.numel(), _p(acc), _st()))
    for g in grads:
        check(_L().mlb_scale(_p(g), g.numel(), _p(acc), float(max_norm), _st()))
    return acc.sqrt()


def adam_step(p, g, m, v, lr, step, beta1=0.9, beta2=0.999, eps=1e-8):
    check(_L().mlb_adam(_p(_chk(p)), _p(_chk(g)), _p(_chk(m)), _p(_chk(v)), p.numel(), lr, beta1, beta2, eps, step, _st()))


def adam_step_dev(p, g, m, v, lr, step_dev, coef_dev, beta1=0.9, beta2=0.999, eps=1e-8):
    """Adam step whose step counter lives on the device (int32 [1], advanced here): graph-capturable."""
    check(_L().mlb_adam_dev(_p(_chk(p)), _p(_chk(g)), _p(_chk(m)), _p(_chk(v)), p.numel(), lr, beta1, beta2, eps,
                            _p(step_dev), _p(coef_dev), _st()))


def egreedy_select(q, epsilon=0.0, u=None, rnd=None):
    """q [M,K] -> (action int32 [M], q_sel [M]); u/rnd pre-drawn exploration randoms (optional)."""
    M, K = q.shape
    act = torch.empty(M, dtype=torch.int32, device=q.device)
    qsel = torch.empty(M, dtype=torch.float32, device=q.device)
    check(_L().mlb_egreedy_select(_p(_chk(q)), _p(u), _p(rnd), float(epsilon), _p(act), _p(qsel), M, K, _st()))
    return act, qsel


def onehot_action(action, servers_per_agent, hot=2, cold=0, out=None):
    """QMIX actions [E, A] int32 (one server index per agent) -> env action [E, A*Sa] uint8."""
    assert action.is_cuda and action.dtype == torch.int32 and action.is_contiguous()
    M = action.numel()
    if out is None:
        out = torch.empty((action.shape[0], action.shape[1] * servers_per_agent), dtype=torch.uint8, device=action.device)
    check(_L().mlb_onehot_action(_p(action), M, servers_per_agent, 1, hot, cold, _p(out), _st()))
    return out


def replay_push(ring, pos_dev, state, action, reward, next_state, done, hidden):
    """ring = (state, action, reward, next_state, done, hidden) ring tensors; one launch (+ the position update)."""
    r_state, r_action, r_reward, r_next, r_done, r_hidden = ring
    n = state.shape[0]
    assert reward.dtype == torch.float64 and done.dtype == torch.uint8 and pos_dev.dtype == torch.int64
    for t in (state, action, next_state, hidden):
        _chk(t)
    check(_L().mlb_replay_push(_p(state), _p(action), _p(reward), _p(next_state), _p(done), _p(hidden), _p(r_state),
                               _p(r_action), _p(r_reward), _p(r_next), _p(r_done), _p(r_hidden), _p(pos_dev), n,
                               r_state.shape[0], r_state.shape[1], r_action.shape[1], r_hidden.shape[1], _st()))


def replay_gather(ring, idx):
    r_state, r_action, r_reward, r_next, r_done, r_hidden = ring
    B = idx.numel()
    f = dict(dtype=torch.float32, device=r_state.device)
    out = (torch.empty((B, r_state.shape[1]), **f), torch.empty((B, r_action.shape[1]), **f), torch.empty((B, 1), **f),
           torch.empty((B, r_state.shape[1]), **f), torch.empty((B, 1), **f), torch.empty((B, r_hidden.shape[1]), **f))
    assert idx.dtype == torch.int64 and idx.is_contiguous()
    check(_L().mlb_replay_gather(_p(r_state), _p(r_action), _p(r_reward), _p(r_next), _p(r_done), _p(r_hidden), _p(idx),
                                 _p(out[0]), _p(out[1]), _p(out[2]), _p(out[3]), _p(out[4]), _p(out[5]), B,
                                 r_state.shape[1], r_action.shape[1], r_hidden.shape[1], _st()))
    return out


def row_max(q):
    M, K = q.shape
    out = torch.empty(M, dtype=torch.float32, device=q.device)
    arg = torch.empty(M, dtype=torch.int32, device=q.device)
    check(_L().mlb_row_max(_p(_chk(q)), _p(out), _p(arg), M, K, _st()))
    return out, arg


def mixer_forward(q, w1, b1, w2, b2, save_hidden=False):
    M, A = q.shape
    E = b1.shape[-1]
    q_tot = torch.empty(M, dtype=torch.float32, device=q.device)
    hidden = torch.empty((M, E), dtype=torch.float32, device=q.device) if save_hidden else None
    check(_L().mlb_mixer_forward(_p(_chk(q)), _p(_chk(w1)), _p(_chk(b1)), _p(_chk(w2)), _p(_chk(b2)),
                                 _p(q_tot), _p(hidden), M, A, E, _st()))
    return q_tot, hidden


def mixer_backward(dq_tot, q, w1, w2, hidden):
    M, A = q.shape
    E = hidden.shape[-1]
    dq = torch.empty_like(q)
    dw1 = torch.empty((M, A * E), dtype=torch.float32, device=q.device)
    db1 = torch.empty((M, E), dtype=torch.float32, device=q.device)
    dw2 = torch.empty((M, E), dtype=torch.float32, device=q.device)
    db2 = torch.empty((M, 1), dtype=torch.float32, device=q.device)
    check(_L().mlb_mixer_backward(_p(_chk(dq_tot)), _p(q), _p(w1), _p(w2), _p(hidden), _p(dq), _p(dw1), _p(db1),
                                  _p(dw2), _p(db2), M, A, E, _st()))
    return dq, dw1, db1, dw2, db2


def tanh_gaussian_forward(mean, log_std_raw, eps, lo=-20.0, hi=2.0, scale=1.0, bias=0.0):
    M, A = mean.shape
    action = torch.empty_like(mean)
    mean_action = torch.empty_like(mean)
    logp = torch.empty((M, 1), dtype=torch.float32, device=mean.device)
    check(_L().mlb_tanh_gaussian_forward(_p(_chk(mean)), _p(_chk(log_std_raw)), _p(eps), lo, hi, scale, bias,
                                         _p(action), _p(logp), _p(mean_action), M, A, _st()))
    return action, logp, mean_action


def tanh_gaussian_backward(mean, log_std_raw, eps, d_action, d_logp, lo=-20.0, hi=2.0, scale=1.0):
    M, A = mean.shape
    d_mean, d_ls = torch.empty_like(mean), torch.empty_like(mean)
    check(_L().mlb_tanh_gaussian_backward(_p(mean), _p(log_std_raw), _p(_chk(eps)), lo, hi, scale, _p(d_action),
                                          _p(d_logp), _p(d_mean), _p(d_ls), M, A, _st()))
    return d_mean, d_ls


def abs_forward(x):
    y = torch.empty_like(x)
    check(_L().mlb_abs_forward(_p(_chk(x)), _p(y), x.numel(), _st()))
    return y


def qmix_td_loss(q_tot, target_q_tot, reward_sum, done, seq_len, gamma):
    """[B,T] float32 tensors, seq_len int32 [B] -> (targets, dq_tot, stats float64[3] = loss, mean q_tot, mean targets)."""
    B, T = q_tot.shape
    targets, dq = torch.empty_like(q_tot), torch.empty_like(q_tot)
    stats = torch.zeros(3, dtype=torch.float64, device=q_tot.device)
    check(_L().mlb_qmix_td_loss(_p(_chk(q_tot)), _p(_chk(target_q_tot)), _p(_chk(reward_sum)), _p(_chk(done)),
                                _p(seq_len), float(gamma), _p(targets), _p(dq), _p(stats), B, T, _st()))
    return targets, dq, stats


def sac_q_target(reward, done, q1n, q2n, logp_next, alpha, gamma):
    y = torch.empty_like(reward)
    check(_L().mlb_sac_q_target(_p(_chk(reward)), _p(_chk(done)), _p(_chk(q1n)), _p(_chk(q2n)), _p(_chk(logp_next)),
                                _p(alpha), float(gamma), _p(y), reward.numel(), _st()))
    return y


def mse_loss(q, y):
    dq = torch.empty_like(q)
    loss = torch.zeros(1, dtype=torch.float64, device=q.device)
    check(_L().mlb_mse_loss(_p(_chk(q)), _p(_chk(y)), _p(dq), _p(loss), q.numel(), _st()))
    return loss, dq


def sac_policy_loss(logp, q1, q2, alpha):
    dlp, dq1, dq2 = torch.empty_like(logp), torch.empty_like(q1), torch.empty_like(q2)
    loss = torch.zeros(1, dtype=torch.float64, device=q1.device)
    check(_L().mlb_sac_policy_loss(_p(_chk(logp)), _p(_chk(q1)), _p(_chk(q2)), _p(alpha), _p(dlp), _p(dq1), _p(dq2),
                                   _p(loss), logp.numel(), _st()))
    return loss, dlp, dq1, dq2


def sac_alpha_loss(logp, log_alpha, target_entropy):
    d = torch.empty(1, dtype=torch.float32, device=logp.device)
    loss = torch.zeros(1, dtype=torch.float64, device=logp.device)
    check(_L().mlb_sac_alpha_loss(_p(_chk(logp)), _p(log_alpha), float(target_entropy), _p(d), _p(loss), logp.numel(), _st()))
    return loss, d


def exp_scalar(x, out=None):
    y = torch.empty_like(x) if out is None else out
    check(_L().mlb_exp_scalar(_p(x), _p(y), _st()))
    return y


# ---- original-paper agents (src/lb/sac_qmix.py, src/lb/sac_gru_discrete.py) ----------------------
def softmax_forward(x):
    """F.softmax over the last dimension (n <= 64 classes)."""
    y = torch.empty_like(x)
    n = x.shape[-1]
    check(_L().mlb_softmax_forward(_p(_chk(x)), _p(y), x.numel() // n, n, _st()))
    return y


def softmax_backward(y, dy):
    dx = torch.empty_like(y)
    n = y.shape[-1]
    check(_L().mlb_softmax_backward(_p(_chk(y)), _p(_chk(dy)), _p(dx), y.numel() // n, n, _st()))
    return dx


def concat_onehot(x, action, n):
    """x [rows, F] float32, action [rows, heads] int32 -> [rows, F + heads*n]."""
    rows, F = x.shape
    heads = action.shape[-1]
    out = torch.empty((rows, F + heads * n), dtype=torch.float32, device=x.device)
    check(_L().mlb_concat_onehot(_p(_chk(x)), _p(action), _p(out), rows, F, heads, n, _st()))
    return out


def categorical(p, u=None, given=None, want_logp=True, want_p=False):
    """Rows of probabilities [..., n] -> (class int32 [...], log p[class] or None, p[class] or None)."""
    n = p.shape[-1]
    rows = p.numel() // n
    shape = p.shape[:-1]
    act = torch.empty(shape, dtype=torch.int32, device=p.device)
    logp = torch.empty(shape, dtype=torch.float32, device=p.device) if want_logp else None
    ps = torch.empty(shape, dtype=torch.float32, device=p.device) if want_p else None
    check(_L().mlb_categorical(_p(_chk(p)), _p(u), _p(given), _p(act), _p(logp), _p(ps), rows, n, _st()))
    return act, logp, ps


def logprob_backward(p, action, g, group):
    d = torch.empty_like(p)
    n = p.shape[-1]
    check(_L().mlb_logprob_backward(_p(_chk(p)), _p(action), _p(_chk(g)), _p(d), p.numel() // n, n, group, _st()))
    return d


def scatter_class(g, action, n):
    d = torch.empty(tuple(g.shape) + (n,), dtype=torch.float32, device=g.device)
    check(_L().mlb_scatter_class(_p(_chk(g)), _p(action), _p(d), g.numel(), n, _st()))
    return d


def td_lambda_targets(reward, target_q, gamma=0.99, td_lambda=0.6):
    B, T = reward.shape
    ret = torch.empty_like(target_q)
    check(_L().mlb_td_lambda_targets(_p(_chk(reward)), _p(_chk(target_q)), _p(ret), gamma, td_lambda, B, T, _st()))
    return ret


def reward_normalize(reward, scale):
    B, T = reward.shape
    out = torch.empty_like(reward)
    check(_L().mlb_reward_normalize(_p(_chk(reward)), _p(out), scale, B, T, _st()))
    return out


def dsac_q_target(reward, q1n, q2n, logp_next, alpha, gamma):
    y = torch.empty_like(reward)
    check(_L().mlb_dsac_q_target(_p(_chk(reward)), _p(_chk(q1n)), _p(_chk(q2n)), _p(_chk(logp_next)), _p(alpha),
                                 float(gamma), _p(y), reward.numel(), _st()))
    return y


def weighted_sum_forward(q, w):
    M, A = q.shape
    out = torch.empty(M, dtype=torch.float32, device=q.device)
    check(_L().mlb_weighted_sum_forward(_p(_chk(q)), _p(_chk(w)), _p(out), M, A, _st()))
    return out


def weighted_sum_backward(g, q, w):
    M, A = q.shape
    dq, dw = torch.empty_like(q), torch.empty_like(w)
    check(_L().mlb_weighted_sum_backward(_p(_chk(g)), _p(q), _p(w), _p(dq), _p(dw), M, A, _st()))
    return dq, dw
