"""Layers with explicit forward / backward on the marllb_b200 policy kernels.

Parameters are float32 CUDA tensors in torch's layouts (nn.Linear weight [out, in]; nn.GRU
weight_ih_l0 [3H, in], gate order r, z, n) and are exposed through `state_dict()` with the
reference modules' key names, so checkpoints move between the reference and this package.
Initialisation re-uses torch.nn's initialisers on the host in the reference's construction
order (same RNG consumption as the reference for the same torch seed); no torch.nn module is
on the compute path.
"""
from __future__ import annotations

from collections import OrderedDict

import torch

from . import ops


class Params:
    """Named float32 CUDA tensors + gradients + Adam moments."""

    def __init__(self, device):
        self.device = device
        self.p = OrderedDict()
        self.g = OrderedDict()

    def add(self, name, tensor):
        t = tensor.detach().to(device=self.device, dtype=torch.float32).contiguous().clone()
        self.p[name] = t
        self.g[name] = torch.zeros_like(t)
        return t

    def zero_grad(self):
        if getattr(self, "_flat_g", None) is not None:   # sole owner of a FlatBucket: one launch
            self._flat_g.zero_()
            return
        for g in self.g.values():
            g.zero_()

    def state_dict(self, prefix=""):
        return OrderedDict((prefix + k, v.detach().clone()) for k, v in self.p.items())

    def load_state_dict(self, sd, prefix=""):
        for k in self.p:
            src = sd[prefix + k]
            if tuple(src.shape) != tuple(self.p[k].shape):
                raise RuntimeError(f"size mismatch for {prefix + k}: {tuple(src.shape)} vs {tuple(self.p[k].shape)}")
            self.p[k].copy_(src.to(device=self.device, dtype=torch.float32))

    def tensors(self):
        return list(self.p.values())

    def grads(self):
        return list(self.g.values())


class FlatBucket:
    """All parameters of ONE optimiser in one flat float32 buffer and all their gradients in
    another (SURVEY 8e: "one flattened gradient bucket per optimiser step").

    The tensors of the given `Params` sets are re-bound to views of the flat buffers (16-byte
    aligned, padding stays zero), so that per step the optimiser is ONE Adam launch, gradient
    clipping ONE norm + ONE scale launch, and the data-parallel reduction ONE all-reduce.
    """

    def __init__(self, param_sets, extra=()):
        """param_sets: list of Params; extra: list of (param, grad) tensor pairs (e.g. log_alpha)."""
        items = []
        for P in param_sets:
            for name in P.p:
                items.append((P, name, P.p[name], P.g[name]))
        for pt, gt in extra:
            items.append((None, None, pt, gt))
        dev = items[0][2].device
        offs, total = [], 0
        for _, _, t, _ in items:
            offs.append(total)
            total += (t.numel() + 3) // 4 * 4
        self.flat_p = torch.zeros(total, dtype=torch.float32, device=dev)
        self.flat_g = torch.zeros(total, dtype=torch.float32, device=dev)
        self.params, self.grads, self._slices = [], [], []
        for (P, name, t, g), o in zip(items, offs):
            pv = self.flat_p[o:o + t.numel()].view(t.shape)
            gv = self.flat_g[o:o + t.numel()].view(t.shape)
            pv.copy_(t)
            gv.copy_(g)
            if P is not None:
                P.p[name], P.g[name] = pv, gv
            self.params.append(pv)
            self.grads.append(gv)
            self._slices.append((o, t.numel(), tuple(t.shape)))
        if len(param_sets) == 1 and not extra:
            param_sets[0]._flat_g = self.flat_g
            param_sets[0]._flat_p = self.flat_p

    def views(self, flat):
        return [flat[o:o + n].view(shape) for o, n, shape in self._slices]


def _dp_world(group=None):
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return 1
    return dist.get_world_size(group)


def allreduce_mean_(flat_g, group=None):
    """Data-parallel gradient reduction over one flat bucket: ONE all-reduce that averages over the ranks, so the
    loss keeps its mean-over-the-global-batch meaning (F.mse_loss / .mean(), sac_agent.py:197-198,216).  NCCL
    averages inside the collective (ncclAvg: no separate scaling launch); gloo (CPU tests) sums, then scales.
    No-op without an initialised process group."""
    import torch.distributed as dist
    world = _dp_world(group)
    if world == 1:
        return flat_g
    if flat_g.is_cuda:
        dist.all_reduce(flat_g, op=dist.ReduceOp.AVG, group=group)
    else:
        dist.all_reduce(flat_g, op=dist.ReduceOp.SUM, group=group)
        flat_g.mul_(1.0 / world)
    return flat_g


_comm_streams = {}


def comm_stream(device):
    """One side stream per device for the gradient all-reduces (SURVEY 5: "launched on a side stream right after
    the last backward GEMM and consumed by the fused Adam kernel")."""
    key = (device.type, device.index)
    if key not in _comm_streams:
        _comm_streams[key] = torch.cuda.Stream(device=device)
    return _comm_streams[key]


class Adam:
    """torch.optim.Adam (default betas / eps, no weight decay) over one FlatBucket."""

    def __init__(self, bucket: FlatBucket, lr, data_parallel=True, max_grad_norm=None):
        self.bucket, self.lr = bucket, lr
        self.params, self.grads = bucket.params, bucket.grads
        self._m = torch.zeros_like(bucket.flat_p)
        self._v = torch.zeros_like(bucket.flat_p)
        self.m, self.v = bucket.views(self._m), bucket.views(self._v)   # per-tensor views (checkpoints)
        self.t = 0
        # the step counter the kernel uses lives on the device (a step replayed from a CUDA graph must not
        # depend on a host value that changes); self.t mirrors it for checkpoints
        self._t_dev = torch.zeros(1, dtype=torch.int32, device=bucket.flat_p.device)
        self._coef_dev = torch.zeros(2, dtype=torch.float32, device=bucket.flat_p.device)
        self.data_parallel, self.max_grad_norm = data_parallel, max_grad_norm
        self._reduce_done = None     # event of an all-reduce in flight on the side stream (reduce_async)

    def reduce_async(self):
        """Start the data-parallel all-reduce of this bucket's gradients on the side stream, right after the
        backward pass that produced them; step() waits for it.  Whatever the caller launches in between on the
        compute stream overlaps the collective (the fork / join is expressed with events, so it is captured into a
        CUDA graph like any other launch).  No-op on one rank."""
        b = self.bucket
        if not self.data_parallel or not b.flat_g.is_cuda or _dp_world() == 1:
            return
        cur = torch.cuda.current_stream(b.flat_g.device)
        side = comm_stream(b.flat_g.device)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            allreduce_mean_(b.flat_g)
            self._reduce_done = torch.cuda.Event()
            self._reduce_done.record(side)

    def step(self):
        """[all-reduce] -> [clip by the GLOBAL norm] -> Adam, each over the whole bucket."""
        b = self.bucket
        if self._reduce_done is not None:
            torch.cuda.current_stream(b.flat_g.device).wait_event(self._reduce_done)
            self._reduce_done = None
        elif self.data_parallel:
            allreduce_mean_(b.flat_g)
        if self.max_grad_norm is not None:
            ops.clip_grad_norm_([b.flat_g], self.max_grad_norm)
        self.t += 1
        if b.flat_p.is_cuda:
            ops.adam_step_dev(b.flat_p, b.flat_g, self._m, self._v, self.lr, self._t_dev, self._coef_dev)
        else:
            ops.adam_step(b.flat_p, b.flat_g, self._m, self._v, self.lr, self.t)

    def state_dict(self):
        """torch.optim.Adam's own layout -- {'state': {i: {step, exp_avg, exp_avg_sq}}, 'param_groups': [...]} with the
        parameters numbered in bucket order (= the reference's optimiser parameter order, sac_agent.py:93-106,
        qmix_agent.py:108-113) -- so checkpoints move between the reference agents and these in both directions."""
        group = dict(torch.optim.Adam([torch.zeros(1)], lr=self.lr).state_dict()["param_groups"][0])
        group["lr"] = self.lr
        group["params"] = list(range(len(self.params)))
        state = {}
        if self.t > 0:                       # torch creates the per-parameter state on the first step
            for i, (m, v) in enumerate(zip(self.m, self.v)):
                state[i] = {"step": torch.tensor(float(self.t)), "exp_avg": m.detach().clone(),
                            "exp_avg_sq": v.detach().clone()}
        return {"state": state, "param_groups": [group]}

    def load_state_dict(self, sd):
        """Accepts torch.optim.Adam's layout (reference checkpoints) and this package's round-1 layout
        ({'step', 'exp_avg': [...], 'exp_avg_sq': [...]})."""
        if "param_groups" in sd:
            groups = sd["param_groups"]
            idx = [i for g in groups for i in g["params"]]
            if len(idx) != len(self.params):
                raise ValueError(f"optimizer state has {len(idx)} parameters, this optimiser has {len(self.params)}")
            g0 = groups[0]
            if tuple(g0.get("betas", (0.9, 0.999))) != (0.9, 0.999) or g0.get("eps", 1e-8) != 1e-8 \
                    or g0.get("weight_decay", 0) != 0 or g0.get("amsgrad", False):
                raise ValueError("only torch.optim.Adam defaults (betas (0.9, 0.999), eps 1e-8, no weight decay / amsgrad) are supported")
            self.lr = float(g0.get("lr", self.lr))
            st = sd["state"]
            if not st:
                self.t = 0
                self._m.zero_()
                self._v.zero_()
            else:
                steps = {int(float(st[i]["step"])) for i in idx if i in st}
                if len(steps) != 1 or any(i not in st for i in idx):
                    raise ValueError("optimizer state must hold every parameter at the same step count")
                self.t = steps.pop()
                for k, i in enumerate(idx):
                    if tuple(st[i]["exp_avg"].shape) != tuple(self.m[k].shape):
                        raise ValueError(f"optimizer state of parameter {i}: shape {tuple(st[i]['exp_avg'].shape)} "
                                         f"vs {tuple(self.m[k].shape)}")
                    self.m[k].copy_(st[i]["exp_avg"])
                    self.v[k].copy_(st[i]["exp_avg_sq"])
        else:
            self.t = int(sd["step"])
            for m, s_ in zip(self.m, sd["exp_avg"]):
                m.copy_(s_)
            for v, s_ in zip(self.v, sd["exp_avg_sq"]):
                v.copy_(s_)
        self._t_dev.fill_(self.t)


class wgrad_on:
    """`with wgrad_on(stream, slot):` -- backward passes issued inside put their PARAMETER-gradient kernels (dW = dy^T x,
    db = colsum(dy)) on `stream`, off the chain that carries the input gradient from layer to layer: nothing downstream
    in the pass reads them, and at update batch sizes each is a small launch that would otherwise sit on the critical
    path.  The operands are kept alive until the join at scope exit (their blocks belong to the issuing stream's
    allocator pool and must not be recycled while the side stream still reads them)."""
    active = None

    def __init__(self, stream, slot):
        self.stream, self.slot, self.keep = stream, slot, []

    def __enter__(self):
        self._outer, wgrad_on.active = wgrad_on.active, self
        return self

    def __exit__(self, *exc):
        wgrad_on.active = self._outer
        torch.cuda.current_stream(self.stream.device).wait_stream(self.stream)
        self.keep.clear()
        return False

    def run(self, fn, *operands):
        self.stream.wait_stream(torch.cuda.current_stream(self.stream.device))
        with ops.side_branch(self.stream, self.slot):
            fn()
        self.keep.append(operands)


def _param_grads(fn, *operands):
    w = wgrad_on.active
    if w is None:
        fn()
    else:
        w.run(fn, *operands)


def linear_backward(P, wname, bname, x, dy, need_dx=True):
    """Accumulate dW += dy^T x, db += colsum(dy); return dx = dy W (x, dy 2-D)."""
    def grads():
        ops.matmul_tn(dy, x, out=P.g[wname], beta=1.0)
        ops.colsum(dy, out=P.g[bname], beta=1.0)
    _param_grads(grads, dy, x)
    return ops.matmul_nn(dy, P.p[wname]) if need_dx else None


class GRUCellSeq:
    """nn.GRU(in, H, batch_first=True) run step by step (agent_network.py:41,76-78; networks.py:60,97)."""

    def __init__(self, P: Params, prefix="gru."):
        self.P, self.k = P, prefix

    def step(self, x, h, save=False):
        """x [B,in], h [B,H] -> h' [B,H]; with save=True also returns the tape entry."""
        P, k = self.P.p, self.k
        gi = ops.linear(x, P[k + "weight_ih_l0"], P[k + "bias_ih_l0"])
        gh = ops.linear(h, P[k + "weight_hh_l0"], P[k + "bias_hh_l0"])
        h_new, gates = ops.gru_gates_forward(gi, gh, h, save_gates=save)
        return (h_new, (x, h, gh, gates)) if save else h_new

    def forward_seq(self, xs, h0):
        """xs [T,B,in] (time-major, contiguous), h0 [B,H] -> hs [T,B,H], tape."""
        P, k = self.P.p, self.k
        T, B, In = xs.shape
        H = h0.shape[-1]
        gi_all = ops.linear(xs.reshape(T * B, In), P[k + "weight_ih_l0"], P[k + "bias_ih_l0"]).reshape(T, B, 3 * H)
        if ops.gru_seq_supported(H):
            # the whole time loop in one launch (csrc/mlb_policy.cu gru_seq_fwd_kernel)
            hs, hprev, ghs, gates = ops.gru_seq_forward(gi_all.contiguous(), P[k + "weight_hh_l0"], P[k + "bias_hh_l0"],
                                                        h0.contiguous())
            return hs, (xs, hprev, ghs, gates)
        hs = torch.empty((T, B, H), dtype=torch.float32, device=xs.device)
        hprev = torch.empty((T, B, H), dtype=torch.float32, device=xs.device)
        ghs = torch.empty((T, B, 3 * H), dtype=torch.float32, device=xs.device)
        gates = torch.empty((T, B, 3 * H), dtype=torch.float32, device=xs.device)
        h = h0
        for t in range(T):
            hprev[t].copy_(h)
            gh = ops.linear(h, P[k + "weight_hh_l0"], P[k + "bias_hh_l0"], out=ghs[t])
            h_new, g = ops.gru_gates_forward(gi_all[t], gh, hprev[t], save_gates=True)
            gates[t].copy_(g)
            hs[t].copy_(h_new)
            h = hs[t]
        return hs, (xs, hprev, ghs, gates)

    def backward_seq(self, dhs, tape, need_dx=False):
        """dhs [T,B,H] gradient w.r.t. every hidden output; accumulates parameter gradients (BPTT)."""
        P, k = self.P, self.k
        xs, hprev, ghs, gates = tape
        T, B, H = dhs.shape
        if ops.gru_seq_supported(H):
            dgi_all, dgh_all, dh_next = ops.gru_seq_backward(dhs.contiguous(), gates, hprev, ghs, P.p[k + "weight_hh_l0"])
            return self._seq_param_grads(dgi_all, dgh_all, xs, hprev, need_dx, dh_next)
        dgi_all = torch.empty_like(gates)
        dgh_all = torch.empty_like(gates)
        dh_next = torch.zeros((B, H), dtype=torch.float32, device=dhs.device)
        for t in range(T - 1, -1, -1):
            dh = dhs[t].clone()
            ops.axpby(1.0, dh_next, 1.0, dh)
            dgi, dgh, dh_direct = ops.gru_gates_backward(dh, gates[t], hprev[t], ghs[t])
            dgi_all[t].copy_(dgi)
            dgh_all[t].copy_(dgh)
            dh_next = ops.matmul_nn(dgh, P.p[k + "weight_hh_l0"])
            ops.axpby(1.0, dh_direct, 1.0, dh_next)
        return self._seq_param_grads(dgi_all, dgh_all, xs, hprev, need_dx, dh_next)

    def _seq_param_grads(self, dgi_all, dgh_all, xs, hprev, need_dx, dh_next):
        P, k = self.P, self.k
        T, B, H = hprev.shape
        In = xs.shape[-1]
        dgi2, dgh2 = dgi_all.reshape(T * B, 3 * H), dgh_all.reshape(T * B, 3 * H)

        def grads():
            ops.matmul_tn(dgi2, xs.reshape(T * B, In), out=P.g[k + "weight_ih_l0"], beta=1.0)
            ops.colsum(dgi2, out=P.g[k + "bias_ih_l0"], beta=1.0)
            ops.matmul_tn(dgh2, hprev.reshape(T * B, H), out=P.g[k + "weight_hh_l0"], beta=1.0)
            ops.colsum(dgh2, out=P.g[k + "bias_hh_l0"], beta=1.0)
        _param_grads(grads, dgi_all, dgh_all, xs, hprev)
        dxs = ops.matmul_nn(dgi2, P.p[k + "weight_ih_l0"]).reshape(T, B, In) if need_dx else None
        return dxs, dh_next
