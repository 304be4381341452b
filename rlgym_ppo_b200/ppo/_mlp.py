"""Linear/ReLU stacks on the tcgen05 kernels: parameter arenas, bf16 operand copies, activation workspaces.

Shared by DiscreteFF (discrete_policy.py) and ValueEstimator (value_estimator.py).  The nn.Module keeps the
reference's `.model` nn.Sequential so state-dict keys and shapes are the reference's (`model.{2i}.weight` [out,in],
`model.{2i}.bias`), but its parameters are VIEWS into one flat fp32 arena and their `.grad`s views into a flat
gradient arena: the fused clip+Adam kernel and the NCCL allreduce see one contiguous buffer per learner.
"""
import os

import torch
import torch.nn as nn

from .. import _lib, ops

BF16 = torch.bfloat16

# Arithmetic of the Linear layers (see include/rlppo.h, "precision mode"):
#   "bf16": plain bf16 tensor-core operands, fp32 accumulation -- the throughput mode (fused whole-network kernels).
#   "fp32": every operand split into hi/mid/lo bf16 parts, 6 products forward / 3 backward on the same tensor cores --
#           fp32-equivalent results (gradients within 1e-3 of the fp32 reference; profiles/r02_precision_study.md).
PRECISIONS = ("bf16", "fp32")
_default_precision = [os.environ.get("RLPPO_PRECISION", "bf16")]


def set_default_precision(precision):
    """Precision of networks built from now on (Learner has no keyword for it: its signature is the reference's)."""
    assert precision in PRECISIONS, f"precision must be one of {PRECISIONS}"
    _default_precision[0] = precision


def default_precision():
    assert _default_precision[0] in PRECISIONS, f"RLPPO_PRECISION must be one of {PRECISIONS}"
    return _default_precision[0]


def build_sequential(input_shape, layer_sizes, out_features, softmax, tanh=False):
    """The reference's layer list (discrete_policy.py:22-31, value_estimator.py:19-28), created on the CPU with
    torch's default initialisation so a given torch.manual_seed yields the reference's initial weights."""
    assert len(layer_sizes) != 0, "AT LEAST ONE LAYER MUST BE SPECIFIED TO BUILD THE NEURAL NETWORK!"
    layers = [nn.Linear(int(input_shape), int(layer_sizes[0])), nn.ReLU()]
    prev = int(layer_sizes[0])
    for size in layer_sizes[1:]:
        layers.append(nn.Linear(prev, int(size)))
        layers.append(nn.ReLU())
        prev = int(size)
    layers.append(nn.Linear(prev, int(out_features)))
    if softmax:
        layers.append(nn.Softmax(dim=-1))
    if tanh:
        layers.append(nn.Tanh())       # continuous_policy.py:37
    return nn.Sequential(*layers)


class Stack:
    """Kernel-side view of one network: dims, arena views, bf16 operands, workspaces."""

    def __init__(self, model, device, precision=None):
        _lib.require_device()
        self.device = torch.device(device)
        self.precision = default_precision() if precision is None else precision
        assert self.precision in PRECISIONS
        self.exact = self.precision == "fp32"
        self.linears = [m for m in model if isinstance(m, nn.Linear)]
        self.in_dim = self.linears[0].in_features
        self.hidden = [l.out_features for l in self.linears[:-1]]
        # A hidden layer of width h runs on the device as pad8(h) units (16-byte rows for TMA): the extra units have zero
        # weight rows and bias in wq, zero columns in the next layer's wq, hence zero activations and zero gradients.
        # Only the bf16 operands and the workspaces are padded; parameters, gradients and state_dict keep true shapes.
        self.hidden_pad = [ops.pad8(h) for h in self.hidden]
        self.out_dim = self.linears[-1].out_features
        self.in_pad = ops.pad8(self.in_dim)
        self.out_pad = ops.pad8(self.out_dim)
        self.n_params = sum(p.numel() for l in self.linears for p in (l.weight, l.bias))
        self.params = None
        self.grads = None
        self._seen_version = -1
        self._ws_rows = 0
        self._ws = None
        # bf16 operands: wq[i] = W_i [out_pad8, in_pad8] (forward B operand, K-major; the fused kernels also read it as
        #                the MN-major B operand of the backward data GEMMs);
        #                wt[i] = W_i^T [in_pad8, out_pad8] (dgrad B operand of the LAYER-WISE kernels only; not needed for
        #                the first layer).  `need_wt` says whether anything reads wt: while the stack runs on the fused
        #                kernels it is neither refreshed by the optimiser launch nor by refresh_operands().
        self.need_wt = True
        # "fp32" mode: wq[i] holds 3 parts (hi|mid|lo, each pad64(in) columns), wt[i] 2 parts of pad64(out) columns
        self.wq, self.wt = [], []
        self.in_ps = ops.pad64(self.in_dim)           # part stride of the split input rows
        for i, l in enumerate(self.linears):
            o8, i8 = ops.pad8(l.out_features), ops.pad8(l.in_features)
            if self.exact:
                self.wq.append(torch.zeros((o8, 3 * ops.pad64(l.in_features)), dtype=BF16, device=self.device))
                self.wt.append(torch.zeros((i8, 2 * ops.pad64(l.out_features)), dtype=BF16, device=self.device)
                               if i > 0 else None)
            else:
                self.wq.append(torch.zeros((o8, i8), dtype=BF16, device=self.device))
                self.wt.append(torch.zeros((i8, o8), dtype=BF16, device=self.device) if i > 0 else None)

    # ---- arenas ---------------------------------------------------------------------------------------
    def bind(self, params_flat, grads_flat):
        """Move the parameters into `params_flat` (exactly n_params f32 on the device) and re-point every
        nn.Parameter (and its .grad) at its slice.  Order = nn.Module.parameters() order = parameters_to_vector
        order (ppo_learner.py:111-116)."""
        assert params_flat.numel() == self.n_params and grads_flat.numel() == self.n_params
        off = 0
        self.w, self.b, self.gw, self.gb = [], [], [], []
        with torch.no_grad():
            for l in self.linears:
                for p, plist, glist in ((l.weight, self.w, self.gw), (l.bias, self.b, self.gb)):
                    n = p.numel()
                    pv = params_flat[off:off + n].view(p.shape)
                    gv = grads_flat[off:off + n].view(p.shape)
                    pv.copy_(p.data)
                    p.data = pv
                    p.grad = gv
                    plist.append(pv)
                    glist.append(gv)
                    off += n
        self.params, self.grads = params_flat, grads_flat
        self._seen_version = -1
        self.__dict__.pop("_net_cache", None)

    def bf16_views(self, arena_offset):
        """rlppo_bf16_view entries (one per Linear) for the fused clip+Adam kernel's in-launch operand refresh."""
        out, off = [], int(arena_offset)
        if self.exact:
            return out      # split operands are rebuilt by refresh_operands() after the step, not inside the optimiser launch
        for i, l in enumerate(self.linears):
            v = _lib.Bf16View()
            v.offset, v.out_f, v.in_f = off, l.out_features, l.in_features
            v.wq, v.wq_ld = self.wq[i].data_ptr(), self.wq[i].stride(0)
            v.wt, v.wt_ld = ((None, 0) if self.wt[i] is None or not self.need_wt
                             else (self.wt[i].data_ptr(), self.wt[i].stride(0)))
            out.append(v)
            off += l.weight.numel() + l.bias.numel()
        return out

    def _version_sig(self):
        """torch version counters of the flat arena AND of every nn.Parameter: bind() re-points each parameter with
        `p.data = view`, which gives the Parameter its own counter, so load_state_dict (param.copy_) moves the
        Parameter's counter and not the arena's."""
        return (self.params._version,) + tuple(p._version for l in self.linears for p in (l.weight, l.bias))

    def mark_operands_fresh(self):
        self._seen_version = self._version_sig()

    def operands_stale(self):
        return self._version_sig() != self._seen_version

    def refresh_operands(self, force=False):
        """fp32 master weights -> bf16 GEMM operands.  Called after every optimiser step (our kernels do not bump
        torch's version counter) and lazily whenever torch-side code (load_state_dict, user edits) touched the arena."""
        if not force and not self.operands_stale():
            return
        for i, l in enumerate(self.linears):
            if self.exact:
                ops.weight_split(self.w[i], self.wq[i], 3, ops.pad64(l.in_features), self.wt[i], 2,
                                 ops.pad64(l.out_features))
            else:
                ops.weight_to_bf16(self.w[i], self.wq[i], self.wt[i] if self.need_wt else None)
        self._seen_version = self._version_sig()

    # ---- whole-network fused kernels (mlp_fused.cu) ---------------------------------------------------------------
    @property
    def fused_ok(self):
        """Shapes the single-kernel path supports; anything else runs layer by layer (mlp_tcgen05.cu)."""
        return (1 <= len(self.hidden) <= 4 and all(h % 64 == 0 and 64 <= h <= 256 for h in self.hidden)
                and self.in_dim <= 256 and self.out_dim <= 128 and not getattr(self, "force_layerwise", False)
                and not self.exact)

    def fused_net(self, x_ld, ws=None, policy_head=False):
        """struct rlppo_fused_net for this stack; `ws` (a workspace) supplies the training outputs."""
        key = (x_ld, id(ws), policy_head)
        cache = self.__dict__.setdefault("_net_cache", {})
        net = cache.get(key)
        if net is not None:
            return net
        net = _lib.FusedNet()
        L = len(self.hidden)
        net.n_hidden, net.in_dim, net.in_ld = L, self.in_dim, x_ld
        for i, h in enumerate(self.hidden):
            net.hidden[i] = h
        n_lin = L + 1 if policy_head else L
        for i in range(n_lin):
            net.wq[i], net.wq_ld[i] = self.wq[i].data_ptr(), self.wq[i].stride(0)
        for i in range(L + 1):
            net.bias[i], net.gbias[i] = self.b[i].data_ptr(), self.gb[i].data_ptr()
        if ws is not None:
            for i in range(L):
                net.h[i], net.h_ld[i] = ws["h"][i].data_ptr(), ws["h"][i].stride(0)
                net.dh[i], net.dh_ld[i] = ws["dh"][i].data_ptr(), ws["dh"][i].stride(0)
            net.dz, net.dz_ld = ws["dz"].data_ptr(), ws["dz"].stride(0)
        cache[key] = net
        return net

    def fused_wgrad_items(self, x, ws, head_dy=None):
        """(dy, x, dW, N, K, db) per Linear after a fused training pass: dW_l += dH_l^T X_{l-1}, db_l += colsum(dH_l) (and
        the policy head's); fed to ops.wgrad_multi.  The fused kernels leave every bias gradient to this launch (the value
        head's scalar one excepted)."""
        L = len(self.hidden)
        items = []
        if head_dy is not None:
            items.append((head_dy, ws["h"][L - 1], self.gw[L], self.out_dim, self.hidden[L - 1], self.gb[L]))
        for i in range(L - 1, -1, -1):
            inp = ws["h"][i - 1] if i > 0 else x
            K = self.hidden[i - 1] if i > 0 else self.in_dim
            items.append((ws["dh"][i], inp, self.gw[i], self.hidden[i], K, self.gb[i]))
        return items

    # ---- workspaces -------------------------------------------------------------------------------------
    def workspace(self, rows):
        """Activation buffers for `rows` rows (grow-only): h[i] bf16 [rows, pad8(hidden_i)]; two gradient ping-pong
        buffers as wide as the widest hidden layer; dz [rows, out_pad]."""
        if rows > self._ws_rows:
            cap = max(rows, 1)
            wmax = max(self.hidden_pad)
            if self.exact:
                # split activations: forward tensors 3 parts, gradients 2 parts, each part pad64(width) columns (zero padded)
                z = lambda parts, w: torch.zeros((cap, parts * ops.pad64(w)), dtype=BF16, device=self.device)  # noqa: E731
                self._ws = {
                    "h": [z(3, h) for h in self.hidden],
                    "d": [z(2, wmax) for _ in range(2)],
                    "dz": z(2, self.out_dim),
                    "z": z(3, self.out_dim),
                    "x": z(3, self.in_dim),
                    "x32": torch.empty((cap, self.in_dim), dtype=torch.float32, device=self.device),
                }
            else:
                self._ws = {
                    "h": [torch.empty((cap, h), dtype=BF16, device=self.device) for h in self.hidden_pad],
                    "d": [torch.empty((cap, wmax), dtype=BF16, device=self.device) for _ in range(2)],
                    "dh": [torch.empty((cap, h), dtype=BF16, device=self.device) for h in self.hidden_pad],
                    "dz": torch.zeros((cap, self.out_pad), dtype=BF16, device=self.device),
                    "z": torch.zeros((cap, 3 * ops.pad64(self.out_dim)), dtype=BF16, device=self.device),
                    "x": torch.zeros((cap, self.in_pad), dtype=BF16, device=self.device),
                }
            self._ws_rows = cap
            self.ws_gen = getattr(self, "ws_gen", 0) + 1      # captured graphs hold these addresses
            self.__dict__.pop("_net_cache", None)
        return self._ws

    # ---- staging ---------------------------------------------------------------------------------------------
    def stage_rows(self, src_f32, dst, mean=None, std=None, clip=5.0, dst_f32=None):
        """f32 [n, in_dim] device rows -> the first GEMM's A operand in `dst` (bf16 rows, or 3 split parts in "fp32" mode),
        optionally standardised (batched_agent_manager.py:303-315)."""
        if self.exact:
            assert dst_f32 is None
            ops.rows_split(src_f32, dst, 3, self.in_ps, mean, std, clip)
        elif mean is None:
            ops.rows_to_bf16(src_f32, dst)
        else:
            ops.rows_to_bf16(src_f32, dst, mean, std, clip, dst_f32=dst_f32)

    # ---- forward / backward of the hidden layers ---------------------------------------------------------------
    def forward_hidden(self, x, M, ws):
        """x bf16 [>=M, in_pad] (or split parts) -> ws['h'][-1] (last hidden activation, post-ReLU)."""
        prev, K, a_ps = x, self.in_dim, self.in_ps
        for i, h in enumerate(self.hidden):
            sp = ops.make_split(3, 3, 3, 3, a_ps, ops.pad64(K), ops.pad64(h)) if self.exact else None
            n8 = self.hidden_pad[i]
            ops.linear_fwd(prev, self.wq[i], self.b[i], ws["h"][i], n8, K, True, M=M, split=sp,
                           bias_n=h if n8 != h else 0)
            prev, K, a_ps = ws["h"][i], h, ops.pad64(h)
        return prev

    def _d_buffers(self, ws):
        """(dL/dH_last buffer, its part stride): ping-pong buffer 0, viewed at the last (padded) hidden width."""
        hl = self.hidden_pad[-1]
        d0 = ws["d"][0]
        if self.exact:
            return d0, ops.pad64(max(self.hidden))
        return (d0[:, :hl] if d0.shape[1] != hl else d0), 0

    def policy_head_train(self, h, M, ws, n_actions, actions, old_logp, adv, inv_b, clip, ent_coef, metrics,
                          logp_out=None):
        """Head GEMM + fused loss epilogue -> d(logits); the head's weight/bias gradients; dL/dH_last (masked).
        Returns dL/dH_last.  (discrete_policy.py:64-80, ppo_learner.py:153-180)"""
        hl = self.hidden[-1]
        sp = None
        if self.exact:
            sp = ops.make_split(3, 3, 3, 2, ops.pad64(hl), ops.pad64(hl), ops.pad64(self.out_dim))
        ops.policy_head_train(h, self.wq[-1], self.b[-1], n_actions, hl, actions, old_logp, adv, inv_b, clip, ent_coef,
                              ws["dz"], metrics, logp_out=logp_out, M=M, split=sp)
        return self.head_backward(h, M, ws)

    def head_backward(self, h, M, ws, gw=None, gb=None):
        """d(loss)/d(last Linear's output) in ws['dz'] -> that Linear's weight / bias gradients (added into gw[-1] /
        gb[-1], by default the gradient arena) and dL/dH_last (masked).  Returns dL/dH_last."""
        gw = self.gw if gw is None else gw
        gb = self.gb if gb is None else gb
        hl = self.hidden[-1]
        dh, d_ps = self._d_buffers(ws)
        if self.exact:
            h_ps, a_ps = ops.pad64(hl), ops.pad64(self.out_dim)
            ops.linear_wgrad(ws["dz"], h, gw[-1], gb[-1], self.out_dim, hl, M=M,
                             split=ops.make_split(2, 2, 2, 1, a_ps, h_ps))
            ops.linear_dgrad(ws["dz"], self.wt[-1], h, dh, self.out_pad, hl, M=M,
                             split=ops.make_split(2, 2, 2, 2, a_ps, a_ps, d_ps))
        else:
            ops.linear_wgrad(ws["dz"], h, gw[-1], gb[-1], self.out_dim, hl, M=M)
            ops.linear_dgrad(ws["dz"], self.wt[-1], h, dh, self.out_pad, hl, M=M)
        return dh

    def policy_head_backward(self, h, M, ws, n_actions, actions, d_logp, d_ent, d_probs, gw, gb):
        """Discrete head for upstream gradients of (log-prob, mean entropy, probabilities) -> d(logits) -> the head's
        gradients into gw / gb.  Returns dL/dH_last."""
        hl = self.hidden[-1]
        sp = ops.make_split(3, 3, 3, 2, ops.pad64(hl), ops.pad64(hl), ops.pad64(self.out_dim)) if self.exact else None
        ops.policy_head_backward(h, self.wq[-1], self.b[-1], n_actions, hl, actions, d_logp, d_ent, d_probs, ws["dz"],
                                 M=M, split=sp)
        return self.head_backward(h, M, ws, gw, gb)

    def value_head_backward(self, h, M, ws, d_values, gw, gb):
        """Value head for an upstream gradient of the values -> its gradients into gw / gb.  Returns dL/dH_last."""
        hl = self.hidden[-1]
        dh, d_ps = self._d_buffers(ws)
        kw = dict(h_parts=3, h_pstride=ops.pad64(hl), dh_parts=2, dh_pstride=d_ps) if self.exact else {}
        ops.value_head_backward(h, self.w[-1], hl, d_values, dh, gw[-1], gb[-1], M=M, **kw)
        return dh

    def stage_dz(self, d_logits, ws):
        """f32 [M, out_dim] upstream gradient of the last Linear's output -> ws['dz'] in the layout head_backward reads."""
        if self.exact:
            ops.rows_split(d_logits, ws["dz"], 2, ops.pad64(self.out_dim))
        else:
            ops.rows_to_bf16(d_logits, ws["dz"])

    def logits(self, h, M, ws):
        """The last Linear WITHOUT a fused head: z = H W^T + b written to ws['z'] as three bf16 parts (fp32-exact logits
        in either precision mode), for the per-row head kernels (rlppo_head_*).  Returns (z, parts, part stride)."""
        hl, zp = self.hidden[-1], ops.pad64(self.out_dim)
        if self.exact:
            sp = ops.make_split(3, 3, 3, 3, ops.pad64(hl), ops.pad64(hl), zp)
        else:
            sp = ops.make_split(1, 1, 1, 3, 0, 0, zp)
        ops.linear_fwd(h, self.wq[-1], self.b[-1], ws["z"], self.out_pad, hl, False, M=M, split=sp, bias_n=self.out_dim)
        return ws["z"], 3, zp

    def dz_view(self, ws):
        """(dz buffer, parts, part stride, columns to write) the head kernels fill for head_backward()."""
        if self.exact:
            return ws["dz"], 2, ops.pad64(self.out_dim), self.out_pad
        return ws["dz"], 1, 0, self.out_pad

    def value_head_train(self, h, M, ws, targets, inv_b, metrics):
        """v = H w + b, MSE and its backward into H_last (value_estimator.py:27, ppo_learner.py:176).  Returns dL/dH_last."""
        hl = self.hidden[-1]
        dh, d_ps = self._d_buffers(ws)
        kw = dict(h_parts=3, h_pstride=ops.pad64(hl), dh_parts=2, dh_pstride=d_ps) if self.exact else {}
        ops.value_head(h, self.w[-1], self.b[-1], hl, targets=targets, inv_batch=inv_b, dh=dh, dw=self.gw[-1],
                       db=self.gb[-1], metrics=metrics, M=M, **kw)
        return dh

    def value_head_infer(self, h, M, out):
        hl = self.hidden[-1]
        kw = dict(h_parts=3, h_pstride=ops.pad64(hl)) if self.exact else {}
        ops.value_head(h, self.w[-1], self.b[-1], hl, values_out=out, M=M, **kw)

    def policy_head_sample(self, h, M, n_actions, **kw):
        hl = self.hidden[-1]
        sp = ops.make_split(3, 3, 3, 1, ops.pad64(hl), ops.pad64(hl)) if self.exact else None
        ops.policy_head_sample(h, self.wq[-1], self.b[-1], n_actions, hl, M=M, split=sp, **kw)

    def backward_hidden(self, x, M, ws, d_last, gw=None, gb=None):
        """d_last = dL/dH_last (bf16 [>=M, pad8(hidden[-1])], already ReLU-masked, padding columns zero).  Accumulates
        dW/db of every hidden layer into gw / gb (default: the gradient arena; wgrad kernels add) and propagates through
        the stack."""
        gw = self.gw if gw is None else gw
        gb = self.gb if gb is None else gb
        d = d_last
        # The bias gradient of layer i-1 comes out of the dgrad epilogue that produces dL/dH_{i-1} (db_below) instead of
        # a separate column-sum pass over that tensor: only the top hidden layer's wgrad sums its own.  Measured on c3 in
        # one box: 47.3 -> 46.4 ms per step (with the first, unpipelined epilogue it was a wash).
        top = len(self.hidden) - 1
        d_ps = ops.pad64(max(self.hidden))        # "fp32" mode: part stride of the gradient ping-pong buffers
        for i in range(top, -1, -1):
            inp = ws["h"][i - 1] if i > 0 else x
            K = self.hidden[i - 1] if i > 0 else self.in_dim
            N = self.hidden[i]
            sp_w = ops.make_split(2, 2, 2, 1, d_ps, ops.pad64(K)) if self.exact else None
            ops.linear_wgrad(d, inp, gw[i], gb[i] if i == top else None, N, K, M=M, split=sp_w)
            if i > 0:
                nxt = ws["d"][0] if d.data_ptr() != ws["d"][0].data_ptr() else ws["d"][1]
                if self.exact:
                    dx = nxt
                    sp_d = ops.make_split(2, 2, 2, 2, d_ps, ops.pad64(N), d_ps)
                else:
                    k8 = self.hidden_pad[i - 1]
                    dx = nxt[:, :k8] if nxt.shape[1] != k8 else nxt
                    sp_d = None
                ops.linear_dgrad(d, self.wt[i], inp, dx, N, K, M=M, db_below=gb[i - 1], split=sp_d)
                d = dx

    # ---- torch autograd ---------------------------------------------------------------------------------------------
    def grad_views(self, flat):
        """Per-Linear (dW, db) views of a flat f32[n_params] buffer, in parameter order (the arena's layout)."""
        gw, gb, off = [], [], 0
        for l in self.linears:
            for p, lst in ((l.weight, gw), (l.bias, gb)):
                lst.append(flat[off:off + p.numel()].view(p.shape))
                off += p.numel()
        return gw, gb

    def refresh_transposed(self):
        """W^T operands for the layer-wise backward.  While the stack trains on the fused kernels nothing keeps them
        current (need_wt False), so they are rebuilt from the master weights here."""
        if self.need_wt:
            return
        for i in range(1, len(self.linears)):
            ops.weight_to_bf16(self.w[i], self.wq[i], self.wt[i])


def autograd_wanted(module, obs):
    """Whether a differentiable method (get_output / forward / get_backprop_data) records its call for torch autograd:
    the module's `autograd` attribute set to True, grad mode on and some parameter requiring grad.  The switch is off by
    default so that these methods keep returning plain tensors, which callers read with .numpy() under grad mode.
    Gradients with respect to the observations are not provided."""
    if not (module.autograd and torch.is_grad_enabled()):
        return False
    if isinstance(obs, torch.Tensor) and obs.requires_grad:
        raise RuntimeError(f"{type(module).__name__}: gradients with respect to the observations are not supported; "
                           "pass obs.detach()")
    return any(p.requires_grad for p in module.parameters())


def grad_f32(g, rows, cols=None):
    """An upstream gradient as the contiguous f32 device rows the backward kernels read (None stays None)."""
    if g is None:
        return None
    shape = (rows,) if cols is None else (rows, cols)
    return g.reshape(shape).to(torch.float32).contiguous()


class StackFunction(torch.autograd.Function):
    """torch autograd through one Linear/ReLU stack and its head, on the kernels.

    apply(stack, run, head_backward, *params):
      run() -> (outputs, n rows, saved): runs the module's ordinary forward (so the outputs are bit for bit what the
               call returns under no_grad) and returns what its head backward needs besides the recomputed activations
               (e.g. a copy of the action rows).  A copy of the staged input rows is kept here.
      head_backward(h, M, ws, grads, gw, gb, saved) -> dL/dH_last: the head's backward kernel for the upstream gradients
               `grads` (one per output, None where no gradient flows), its weight / bias gradients into gw[-1] / gb[-1].
    The parameters are saved with save_for_backward, so an in-place edit of a weight between the forward and the backward
    raises torch's version-counter error.  The backward recomputes the hidden activations with the layer-wise kernels
    from the saved input rows; where the forward ran on a whole-network fused kernel (ValueEstimator.forward at fused
    shapes in bf16) a recomputed ReLU mask can differ from the forward's in units whose pre-activation is within bf16
    rounding of zero -- the same deviation between the fused and layer-wise kernels the learner already accepts.  The
    gradients come back as views of one fresh zeroed flat buffer; autograd adds them into `.grad`, which stays the
    learner's arena view where it is one.  Not supported: double backward (create_graph=True raises), and running
    PPOLearner.learn() between a forward and its backward (the learner's kernels do not bump torch's version counters,
    so that edit goes undetected)."""

    @staticmethod
    def forward(ctx, stack, run, head_backward, *params):
        outs, n, saved = run()
        ctx.stack, ctx.head_backward, ctx.n, ctx.saved = stack, head_backward, n, saved
        ctx.x = stack._ws["x"][:n].clone() if n else None
        ctx.save_for_backward(*params)
        ctx.set_materialize_grads(False)
        return outs

    @staticmethod
    def backward(ctx, *grads):
        if torch.is_grad_enabled():
            raise RuntimeError("the rlgym_ppo_b200 networks support first-order gradients only (create_graph=True / "
                               "double backward is not supported)")
        params = ctx.saved_tensors          # raises if a parameter was modified in place since the forward
        st, M = ctx.stack, ctx.n
        flat = torch.zeros(st.n_params, dtype=torch.float32, device=st.device)
        gw, gb = st.grad_views(flat)
        if M and any(g is not None for g in grads):
            st.refresh_transposed()
            ws = st.workspace(M)
            h = st.forward_hidden(ctx.x, M, ws)
            dh = ctx.head_backward(h, M, ws, grads, gw, gb, ctx.saved)
            st.backward_hidden(ctx.x, M, ws, dh, gw, gb)
        out = []
        for w, b in zip(gw, gb):
            out += [w, b]
        assert len(out) == len(params)
        return (None, None, None) + tuple(out)
