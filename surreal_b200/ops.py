"""Torch-tensor front end of the C-ABI: device buffers come from torch, kernels from libsurreal_b200.

Nothing here computes on the CPU or through torch ops on the hot path; torch only owns memory and
streams (``tensor.data_ptr()`` / ``torch.cuda.current_stream()``).
"""
import ctypes as C
import os

import torch

from . import _lib
from ._lib import Mlp, ZFilter, Rows, ACT_NONE, ACT_RELU, ACT_TANH, MAX_LAYERS, check  # noqa: F401


def _ru(v, m):
    return (v + m - 1) // m * m


def _stream():
    _lib.ensure_device()
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _f32c(t):
    assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous(), \
        'expected a contiguous float32 CUDA tensor, got %s %s' % (t.dtype, t.device)
    return t


class FlatNet:
    """An MLP whose parameters live in ONE flat fp32 device buffer in the kernel layout
    (W[l] = [in_l][ldw_l], the transpose of torch.nn.Linear.weight; ldw = out rounded up to 4;
    padding stays zero).  Gradients / Adam moments use buffers of the same layout, so optimiser and
    NCCL all-reduce are single flat kernels / one collective.  ``extra`` trailing floats hold
    non-layer parameters (PPO's log_var, builders.py:112)."""

    def __init__(self, dims, acts, device, aux_layer=-1, aux_dim=0, extra=0):
        assert 1 <= len(dims) - 1 <= MAX_LAYERS and len(acts) == len(dims) - 1
        self.dims = list(dims)
        self.acts = list(acts)
        self.aux_layer, self.aux_dim = aux_layer, (aux_dim if aux_layer >= 0 else 0)
        self.n_layers = len(dims) - 1
        self.layout = []
        off = 0
        for l in range(self.n_layers):
            K = dims[l] + (self.aux_dim if aux_layer == l else 0)
            N = dims[l + 1]
            ldw = _ru(N, 4)
            self.layout.append(dict(w=off, b=off + K * ldw, K=K, N=N, ldw=ldw))
            off += K * ldw + ldw
        self.extra = extra
        self.extra_off = off
        off += _ru(extra, 4)
        self.size = off
        self.device = torch.device(device)
        self.params = torch.zeros(off, dtype=torch.float32, device=self.device)

    # -- views -----------------------------------------------------------------------------------
    def W(self, l, buf=None):
        lay = self.layout[l]
        buf = self.params if buf is None else buf
        return buf[lay['w']:lay['w'] + lay['K'] * lay['ldw']].view(lay['K'], lay['ldw'])

    def b(self, l, buf=None):
        lay = self.layout[l]
        buf = self.params if buf is None else buf
        return buf[lay['b']:lay['b'] + lay['ldw']]

    def extra_view(self, buf=None):
        buf = self.params if buf is None else buf
        return buf[self.extra_off:self.extra_off + self.extra]

    def set_layer(self, l, weight, bias):
        """weight: [out, in] (torch.nn.Linear convention), bias: [out]."""
        N = self.layout[l]['N']
        self.W(l)[:, :N] = torch.as_tensor(weight, dtype=torch.float32).t().to(self.device)
        self.b(l)[:N] = torch.as_tensor(bias, dtype=torch.float32).to(self.device)

    def get_layer(self, l, buf=None):
        N = self.layout[l]['N']
        return self.W(l, buf)[:, :N].t().contiguous(), self.b(l, buf)[:N].clone()

    def load_layers(self, layers, extra=None):
        for l, (w, b) in enumerate(layers):
            self.set_layer(l, w, b)
        if extra is not None:
            self.extra_view()[:] = torch.as_tensor(extra, dtype=torch.float32).reshape(-1).to(self.device)
        return self

    def clone_like(self):
        n = FlatNet(self.dims, self.acts, self.device, self.aux_layer, self.aux_dim, self.extra)
        n.params.copy_(self.params)
        return n

    def desc(self, buf=None):
        """ctypes descriptor over ``buf`` (defaults to the live parameters)."""
        buf = self.params if buf is None else buf
        m = Mlp()
        m.n_layers = self.n_layers
        for i, d in enumerate(self.dims):
            m.dims[i] = d
        base = buf.data_ptr()
        for l, lay in enumerate(self.layout):
            m.act[l] = self.acts[l]
            m.W[l] = base + 4 * lay['w']
            m.b[l] = base + 4 * lay['b']
            m.ldw[l] = lay['ldw']
        m.aux_layer = self.aux_layer
        m.aux_dim = self.aux_dim
        return m


def zfilter_desc(stats, eps=1e-5):
    z = ZFilter()
    z.stats = stats.data_ptr() if stats is not None else None
    z.eps = eps
    return z


class PackedWeights:
    """Per-step inference copy of a FlatNet's weights in tensor-core fragment order (sb200_mlp_pack_tf32), for
    mlp_forward_packed.  The owner calls ``refresh()`` whenever the parameters may have changed -- the agents do
    it at every parameter fetch and at the top of every rollout chunk, so a pack can never outlive its version."""

    def __init__(self, net):
        self.net = net
        d = net.desc()
        n = int(_lib.lib().sb200_mlp_pack_floats(C.byref(d)))
        self.supported = n > 0
        self.buf = torch.zeros(max(n, 4), dtype=torch.float32, device=net.device) if self.supported else None

    def refresh(self):
        if self.supported:
            d = self.net.desc()
            check(_lib.lib().sb200_mlp_pack_tf32(C.byref(d), _ptr(self.buf), _stream()), 'sb200_mlp_pack_tf32')
        return self


def mlp_forward_packed(packed, x, zf_stats=None, zf_eps=1e-5, aux=None, out=None):
    """Small-batch inference forward on pre-packed weights; x: [rows, D] contiguous-row CUDA tensor."""
    net = packed.net
    assert packed.supported and x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
    r = Rows()
    r.x, r.x_next, r.ldx, r.rows, r.win_n = x.data_ptr(), None, x.stride(0), x.shape[0], 0
    if net.aux_layer >= 0:
        assert aux is not None and aux.is_cuda and aux.stride(-1) == 1
        r.aux, r.aux_ld = aux.data_ptr(), aux.stride(0)
    else:
        r.aux, r.aux_ld = None, 0
    r.save_x, r.ld_save_x = None, 0
    if out is None:
        out = torch.empty(x.shape[0], net.dims[-1], dtype=torch.float32, device=x.device)
    zf = zfilter_desc(zf_stats, zf_eps)
    d = net.desc()
    check(_lib.lib().sb200_mlp_forward_packed_f32(C.byref(d), _ptr(packed.buf), C.byref(zf), C.byref(r), _ptr(out),
                                                  out.stride(0), _stream()), 'sb200_mlp_forward_packed_f32')
    return out


class Tc5Forward:
    """Large-batch forward of a FlatNet on the tcgen05 / TMEM kernel (sb200_mlp_forward_tc5_f32).  Owns the workspace of
    the per-call weight images; ``supported(rows)`` says whether the shape qualifies (else callers use mlp_forward)."""

    def __init__(self, net):
        self.net = net
        d = net.desc()
        n = int(_lib.lib().sb200_mlp_tc5_workspace_bytes(C.byref(d)))
        self.ws = torch.zeros(n, dtype=torch.uint8, device=net.device) if n > 0 else None

    def supported(self, rows):
        if self.ws is None or os.environ.get('SB200_TC5', '1') == '0':
            return False
        d = self.net.desc()
        return bool(_lib.lib().sb200_mlp_tc5_supported(C.byref(d), int(rows)))

    def __call__(self, x, out, zf_stats=None, zf_eps=1e-5, x_next=None, win_n=0, params=None):
        """x: [rows, D] (contiguous rows) or [B, n, D] + x_next [B, 1, D] with win_n = n; out: [rows, out_dim]."""
        net = self.net
        r = Rows()
        if win_n > 0:
            _f32c(x), _f32c(x_next)
            r.x, r.x_next, r.ldx, r.rows, r.win_n = x.data_ptr(), x_next.data_ptr(), net.dims[0], x.shape[0] * (win_n + 1), win_n
        else:
            x2 = x.reshape(-1, x.shape[-1])
            assert x2.stride(1) == 1
            r.x, r.x_next, r.ldx, r.rows, r.win_n = x2.data_ptr(), None, x2.stride(0), x2.shape[0], 0
        r.aux, r.aux_ld, r.save_x, r.ld_save_x = None, 0, None, 0
        zf = zfilter_desc(zf_stats, zf_eps)
        d = net.desc(params)
        check(_lib.lib().sb200_mlp_forward_tc5_f32(C.byref(d), C.byref(zf), C.byref(r), _ptr(out), out.stride(0), _ptr(self.ws),
                                                   _stream()), 'sb200_mlp_forward_tc5_f32')
        return out


_dual_side = {}


def mlp_forward_dual(net, x, zf_stats=None, zf_eps=1e-5, out=None, frac=None):
    """Large-batch forward with BOTH math pipes busy: the first part of the rows runs on tensor cores (3xTF32
    mma.sync tiles), the rest on the fp32 FMA pipe, as two kernels that fit one SM together, launched on two
    streams (a fork / join inside a captured graph).  Each alone is bound by its own pipe's issue rate
    (mma.sync TF32: ~48 TFLOP/s effective after the 3x split; FFMA: 72 TFLOP/s peak)."""
    import os
    rows = x.shape[0]
    frac = float(os.environ.get('SB200_DUAL_FRAC', '0.5')) if frac is None else frac
    r1 = int(rows * frac) // 64 * 64
    if r1 <= 0 or r1 >= rows:
        return mlp_forward(net, x, zf_stats=zf_stats, zf_eps=zf_eps, out=out)
    if out is None:
        out = torch.empty(rows, net.dims[-1], dtype=torch.float32, device=x.device)
    main = torch.cuda.current_stream()
    side = _dual_side.get(x.device)
    if side is None:
        side = _dual_side[x.device] = torch.cuda.Stream(device=x.device)
    side.wait_stream(main)
    mlp_forward(net, x[:r1], zf_stats=zf_stats, zf_eps=zf_eps, out=out[:r1], variant=1)
    with torch.cuda.stream(side):
        mlp_forward(net, x[r1:], zf_stats=zf_stats, zf_eps=zf_eps, out=out[r1:], variant=2)
    main.wait_stream(side)
    return out


def mlp_forward(net, x, zf_stats=None, zf_eps=1e-5, x_next=None, win_n=0, aux=None, save_all=False,
                params=None, out=None, rows=None, ldx=None, saves=None, save_x=None, variant=0):
    """Run the fused forward.

    ``x``: [rows, D] (any row stride via ``ldx``), or [B, n, D] with ``x_next`` [B, 1, D] and win_n=n for
    the virtual cat of ppo.py:376-383.  Returns the network output [rows, out_dim]; with ``save_all`` a
    list of every layer's post-activation output.  ``saves``: optional explicit list of per-layer output
    buffers ([rows, ld] each, or None) -- used by MlpTrainer; ``save_x`` receives the z-filtered input."""
    L = _lib.lib()
    assert x.is_cuda and x.dtype == torch.float32
    D = net.dims[0]
    r = Rows()
    if win_n > 0:
        _f32c(x), _f32c(x_next)
        B = x.shape[0]
        assert x.shape[1] == win_n and x.shape[2] == D
        nrows = B * (win_n + 1)
        r.x, r.x_next, r.ldx, r.rows, r.win_n = x.data_ptr(), x_next.data_ptr(), D, nrows, win_n
    else:
        if rows is None:
            x2 = x.reshape(-1, x.shape[-1]) if x.is_contiguous() else x
            assert x2.dim() == 2 and x2.stride(1) == 1
            nrows, stride = x2.shape[0], x2.stride(0)
        else:
            nrows, stride = rows, ldx
            x2 = x
        r.x, r.x_next, r.ldx, r.rows, r.win_n = x2.data_ptr(), None, stride, nrows, 0
    if net.aux_layer >= 0:
        assert aux is not None and aux.is_cuda and aux.stride(-1) == 1
        r.aux, r.aux_ld = aux.data_ptr(), aux.stride(0)
    else:
        r.aux, r.aux_ld = None, 0
    if save_x is not None:
        r.save_x, r.ld_save_x = save_x.data_ptr(), save_x.stride(0)
    else:
        r.save_x, r.ld_save_x = None, 0
    outs = []
    if saves is None:
        saves = [None] * net.n_layers
        for l in range(net.n_layers):
            last = l == net.n_layers - 1
            if save_all or last:
                t = out if (last and out is not None) else torch.empty(nrows, net.dims[l + 1], dtype=torch.float32,
                                                                       device=x.device)
                saves[l] = t
                outs.append(t)
    saves = list(saves) + [None] * (MAX_LAYERS - len(saves))
    sv = (C.c_void_p * MAX_LAYERS)(*[(t.data_ptr() if t is not None else None) for t in saves])
    ld = (C.c_int64 * MAX_LAYERS)(*[(t.stride(0) if t is not None else 0) for t in saves])
    zf = zfilter_desc(zf_stats, zf_eps)
    d = net.desc(params)
    if variant:
        check(L.sb200_mlp_forward_variant_f32(C.byref(d), C.byref(zf), C.byref(r), sv, ld, int(variant), _stream()),
              'sb200_mlp_forward_variant_f32')
    else:
        check(L.sb200_mlp_forward_f32(C.byref(d), C.byref(zf), C.byref(r), sv, ld, _stream()), 'sb200_mlp_forward_f32')
    if not outs:
        return None
    return outs if save_all else outs[-1]


class MlpTrainer:
    """Forward-with-saved-activations, hand-written backward and Adam for one FlatNet on a fixed
    batch size M.  All buffers are allocated once; every method only launches kernels (graph-safe)."""

    def __init__(self, net, M, lr, clip_mode=0, clip_value=0.0, weight_decay=0.0, splits=None, input_grad=False):
        L = _lib.lib()
        self.net, self.M = net, M
        dev = net.device
        self.splits = splits if splits is not None else max(1, min(16, M // 128))
        z = lambda *sh: torch.zeros(*sh, dtype=torch.float32, device=dev)  # noqa: E731
        self.slabs = z(self.splits, net.size)
        self.grad, self.exp_avg, self.exp_avg_sq = z(net.size), z(net.size), z(net.size)
        self.ws = torch.zeros(L.sb200_optim_workspace_bytes(), dtype=torch.uint8, device=dev)
        self.lr = torch.tensor([lr], dtype=torch.float64, device=dev)
        self.clip_mode, self.clip_value, self.weight_decay = clip_mode, float(clip_value), float(weight_decay)
        self.x_in = z(M, _ru(net.dims[0], 4))
        self.h = [z(M, _ru(n, 4)) for n in net.dims[1:]]          # post-activation outputs
        self.d = [z(M, _ru(n, 4)) for n in net.dims[1:]]          # gradients w.r.t. pre-activations
        self.aux = None
        self._aux_pad = None
        # gradient w.r.t. the pre-activation of whatever produced the network input (times relu'(input)): the CNN stem's
        # Linear layer sits in front of the PPO heads in pixel mode
        # 'aux': the gradient w.r.t. the aux input of layer 0 instead (times relu'(aux)): the CNN features next to the low-dim
        # inputs of a mixed observation
        dx0_w = net.aux_dim if input_grad == 'aux' else net.dims[0]
        self.dx0 = z(M, _ru(dx0_w, 4)) if input_grad else None
        self.input_grad = input_grad            # True / 'relu': times relu'(input) (CNN stem's Linear+ReLU); 'linear': as is (LSTM output)
        self.overlap_dw = os.environ.get('SB200_OVERLAP_DW', '1') != '0'
        self._side = None
        if net.aux_layer >= 0 and net.aux_dim % 4 != 0:       # pre-allocated: nothing may allocate during graph capture
            self._aux_pad = z(M, _ru(net.aux_dim, 4))

    @property
    def out(self):
        return self.h[-1][:, :self.net.dims[-1]]

    def forward(self, x, zf_stats=None, zf_eps=1e-5, aux=None, rows=None, ldx=None):
        if aux is not None and (aux.stride(0) % 4 != 0 or aux.data_ptr() % 16 != 0):
            # the backward GEMMs read rows with 16-byte vector loads: re-home odd-width aux inputs once
            if self._aux_pad is None:
                self._aux_pad = torch.zeros(self.M, _ru(self.net.aux_dim, 4), dtype=torch.float32,
                                            device=self.net.device)
            self._aux_pad[:, :self.net.aux_dim].copy_(aux[:, :self.net.aux_dim])
            aux = self._aux_pad
        self.aux = aux
        mlp_forward(self.net, x, zf_stats=zf_stats, zf_eps=zf_eps, aux=aux, rows=rows, ldx=ldx,
                    saves=self.h, save_x=self.x_in)
        return self.out

    def backward(self, need_dx0=False):
        """self.d[-1] must hold dL/d(pre-activation of the last layer).

        The dX chain (layer l needs dY_l and W_l) is the critical path; the weight-gradient GEMMs (dW_l needs dY_l and
        the saved input of layer l) hang off it.  With ``overlap_dw`` they are launched on a side stream that forks
        after each dY_l is ready and joins before step(): inside a captured graph these become parallel branches."""
        L, net, M = _lib.lib(), self.net, self.M
        base = self.slabs.data_ptr()
        main = torch.cuda.current_stream()
        side = None
        if self.overlap_dw:
            if self._side is None:
                self._side = torch.cuda.Stream(device=net.device)
            side = self._side

        def dw_layer(l, st):
            lay = net.layout[l]
            K0, N, ldw = net.dims[l], lay['N'], lay['ldw']
            X = self.x_in if l == 0 else self.h[l - 1]
            dY = self.d[l]
            check(L.sb200_linear_bwd_dw_f32(_ptr(X), X.stride(0), _ptr(dY), dY.stride(0),
                                            C.c_void_p(base + 4 * lay['w']), C.c_void_p(base + 4 * lay['b']),
                                            net.size, self.splits, ldw, M, K0, N, st), 'sb200_linear_bwd_dw_f32')
            if net.aux_layer == l:
                a = self.aux
                check(L.sb200_linear_bwd_dw_f32(_ptr(a), a.stride(0), _ptr(dY), dY.stride(0),
                                                C.c_void_p(base + 4 * (lay['w'] + K0 * ldw)), None, net.size,
                                                self.splits, ldw, M, net.aux_dim, N, st), 'sb200_linear_bwd_dw_f32(aux)')

        for l in reversed(range(net.n_layers)):
            lay = net.layout[l]
            K0, N, ldw = net.dims[l], lay['N'], lay['ldw']
            dY = self.d[l]
            if side is not None:
                side.wait_stream(main)                  # dY_l is ready on the main stream
            if l > 0:                                   # critical path first
                Xa = self.h[l - 1]
                dX = self.d[l - 1]
                check(L.sb200_linear_bwd_dx_f32(_ptr(dY), dY.stride(0), C.c_void_p(net.params.data_ptr() + 4 * lay['w']),
                                                ldw, _ptr(Xa), Xa.stride(0), _ptr(dX), dX.stride(0), M, N, K0, _stream()),
                      'sb200_linear_bwd_dx_f32')
            if side is not None:
                with torch.cuda.stream(side):
                    dw_layer(l, _stream())
            else:
                dw_layer(l, _stream())
        if self.input_grad == 'aux':
            lay = net.layout[0]
            w_aux = net.params.data_ptr() + 4 * (lay['w'] + net.dims[0] * lay['ldw'])
            check(L.sb200_linear_bwd_dx_f32(_ptr(self.d[0]), self.d[0].stride(0), C.c_void_p(w_aux), lay['ldw'], _ptr(self.aux),
                                            self.aux.stride(0), _ptr(self.dx0), self.dx0.stride(0), M, lay['N'], net.aux_dim,
                                            _stream()), 'sb200_linear_bwd_dx_f32(aux input)')
        elif self.dx0 is not None:
            lay = net.layout[0]
            check(L.sb200_linear_bwd_dx_f32(_ptr(self.d[0]), self.d[0].stride(0), C.c_void_p(net.params.data_ptr() + 4 * lay['w']),
                                            lay['ldw'], _ptr(None if self.input_grad == 'linear' else self.x_in), self.x_in.stride(0), _ptr(self.dx0), self.dx0.stride(0), M,
                                            lay['N'], net.dims[0], _stream()), 'sb200_linear_bwd_dx_f32(input)')
        if side is not None:
            main.wait_stream(side)

    def backward_inputs(self, stop_layer=1):
        """Only the dX chain from the last layer down to ``stop_layer`` (fills self.d[stop_layer-1 ...]); no weight
        gradients -- the DDPG actor loss back-propagates THROUGH the critic without updating it."""
        L, net, M = _lib.lib(), self.net, self.M
        for l in reversed(range(stop_layer + 1, net.n_layers)):
            lay = net.layout[l]
            dY, Xa, dX = self.d[l], self.h[l - 1], self.d[l - 1]
            check(L.sb200_linear_bwd_dx_f32(_ptr(dY), dY.stride(0), C.c_void_p(net.params.data_ptr() + 4 * lay['w']),
                                            lay['ldw'], _ptr(Xa), Xa.stride(0), _ptr(dX), dX.stride(0), M, lay['N'],
                                            net.dims[l], _stream()), 'sb200_linear_bwd_dx_f32')

    def grad_wrt_aux(self, l, out):
        """d loss / d aux input of layer l (the DDPG actor gradient dQ/da, ddpg.py:324-330)."""
        L, net = _lib.lib(), self.net
        lay = net.layout[l]
        dY = self.d[l]
        w_aux = net.params.data_ptr() + 4 * (lay['w'] + net.dims[l] * lay['ldw'])
        check(L.sb200_linear_bwd_dx_f32(_ptr(dY), dY.stride(0), C.c_void_p(w_aux), lay['ldw'], None, 0, _ptr(out),
                                        out.stride(0), self.M, lay['N'], net.aux_dim, _stream()),
              'sb200_linear_bwd_dx_f32(aux)')

    def step(self, norm_out=None, stop_flag=None):
        L, net = _lib.lib(), self.net
        st = _stream()
        dp = getattr(self, 'dp', None)
        if dp is None:
            check(L.sb200_grad_reduce_norm_f32(_ptr(self.slabs), net.size, self.splits, _ptr(self.grad), net.size,
                                               1.0, 1, _ptr(self.ws), _ptr(stop_flag), st),
                  'sb200_grad_reduce_norm_f32')
        else:
            # local slabs -> local grad; ONE flat all-reduce; average + global norm + step count
            check(L.sb200_grad_reduce_norm_f32(_ptr(self.slabs), net.size, self.splits, _ptr(self.grad), net.size,
                                               1.0, 0, _ptr(self.ws), None, st), 'sb200_grad_reduce_norm_f32')
            # one kernel over NVLink peer memory: all-reduce + average + global norm + step count; else NCCL + a second pass
            if not (hasattr(dp, 'reduce_grad_') and dp.reduce_grad_(self.grad, self.ws, stop_flag)):
                check(L.sb200_grad_reduce_norm_f32(_ptr(self.grad), net.size, 1, _ptr(self.grad), net.size,
                                                   1.0 / dp.world, 1, _ptr(self.ws), _ptr(stop_flag), st),
                      'sb200_grad_reduce_norm_f32')
        check(L.sb200_clip_adam_f32(_ptr(net.params), _ptr(self.grad), _ptr(self.exp_avg), _ptr(self.exp_avg_sq),
                                    net.size, _ptr(self.lr), 0.9, 0.999, 1e-8, self.weight_decay, self.clip_mode,
                                    self.clip_value, _ptr(self.ws), _ptr(norm_out), _ptr(stop_flag), st),
              'sb200_clip_adam_f32')

    def set_lr(self, lr):
        self.lr.fill_(float(lr))

    def state_dict(self):
        """Adam moments (kernel layout), the optimiser workspace (holds the step count) and the learning rate."""
        return {'exp_avg': self.exp_avg.detach().clone(), 'exp_avg_sq': self.exp_avg_sq.detach().clone(),
                'workspace': self.ws.detach().clone(), 'lr': float(self.lr.item()), 'layout': list(self.net.dims)}

    def load_state_dict(self, sd):
        assert list(sd['layout']) == list(self.net.dims), 'optimizer state belongs to a different network'
        self.exp_avg.copy_(torch.as_tensor(sd['exp_avg']).to(self.net.device))
        self.exp_avg_sq.copy_(torch.as_tensor(sd['exp_avg_sq']).to(self.net.device))
        self.ws.copy_(torch.as_tensor(sd['workspace']).to(self.net.device))
        self.set_lr(sd['lr'])


class EpochKernel:
    """Argument block (`sb200_epochs`) of the persistent learner kernel for ONE optimiser, bound to one MlpTrainer:
    ``mode`` 0 clip / 1 adapt (policy) or 2 (value).  Built once (fixed buffers: graph-safe); two of them make an
    EpochPair, which is what launches (csrc/epoch2.cu)."""

    def __init__(self, trainer, mode, x, ldx, M, zf_stats, zf_eps, stats, epochs, norm_out=None, stop_flag=None,
                 actions=None, lda=0, adv=None, behave_pd=None, ldb=0, ref_pd=None, ldr=0, returns=None, hyper=None,
                 eta=0.0, kl_target=0.0, stop_threshold=0.0, cta_shift=0, grid=None):
        from ._lib import Epochs
        L = _lib.lib()
        net = trainer.net
        assert M == trainer.M
        self.trainer = trainer
        self._desc = net.desc()
        self._keep = (x, zf_stats, stats, norm_out, stop_flag, actions, adv, behave_pd, ref_pd, returns, hyper)
        a = Epochs()
        a.net = C.addressof(self._desc)
        a.params, a.n_params, a.extra_off = net.params.data_ptr(), net.size, net.extra_off
        a.x, a.ldx, a.M = x.data_ptr(), int(ldx), int(M)
        a.zf_stats = zf_stats.data_ptr() if zf_stats is not None else None
        a.zf_eps = float(zf_eps)
        h, d = trainer.h, trainer.d
        a.x_in = trainer.x_in.data_ptr()
        a.h1, a.h2, a.out, a.d1, a.d2, a.dpre = (h[0].data_ptr(), h[1].data_ptr(), h[2].data_ptr(), d[0].data_ptr(),
                                                 d[1].data_ptr(), d[2].data_ptr())
        a.slabs, a.splits, a.grad = trainer.slabs.data_ptr(), trainer.splits, trainer.grad.data_ptr()
        a.exp_avg, a.exp_avg_sq = trainer.exp_avg.data_ptr(), trainer.exp_avg_sq.data_ptr()
        a.lr, a.weight_decay = trainer.lr.data_ptr(), trainer.weight_decay
        a.clip_mode, a.clip_value = trainer.clip_mode, trainer.clip_value
        a.opt_workspace = trainer.ws.data_ptr()
        a.norm_out = norm_out.data_ptr() if norm_out is not None else None
        a.mode = int(mode)
        g = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
        a.actions, a.lda, a.adv = g(actions), int(lda), g(adv)
        a.behave_pd, a.ldb, a.ref_pd, a.ldr = g(behave_pd), int(ldb), g(ref_pd), int(ldr)
        a.returns, a.hyper = g(returns), g(hyper)
        a.eta, a.kl_target, a.stop_threshold = float(eta), float(kl_target), float(stop_threshold)
        a.stats, a.stop_flag, a.epochs = stats.data_ptr(), g(stop_flag), int(epochs)
        a.workspace = None                                  # the pair owns the workspace
        a.grid = int(grid) if grid is not None else 0            # 0: one CTA per SM (the library asks the device)
        a.cta_shift = int(cta_shift)
        a.par = None
        self.args = a

    def set_peer(self, peer):
        """Data-parallel: average the KL scalar and the flat gradient over the ranks of ``peer`` (a PeerChannel) in-kernel."""
        self._peer = peer
        self.args.par = C.addressof(peer.ctx) if peer is not None else None



class EpochPair:
    """Second-generation persistent learner kernel (csrc/epoch2.cu): the policy optimiser AND the value optimiser of one
    ``learn()`` in ONE launch.  Built from two EpochKernel argument blocks (``value`` may be None)."""

    def __init__(self, policy, value=None):
        L = _lib.lib()
        self.policy, self.value = policy, value
        self._pa = C.byref(policy.args)
        self._va = C.byref(value.args) if value is not None else None
        nbytes = int(L.sb200_ppo_epochs2_workspace_bytes(self._pa, self._va))
        assert nbytes > 0
        self.ws = torch.zeros(nbytes + 256, dtype=torch.uint8, device=policy.trainer.net.device)
        self._ws_ptr = (self.ws.data_ptr() + 255) // 256 * 256

    @staticmethod
    def supported(policy, value=None):
        return bool(_lib.lib().sb200_ppo_epochs2_supported(C.byref(policy.args), C.byref(value.args) if value is not None else None))

    def run(self):
        check(_lib.lib().sb200_ppo_epochs2_f32(self._pa, self._va, C.c_void_p(self._ws_ptr), _stream()), 'sb200_ppo_epochs2_f32')
        return self.policy.trainer.out

    PHASES = ('setup', 'P1 rows', 'barrier', 'gate+stats', 'P2 dW', 'barrier', 'P3 reduce', 'barrier', 'P4 adam', 'barrier')

    def profile(self, reset=True):
        """Accumulated clock64 cycles per phase since the last reset: [(phase, CTA 0, last CTA)]."""
        buf = (C.c_uint64 * 32)()
        check(_lib.lib().sb200_ppo_epochs2_profile(C.c_void_p(self._ws_ptr), buf, int(reset), _stream()), 'sb200_ppo_epochs2_profile')
        return [(name, int(buf[i]), int(buf[16 + i])) for i, name in enumerate(self.PHASES)]

    def cta_profile(self):
        """Per-CTA accumulated cycles [192][8] (0 P1, 1 P2, 2 forward, 3 forward GEMMs, 4 loss rows + d2, 5 d1 GEMM); cleared on read."""
        buf = (C.c_uint64 * (192 * 8))()
        check(_lib.lib().sb200_ppo_epochs2_cta_profile(C.c_void_p(self._ws_ptr), buf, _stream()), 'sb200_ppo_epochs2_cta_profile')
        return [[int(buf[c * 8 + k]) for k in range(8)] for c in range(192)]


class GraphRunner:
    """Capture a fixed launch sequence once into a CUDA graph and replay it (B200: a launch-bound inner loop of
    hundreds of small kernels becomes ONE submission).  Capture records without executing, so state is advanced
    exactly once per call: the first call captures and immediately replays."""

    def __init__(self):
        self.graph = None
        self.kernels = 0

    def run(self, fn):
        L = _lib.lib()
        if self.graph is None:
            import gc
            _lib.ensure_device()
            # Objects of earlier learners (captured graphs with private memory pools) may be waiting for the garbage
            # collector; if it ran DURING the capture their cudaFree would invalidate it (cudaErrorStreamCaptureInvalidated:
            # seen in the full test suite, never in a fresh process).  Collect now, keep the collector off while capturing.
            gc.collect()
            torch.cuda.synchronize()
            before = int(L.sb200_launch_counter(0))
            g = torch.cuda.CUDAGraph()
            gc_was_on = gc.isenabled()
            gc.disable()
            try:
                with torch.cuda.graph(g):
                    fn()
            finally:
                if gc_was_on:
                    gc.enable()
            self.kernels = int(L.sb200_launch_counter(0)) - before    # recorded, not yet executed
            L.sb200_launch_counter_add(C.c_uint64(-self.kernels & 0xFFFFFFFFFFFFFFFF))
            self.graph = g
        self.graph.replay()
        L.sb200_launch_counter_add(self.kernels)


def graphs_enabled():
    import os
    return os.environ.get('SB200_CUDA_GRAPH', '1') != '0'


_gae_ws = {}


def gae_window(rewards, values, dones, gamma, lam, horizon=None, norm_adv=True, reward_scale=1.0, adv=None, ret=None,
               ws=None):
    """rewards [B,n], values [B,n+1] raw critic output, dones [B,n] -> (adv [B,E], ret [B,E])."""
    L = _lib.lib()
    _f32c(rewards), _f32c(values), _f32c(dones)
    B, n = rewards.shape
    H = n if horizon is None else int(horizon)
    E = n - H + 1
    if adv is None:
        adv = torch.empty(B, E, dtype=torch.float32, device=rewards.device)
    if ret is None:
        ret = torch.empty(B, E, dtype=torch.float32, device=rewards.device)
    if ws is None:
        key = rewards.device
        if key not in _gae_ws:
            _gae_ws[key] = torch.zeros(max(16, L.sb200_gae_workspace_bytes(B, n, H)), dtype=torch.uint8,
                                       device=rewards.device)
        ws = _gae_ws[key]
    check(L.sb200_gae_window_f32(_ptr(rewards), _ptr(values), _ptr(dones), B, n, H, float(gamma), float(lam),
                                 float(reward_scale), int(bool(norm_adv)), _ptr(adv), _ptr(ret), _ptr(ws),
                                 _stream()), 'sb200_gae_window_f32')
    return adv, ret


def make_pd(mean, log_var, B, A, pd, log_noise=None):
    check(_lib.lib().sb200_make_pd_f32(_ptr(mean), mean.stride(0), _ptr(log_var), _ptr(log_noise), B, A, _ptr(pd),
                                       pd.stride(0), _stream()), 'sb200_make_pd_f32')
    return pd


def zfilter_update(x, rows, D, ldx, stats):
    check(_lib.lib().sb200_zfilter_update_f32(_ptr(x), ldx, rows, D, _ptr(stats), _stream()), 'sb200_zfilter_update_f32')
