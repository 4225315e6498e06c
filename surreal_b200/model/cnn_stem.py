"""CNN stem of the pixel path -- host-side mirror of CNNStemNetwork (surreal/model/model_builders/builders.py:8-33):

    uint8 frames / 255 -> Conv2d(16, k8, s4) + ReLU -> Conv2d(32, k4, s2) + ReLU -> Flatten -> Linear(D_out) + ReLU

All parameters live in ONE flat fp32 device buffer (conv weights in the kernel layout [(c, ky, kx)][COUT], the Linear layer in
FlatNet's [in][out] layout), so that each of the two optimisers that train the shared stem (ppo_net.py:202-224) keeps its
own flat Adam state over it and the data-parallel learner reduces it with one collective.  The convolutions are
csrc/stem.cu, the Linear layer the MLP kernels (csrc/mlp_fwd*.cu, mlp_bwd.cu)."""
import collections
import ctypes as C

import torch

from .. import _lib, ops
from .._lib import check


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _conv_out(h, k, s):
    return (h - k) // s + 1


class CNNStem:
    K1, S1, C1 = 8, 4, 16
    K2, S2, C2 = 4, 2, 32

    def __init__(self, obs_shape, d_out, device):
        self.C, self.H, self.W = (int(v) for v in obs_shape)
        self.d_out = int(d_out)
        self.device = torch.device(device)
        self.H1, self.W1 = _conv_out(self.H, self.K1, self.S1), _conv_out(self.W, self.K1, self.S1)
        self.H2, self.W2 = _conv_out(self.H1, self.K2, self.S2), _conv_out(self.W1, self.K2, self.S2)
        assert self.H2 >= 1 and self.W2 >= 1, 'frame too small for the k8s4 / k4s2 stem'
        self.taps1, self.taps2 = self.C * self.K1 * self.K1, self.C1 * self.K2 * self.K2
        self.flat = self.C2 * self.H2 * self.W2
        # flat parameter layout: [conv1 Wk | b1 | conv2 Wk | b2 | fc (FlatNet layout: W[flat][ldw] | b[ldw])]
        o = 0
        self.off = {}
        for name, n in (('w1', self.taps1 * self.C1), ('b1', self.C1), ('w2', self.taps2 * self.C2), ('b2', self.C2)):
            self.off[name] = (o, n)
            o += n
        self.fc = ops.FlatNet([self.flat, self.d_out], [ops.ACT_RELU], self.device)
        self.off['fc'] = (o, self.fc.size)
        self.size = o + self.fc.size
        self.params = torch.zeros(self.size, dtype=torch.float32, device=self.device)
        self.fc.params = self.seg('fc')                          # the FlatNet now lives inside the stem's flat buffer
        self._init_default()

    # -- views / parameters ---------------------------------------------------------------------------------------
    def seg(self, name, buf=None):
        o, n = self.off[name]
        return (self.params if buf is None else buf)[o:o + n]

    def _init_default(self):
        """torch's default Conv2d / Linear initialisation (torchx's own default is unpinned; parity tests inject weights)."""
        c1 = torch.nn.Conv2d(self.C, self.C1, self.K1, self.S1)
        c2 = torch.nn.Conv2d(self.C1, self.C2, self.K2, self.S2)
        fc = torch.nn.Linear(self.flat, self.d_out)
        self.load_torch(c1.weight.detach(), c1.bias.detach(), c2.weight.detach(), c2.bias.detach(), fc.weight.detach(),
                        fc.bias.detach())

    def load_torch(self, w1, b1, w2, b2, wfc, bfc):
        """torch layouts: conv [COUT][C][k][k], linear [out][in]."""
        f = lambda t: torch.as_tensor(t, dtype=torch.float32)  # noqa: E731
        self.seg('w1').copy_(f(w1).reshape(self.C1, -1).t().contiguous().reshape(-1).to(self.device))
        self.seg('b1').copy_(f(b1).to(self.device))
        self.seg('w2').copy_(f(w2).reshape(self.C2, -1).t().contiguous().reshape(-1).to(self.device))
        self.seg('b2').copy_(f(b2).to(self.device))
        self.fc.set_layer(0, f(wfc), f(bfc))

    def state_items(self, prefix='cnn_stem.model.seq.'):
        """(key, tensor) pairs under the reference's module names (Sequential indices 0, 2, 5; builders.py:11-18)."""
        w1 = self.seg('w1').view(self.taps1, self.C1).t().reshape(self.C1, self.C, self.K1, self.K1).clone()
        w2 = self.seg('w2').view(self.taps2, self.C2).t().reshape(self.C2, self.C1, self.K2, self.K2).clone()
        wfc, bfc = self.fc.get_layer(0)
        return [(prefix + '0.weight', w1), (prefix + '0.bias', self.seg('b1').clone()), (prefix + '2.weight', w2),
                (prefix + '2.bias', self.seg('b2').clone()), (prefix + '5.weight', wfc), (prefix + '5.bias', bfc)]

    def load_state(self, sd, prefix='cnn_stem.model.seq.'):
        self.load_torch(sd[prefix + '0.weight'], sd[prefix + '0.bias'], sd[prefix + '2.weight'], sd[prefix + '2.bias'],
                        sd[prefix + '5.weight'], sd[prefix + '5.bias'])

    # -- forward --------------------------------------------------------------------------------------------------
    def buffers(self, rows):
        f = lambda *s: torch.empty(*s, dtype=torch.float32, device=self.device)  # noqa: E731
        return dict(a1=f(rows, self.C1, self.H1, self.W1), a2=f(rows, self.flat), feat=f(rows, self.d_out))

    def forward(self, frames, bufs, params=None, rows=None, row_bytes=None):
        """frames: uint8 [rows, C, H, W] contiguous (raw 0..255; scaled by 1/255 inside, ppo_net.py:370) -> feat [rows, d_out].
        With ``row_bytes``, ``frames`` is any CUDA tensor whose first byte is the first frame and ``rows`` frames sit
        ``row_bytes`` apart (read in place from mixed observation records, utils.obs_layout).
        ``bufs`` (from ``buffers(rows)``) receives the intermediate activations a1 / a2 (needed by the backward pass)."""
        L, st = _lib.lib(), ops._stream()
        P = self.params if params is None else params
        if row_bytes is None:
            assert frames.dtype == torch.uint8 and frames.is_cuda and frames.is_contiguous()
            rows = frames.shape[0]
            check(L.sb200_conv_forward_f32(1, _p(frames), 1, rows, self.C, self.H, self.W, _p(self.seg('w1', P)),
                                           _p(self.seg('b1', P)), 1.0 / 255.0, _p(bufs['a1']), st), 'sb200_conv_forward_f32(1)')
        else:
            assert frames.is_cuda and row_bytes >= self.C * self.H * self.W
            check(L.sb200_conv1_forward_u8_strided(_p(frames), int(row_bytes), rows, self.C, self.H, self.W, _p(self.seg('w1', P)),
                                                   _p(self.seg('b1', P)), 1.0 / 255.0, _p(bufs['a1']), st),
                  'sb200_conv1_forward_u8_strided')
        check(L.sb200_conv_forward_f32(2, _p(bufs['a1']), 0, rows, self.C1, self.H1, self.W1, _p(self.seg('w2', P)),
                                       _p(self.seg('b2', P)), 1.0, _p(bufs['a2']), st), 'sb200_conv_forward_f32(2)')
        ops.mlp_forward(self.fc, bufs['a2'], params=self.seg('fc', P), out=bufs['feat'])
        return bufs['feat']


class StemTrainer:
    """Saved activations, backward and gradient slabs of the stem for ONE optimiser on a fixed number of frames M."""

    def __init__(self, stem, M, splits=None):
        self.stem, self.M = stem, M
        dev = stem.device
        self.splits = splits if splits is not None else max(1, min(16, M // 16))
        z = lambda *s: torch.zeros(*s, dtype=torch.float32, device=dev)  # noqa: E731
        self.bufs = stem.buffers(M)
        self.slabs = z(self.splits, stem.size)
        self.exp_avg, self.exp_avg_sq = z(stem.size), z(stem.size)
        self.d_fc = z(M, ops._ru(stem.d_out, 4))                  # gradient w.r.t. the Linear layer's pre-activation
        self.d_a2 = z(M, stem.flat)                               # ... conv2's pre-activation
        self.d_a1 = z(M, stem.C1, stem.H1, stem.W1)               # ... conv1's pre-activation
        self.frames = None
        self.row_bytes = None

    def forward(self, frames, row_bytes=None):
        """``row_bytes``: the M frames are read in place, ``row_bytes`` apart (see CNNStem.forward)."""
        self.frames, self.row_bytes = frames, row_bytes
        return self.stem.forward(frames, self.bufs, rows=self.M, row_bytes=row_bytes)

    def backward(self, d_feat_pre):
        """``d_feat_pre`` [M, >= d_out]: gradient w.r.t. the Linear layer's PRE-activation (the head's input gradient already
        multiplied by relu'(feat)).  Fills the slabs with partial gradients of every stem parameter."""
        s, L, st = self.stem, _lib.lib(), ops._stream()
        M, b = self.M, self.bufs
        base = self.slabs.data_ptr()
        o_fc = s.off['fc'][0]
        lay = s.fc.layout[0]
        # Linear: dW / db into the slabs, dX (times relu'(a2)) -> conv2's pre-activation gradient
        check(L.sb200_linear_bwd_dw_f32(_p(b['a2']), b['a2'].stride(0), _p(d_feat_pre), d_feat_pre.stride(0),
                                        C.c_void_p(base + 4 * (o_fc + lay['w'])), C.c_void_p(base + 4 * (o_fc + lay['b'])),
                                        s.size, self.splits, lay['ldw'], M, s.flat, s.d_out, st), 'sb200_linear_bwd_dw_f32(stem fc)')
        check(L.sb200_linear_bwd_dx_f32(_p(d_feat_pre), d_feat_pre.stride(0), C.c_void_p(s.fc.params.data_ptr() + 4 * lay['w']),
                                        lay['ldw'], _p(b['a2']), b['a2'].stride(0), _p(self.d_a2), self.d_a2.stride(0), M, s.d_out,
                                        s.flat, st), 'sb200_linear_bwd_dx_f32(stem fc)')
        o_w2, o_b2 = s.off['w2'][0], s.off['b2'][0]
        check(L.sb200_conv_backward_dw_f32(2, _p(b['a1']), 0, _p(self.d_a2), M, s.C1, s.H1, s.W1, 1.0, C.c_void_p(base + 4 * o_w2),
                                           C.c_void_p(base + 4 * o_b2), s.size, self.splits, st), 'sb200_conv_backward_dw_f32(2)')
        check(L.sb200_conv_backward_dx_f32(2, _p(self.d_a2), _p(s.seg('w2')), _p(b['a1']), M, s.C1, s.H1, s.W1, _p(self.d_a1), st),
              'sb200_conv_backward_dx_f32')
        o_w1, o_b1 = s.off['w1'][0], s.off['b1'][0]
        if self.row_bytes is None:
            check(L.sb200_conv_backward_dw_f32(1, _p(self.frames), 1, _p(self.d_a1), M, s.C, s.H, s.W, 1.0 / 255.0,
                                               C.c_void_p(base + 4 * o_w1), C.c_void_p(base + 4 * o_b1), s.size, self.splits, st),
                  'sb200_conv_backward_dw_f32(1)')
        else:
            check(L.sb200_conv1_backward_dw_u8_strided(_p(self.frames), int(self.row_bytes), _p(self.d_a1), M, s.C, s.H, s.W,
                                                       1.0 / 255.0, C.c_void_p(base + 4 * o_w1), C.c_void_p(base + 4 * o_b1),
                                                       s.size, self.splits, st), 'sb200_conv1_backward_dw_u8_strided')

    def state_dict(self):
        return {'exp_avg': self.exp_avg.detach().clone(), 'exp_avg_sq': self.exp_avg_sq.detach().clone()}

    def load_state_dict(self, sd):
        self.exp_avg.copy_(torch.as_tensor(sd['exp_avg']).to(self.stem.device))
        self.exp_avg_sq.copy_(torch.as_tensor(sd['exp_avg_sq']).to(self.stem.device))


def joint_step(head, stem_tr, grad, norm_out=None, stop_flag=None):
    """One optimiser step over a head network (ops.MlpTrainer) AND the shared stem: the reference clips the global norm of
    head + stem parameters together (get_actor_params / get_critic_params, ppo_net.py:202-224; ppo.py:244-246,349-351)
    and steps ONE Adam over both.  ``grad`` = [head gradient | stem gradient] is one contiguous buffer so that the norm
    (and a data-parallel all-reduce) sees everything at once; head.ws carries the shared step count / norm."""
    L, st = _lib.lib(), ops._stream()
    nh, ns = head.net.size, stem_tr.stem.size
    gh, gs = grad[:nh], grad[nh:nh + ns]
    sf = C.c_void_p(stop_flag.data_ptr()) if stop_flag is not None else None
    check(L.sb200_grad_reduce_norm_f32(_p(head.slabs), nh, head.splits, _p(gh), nh, 1.0, 0, _p(head.ws), sf, st),
          'sb200_grad_reduce_norm_f32(head)')
    check(L.sb200_grad_reduce_norm_f32(_p(stem_tr.slabs), ns, stem_tr.splits, _p(gs), ns, 1.0, 0, _p(head.ws), sf, st),
          'sb200_grad_reduce_norm_f32(stem)')
    dp = getattr(head, 'dp', None)
    scale = 1.0
    if dp is not None:
        dp.sum_(grad)
        scale = 1.0 / dp.world
    check(L.sb200_grad_reduce_norm_f32(_p(grad), nh + ns, 1, _p(grad), nh + ns, scale, 1, _p(head.ws), sf, st),
          'sb200_grad_reduce_norm_f32(joint norm)')
    for params, g, m, v, n, no in ((head.net.params, gh, head.exp_avg, head.exp_avg_sq, nh, norm_out),
                                   (stem_tr.stem.params, gs, stem_tr.exp_avg, stem_tr.exp_avg_sq, ns, None)):
        check(L.sb200_clip_adam_f32(_p(params), _p(g), _p(m), _p(v), n, _p(head.lr), 0.9, 0.999, 1e-8, head.weight_decay,
                                    head.clip_mode, head.clip_value, _p(head.ws), _p(no), sf, st), 'sb200_clip_adam_f32')
