"""Drop-in mirror of the reference's model facade for the TTA path, backed by the native engine.

Mirrors (same names, argument meaning and error behaviour):
  * `ExternalModel_Adapt`  -- src/external_model_adapt.py:29-660
  * `MsgChnModel_Adapt`    -- src/msg_chn_model_adapt.py:12-556
  * `OutlierRemoval`       -- src/net_utils.py:750-811
The reference driver's call sequence (src/tta_main.py:309-354, 583-633) works unchanged:

    model = ExternalModel_Adapt('msg_chn', min_predict_depth, max_predict_depth, max_input_depth, device=...)
    model._prepare_head('meta_selfsup_seq_2layers_ema'); model.restore_model(ckpt)
    optimizer = torch.optim.Adam(model.adapt_parameters('meta'), lr=...)
    out, emb, ref = model.forward(image=..., sparse_depth=..., loss_type='adapt_meta_selfsup_seq_ema_reverse')
    loss, info = model.compute_loss(input_rgb=..., output_depth=out, ..., loss_type='adapt')
    optimizer.zero_grad(); loss.backward(); optimizer.step()

plus one extension, `tta_step(...)`, which runs the whole per-frame step (outlier removal, forward,
losses, backward, Adam) inside the library without returning to Python.  All arithmetic is done by
libptta_b200.so; torch supplies device memory, streams and the autograd glue only."""
import math
from collections import OrderedDict

import torch

from . import ops
from .engine import MsgChnEngine

ADAPT_LOSS_TYPE = 'adapt_meta_selfsup_seq_ema_reverse'


class OutlierRemoval(object):
    """src/net_utils.py:750-811 -- 7x7 min-filter outlier rejection on the sparse depth."""

    def __init__(self, kernel_size=7, threshold=1.5):
        self.kernel_size = kernel_size
        self.threshold = threshold

    def remove_outliers(self, sparse_depth, validity_map=None):
        # the validity map is a function of the sparse depth (src/tta_main.py:583-586); it is recomputed in-kernel
        return ops.outlier_removal(sparse_depth.contiguous(), self.kernel_size, self.threshold)


# ---------------------------------------------------------------------------------------------------------
# parameter construction (shapes / initialisers of network_exp_msg_chn_adapt.py:166-335, 1022-1098)
# ---------------------------------------------------------------------------------------------------------
def _conv_init(sd, name, cout, cin, transposed=False):
    w = torch.empty((cin, cout, 3, 3) if transposed else (cout, cin, 3, 3))
    torch.nn.init.xavier_normal_(w)                      # :188-194
    sd[name + '.weight'] = w
    sd[name + '.bias'] = torch.full((cout,), 0.01)


def _bn_init(sd, name, c):
    sd[name + '.weight'] = torch.ones(c)
    sd[name + '.bias'] = torch.zeros(c)
    sd[name + '.running_mean'] = torch.zeros(c)
    sd[name + '.running_var'] = torch.ones(c)
    sd[name + '.num_batches_tracked'] = torch.tensor(0, dtype=torch.long)


def _default_conv_init(w):
    torch.nn.init.kaiming_uniform_(w, a=math.sqrt(5))    # nn.Conv2d / nn.Linear default
    return w


def _linear_init(sd, name, cout, cin):
    sd[name + '.weight'] = _default_conv_init(torch.empty(cout, cin))
    bound = 1.0 / math.sqrt(cin)
    sd[name + '.bias'] = torch.empty(cout).uniform_(-bound, bound)


def _mlp_init(sd, name, dim, out, hidden):
    _linear_init(sd, name + '.0', hidden, dim)
    _bn_init(sd, name + '.1', hidden)
    _linear_init(sd, name + '.3', out, hidden)


def build_base_state():
    """network_adapt.__init__ (network_exp_msg_chn_adapt.py:313-335): three depth encoder/decoder pairs + RGB encoder."""
    sd = OrderedDict()

    def encoder(prefix, cin, n_enc):
        _conv_init(sd, prefix + '.init.0', 32, cin)
        _conv_init(sd, prefix + '.init.2', 32, 32)
        for k in range(1, n_enc + 1):
            _conv_init(sd, '%s.enc%d.1' % (prefix, k), 32, 32)
            _conv_init(sd, '%s.enc%d.3' % (prefix, k), 32, 32)

    def decoder(prefix):
        for blk in ('dec2', 'dec1'):
            _conv_init(sd, '%s.%s.1' % (prefix, blk), 32, 32, transposed=True)
            _conv_init(sd, '%s.%s.3' % (prefix, blk), 32, 32)
        _conv_init(sd, prefix + '.prdct.1', 32, 32)
        _conv_init(sd, prefix + '.prdct.3', 1, 32)

    encoder('rgb_encoder', 3, 4)
    encoder('depth_encoder1', 1, 2); decoder('depth_decoder1')
    encoder('depth_encoder2', 2, 2); decoder('depth_decoder2')
    encoder('depth_encoder3', 2, 2); decoder('depth_decoder3')
    return sd


def add_head_state(sd, mode):
    """network_adapt._prepare_head (network_exp_msg_chn_adapt.py:1022-1087)."""
    if 'selfsup' in mode:
        _mlp_init(sd, 'proj', 32, 512, 512)
        if 'ema' in mode:
            for k in [k for k in sd if k.startswith('proj.')]:
                sd['proj_t.' + k[5:]] = sd[k].clone()
        _mlp_init(sd, 'pred', 512, 512, 512)
    if 'meta' in mode:
        if 'seq' not in mode:
            raise NotImplementedError('only the sequential ("seq") meta layer is implemented: %s' % mode)
        if '1layer' in mode:
            # nn.Conv2d's own initialisation first (it consumes the RNG), then the Kaiming fan-out draw over the weight (:1066-1068)
            w = _default_conv_init(torch.empty(32, 32, 3, 3))
            b = torch.empty(32).uniform_(-1.0 / math.sqrt(288), 1.0 / math.sqrt(288))
            torch.nn.init.kaiming_normal_(w, mode='fan_out', nonlinearity='relu')
            sd['conv1_rgb_meta.weight'] = w
            sd['conv1_rgb_meta.bias'] = b
        elif '2layers' in mode:
            p = 'conv1_rgb_meta.conv1_meta'
            sd[p + '.0.0.weight'] = _default_conv_init(torch.empty(128, 32, 3, 3))
            _bn_init(sd, p + '.0.1', 128)
            sd[p + '.1.weight'] = _default_conv_init(torch.empty(32, 128, 3, 3))
            sd[p + '.1.bias'] = torch.empty(32).uniform_(-1.0 / math.sqrt(1152), 1.0 / math.sqrt(1152))
            _bn_init(sd, p + '.2', 32)
        else:
            raise NotImplementedError(mode)
    return sd


_PARAM_SUFFIX = ('.weight', '.bias')


# ---------------------------------------------------------------------------------------------------------
# autograd glue: the engine computes every gradient; these Functions only route them
# ---------------------------------------------------------------------------------------------------------
class _ForwardFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, wrapper, image, sparse_depth, *params):
        eng = wrapper._engine_for(image)
        eng.pack_adapted()                     # the optimizer may have stepped the fp32 masters since the last call
        eng.forward(image, sparse_depth, None, True)     # the facade already clamped the sparse depth
        ctx.wrapper, ctx.eng, ctx.n_params = wrapper, eng, len(params)
        n, h, w = eng.n, eng.h, eng.w
        out = eng.tensor('output').view(n, 1, h, w).clone()
        emb, ref = eng.tensor('emb').view(-1, 512), eng.tensor('ref').view(-1, 512)
        ctx.mark_non_differentiable(emb)       # emb = pred(proj(z_zero.detach())): no path to the adapted tensors
        return out, emb, ref

    @staticmethod
    def backward(ctx, g_out, g_emb, g_ref):
        eng, wrapper = ctx.eng, ctx.wrapper
        go, gr = eng.tensor('g_output'), eng.tensor('g_ref')
        if g_out is not None and g_out.data_ptr() != go.data_ptr():
            go.view(-1).copy_(g_out.reshape(-1))
        if g_ref is not None and g_ref.data_ptr() != gr.data_ptr():
            gr.view(-1).copy_(g_ref.reshape(-1))
        eng.network_backward()
        grads = [wrapper._grad_views[k].clone() for k in wrapper._adapt_names]
        return (None, None, None) + tuple(grads)


class _LossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, eng, output_depth, embedding, reference, image_raw, sparse_depth, validity_map, cap, w_sd, w_sm, w_cos):
        # the engine evaluates the loss on its own copies of (output, emb, ref) from the forward that produced them
        eng.loss(image_raw, sparse_depth, validity_map, cap, w_sd, w_sm, w_cos)
        ctx.eng = eng
        scal = eng.tensor('losses').view(-1)
        loss, parts = scal[0].clone(), scal[1:4].clone()
        ctx.mark_non_differentiable(parts)
        return loss, parts

    @staticmethod
    def backward(ctx, g_loss, g_parts):
        eng = ctx.eng
        eng.loss_backward(float(g_loss))       # a host read of the upstream scalar (1.0 for loss.backward())
        n, h, w = eng.n, eng.h, eng.w
        return (None, eng.tensor('g_output').view(n, 1, h, w), None, eng.tensor('g_ref').view(-1, 512),
                None, None, None, None, None, None, None)


class _InitForwardFn(torch.autograd.Function):
    """stage-1 forward (loss_type 'init_meta...': network_exp_msg_chn_adapt.py:559-607): the real branch with the meta layer in train mode"""

    @staticmethod
    def forward(ctx, wrapper, image, sparse_depth, *params):
        eng = wrapper._engine_for(image)
        eng.pack_adapted()
        eng.forward(image, sparse_depth, None, 2)
        ctx.wrapper, ctx.eng = wrapper, eng
        return eng.tensor('output').view(eng.n, 1, eng.h, eng.w).clone()

    @staticmethod
    def backward(ctx, g_out):
        eng, wrapper = ctx.eng, ctx.wrapper
        go = eng.tensor('g_output')
        if g_out.data_ptr() != go.data_ptr():
            go.view(-1).copy_(g_out.reshape(-1))
        eng.network_backward()
        return (None, None, None) + tuple(wrapper._grad_views[k].clone() for k in wrapper._adapt_names)


class _L2LossFn(torch.autograd.Function):
    """MsgChnModel_Adapt.compute_loss(loss_type='pretrain') (src/msg_chn_model_adapt.py:224-264) on the engine's last prediction"""

    @staticmethod
    def forward(ctx, eng, output_depth, ground_truth, max_predict_depth):
        eng.l2_loss(ground_truth, max_predict_depth)
        ctx.eng = eng
        return eng.tensor('losses').view(-1)[0].clone()

    @staticmethod
    def backward(ctx, g_loss):
        eng = ctx.eng
        eng.l2_loss_backward(float(g_loss))
        return None, eng.tensor('g_output').view(eng.n, 1, eng.h, eng.w), None, None


class _HeadForwardFn(torch.autograd.Function):
    """stage-2 forward (loss_type 'head_meta_selfsup_seq_ema_reverse': network_exp_msg_chn_adapt.py:609-699, mode [reverse, seq, ema]):
    frozen network on the frame and on the zero image, EMA copy of proj, emb = pred(proj(z_zero).detach()), ref = proj(z_real).detach()"""

    @staticmethod
    def forward(ctx, wrapper, image, sparse_depth, *params):
        eng = wrapper._engine_for(image)
        eng.pack_adapted()
        eng.forward(image, sparse_depth, None, 1)
        eng.ema_update_head(0.999)
        ctx.wrapper, ctx.eng = wrapper, eng
        emb, ref = eng.tensor('emb').view(-1, 512), eng.tensor('ref').view(-1, 512)
        ctx.mark_non_differentiable(ref)
        return emb, ref

    @staticmethod
    def backward(ctx, g_emb, g_ref):
        eng, wrapper = ctx.eng, ctx.wrapper
        ge = eng.tensor('g_emb')
        if g_emb.data_ptr() != ge.data_ptr():
            ge.view(-1).copy_(g_emb.reshape(-1))
        eng.head_backward()
        return (None, None, None) + tuple(wrapper._grad_views[k].clone() for k in wrapper._adapt_names)


class _CosLossFn(torch.autograd.Function):
    """ExternalModel_Adapt.prepare_loss (src/external_model_adapt.py:524-540) on the engine's last (emb, ref)"""

    @staticmethod
    def forward(ctx, eng, embedding, reference):
        eng.cos_loss()
        ctx.eng = eng
        return eng.tensor('losses').view(-1)[0].clone()

    @staticmethod
    def backward(ctx, g_loss):
        eng = ctx.eng
        eng.cos_loss_backward(float(g_loss))
        return None, eng.tensor('g_emb').view(-1, 512), None


HEAD_TRAINED = ('pred.0.weight', 'pred.0.bias', 'pred.1.weight', 'pred.1.bias', 'pred.3.weight', 'pred.3.bias')


class MsgChnModel_Adapt(object):
    """src/msg_chn_model_adapt.py -- MSG-CHN wrapper (state dict, adapted-parameter selection, checkpoints)."""

    def __init__(self, max_predict_depth=100.0, device=torch.device('cuda')):
        self.max_predict_depth = max_predict_depth
        self.device = torch.device(device)
        self.training = True
        self.prepare_mode = None
        self._sd = build_base_state()
        self._engines = {}
        self._adapt_names = []
        self._params = None
        self._grad_views = {}
        self._flat = {}
        self.img_scale = (1.0, 1.0, 1.0)
        self.img_shift = (0.0, 0.0, 0.0)
        self._adam_step = 0
        self.engine_options = {}       # ptta_msgchn_set_option(name, value) applied to every engine this wrapper creates
        self._trainable = 'meta'       # which tensors the flat parameter / gradient / Adam buffers cover: 'meta' (TTA, stage 1) or 'head' (stage 2)

    # -- construction ---------------------------------------------------------------------------------
    def _prepare_head(self, mode=''):
        self.prepare_mode = mode
        add_head_state(self._sd, mode)
        self._materialise()

    def _materialise(self):
        """Move the state to the device; adapted tensors become views of one flat fp32 buffer (as do their
        gradients and Adam moments) so that the fused Adam kernel covers them in one launch."""
        if self.device.type != 'cuda':
            raise RuntimeError('the TTA step runs on CUDA only (no CPU fallback); got device %s' % self.device)
        for k, v in list(self._sd.items()):
            want = torch.int64 if k.endswith('num_batches_tracked') else torch.float32
            self._sd[k] = v.detach().to(self.device, want).contiguous()
        if self._trainable == 'head':           # stage 2: of the tensors head_main.py:268 hands to Adam only pred.* ever gets a gradient
            self._adapt_names = [k for k in HEAD_TRAINED if k in self._sd]
        else:
            self._adapt_names = [k for k in self._sd if 'meta' in k and k.endswith(_PARAM_SUFFIX)]   # msg_chn_model_adapt.py:392-396
        total = sum(self._sd[k].numel() for k in self._adapt_names)
        self._flat = {name: torch.zeros(total, dtype=torch.float32, device=self.device) for name in ('param', 'grad', 'm', 'v')}
        # Adam step counter + hyper-parameters: ONE device block per wrapper, bound into every engine (all shapes share the
        # moments, so they must share the bias-correction step as well)
        self._adam_hyper = torch.zeros(64, dtype=torch.uint8, device=self.device)
        self._grad_views, self._m_views, self._v_views = {}, {}, {}
        self._param_objs = OrderedDict()
        off = 0
        for k in self._adapt_names:
            t = self._sd[k]
            n = t.numel()
            view = self._flat['param'][off:off + n].view(t.shape)
            view.copy_(t)
            p = torch.nn.Parameter(view, requires_grad=True)
            self._param_objs[k] = p
            self._sd[k] = p.data
            self._grad_views[k] = self._flat['grad'][off:off + n].view(t.shape)
            self._m_views[k] = self._flat['m'][off:off + n].view(t.shape)
            self._v_views[k] = self._flat['v'][off:off + n].view(t.shape)
            off += n
        for e in self._engines.values():
            e.close()
        self._engines = {}

    def _engine_for(self, image):
        if self.prepare_mode is None:
            raise RuntimeError('_prepare_head(mode) must be called before forward (src/tta_main.py:322)')
        key = (image.shape[0], image.shape[2], image.shape[3])
        self._last_key = key
        eng = self._engines.get(key)
        if eng is None:
            n, h, w = key          # H, W need not be multiples of 16: the engine pads and flip-ensembles (src/msg_chn_model_adapt.py:58-125)
            state = {k: (v.data if isinstance(v, torch.nn.Parameter) else v) for k, v in self._sd.items()}
            options = dict(self.engine_options)
            if self._trainable == 'head':
                options.update(trainable_head=1, skip_dec3=1)
            eng = MsgChnEngine(n, h, w, self.prepare_mode, state, self._grad_views, self._m_views, self._v_views,
                               options=options, adam_hyper=self._adam_hyper)
            if getattr(self, '_comm', None) is not None:      # shared-model mode (sharding.enable_shared_model): every engine joins it
                eng.set_comm(self._comm)
            self._engines[key] = eng
        return eng

    # -- reference API ----------------------------------------------------------------------------------
    def forward(self, image, sparse_depth, intrinsics=None, crop_mask=None, loss_type='pretrain'):
        if self.prepare_mode is None:
            raise RuntimeError('_prepare_head(mode) must be called before forward (src/tta_main.py:322)')
        image = image.contiguous()
        sparse_depth = sparse_depth.contiguous()
        if self.training and 'init_meta' in loss_type:           # stage 1 (network_exp_msg_chn_adapt.py:344-360)
            if self._trainable != 'meta':
                raise RuntimeError('stage-1 forward after prepare_parameters(\'head...\'): the trained set is the predictor head')
            out = _InitForwardFn.apply(self, image, sparse_depth, *self._param_objs.values())
            eng = self._engine_for(image)
            with torch.no_grad():                                  # the two coarser scales carry weight 0 in the loss (W:240-242): detached copies
                p11 = eng.tensor('real.p11').view(eng.n, 1, eng.h, eng.w).clone()
                o14 = eng.tensor('real.d1.out').view(eng.n, 1, eng.h // 4, eng.w // 4)
                o14 = torch.nn.functional.interpolate(o14, scale_factor=4, mode='bilinear', align_corners=True)
            return [out, p11, o14]
        if self.training and 'head' in loss_type and 'adapt' not in loss_type:      # stage 2 (:362-376)
            if self._trainable != 'head':
                raise RuntimeError('stage-2 forward needs prepare_parameters(\'head_selfsup_ema\') first (src/head_main.py:268)')
            if not all(s in loss_type for s in ('reverse', 'seq', 'ema')):
                raise NotImplementedError('stage-2 forward: only the [reverse, seq, ema] mode of the shipped scripts is implemented: %s' % loss_type)
            emb, ref = _HeadForwardFn.apply(self, image, sparse_depth, *self._param_objs.values())
            return None, emb, ref
        if self.training and 'adapt' in loss_type:
            if self._trainable != 'meta':
                raise RuntimeError('adaptation forward after prepare_parameters(\'head...\'): call adapt_parameters on a fresh model')
            out, emb, ref = _ForwardFn.apply(self, image, sparse_depth, *self._param_objs.values())
            return out, emb, ref
        eng = self._engine_for(image)
        eng.pack_adapted()
        with torch.no_grad():
            eng.forward(image, sparse_depth, None, False)
            return eng.tensor('output').view(eng.n, 1, eng.h, eng.w).clone()

    def parameters(self):
        return [torch.nn.Parameter(v, requires_grad=False) if k not in self._param_objs else self._param_objs[k]
                for k, v in self._sd.items() if k.endswith(_PARAM_SUFFIX)]

    def adapt_parameters(self, mode=''):
        if mode != 'meta':
            raise NotImplementedError('adapt mode %r: only "meta" is on the native path (msg_chn_model_adapt.py:392-396)' % mode)
        if self._trainable != 'meta':
            raise RuntimeError('adapt_parameters after prepare_parameters(\'head...\'): build a fresh model for adaptation')
        return torch.nn.ParameterList(list(self._param_objs.values()))

    def prepare_parameters(self, mode=''):
        """src/msg_chn_model_adapt.py:287-339 -- the tensors a preparation stage trains.  As in the reference, the call (re)creates
        the layers `mode` names from torch's global RNG: 'head_selfsup_ema' (src/head_main.py:268) draws new proj / proj_t / pred heads
        (twice, W:295-298) and returns proj.* and pred.*; 'meta_seq_<k>' (src/init_main.py:288) draws a new meta layer and returns it."""
        if 'head' in mode:
            if self.prepare_mode is None:
                raise RuntimeError('_prepare_head(mode) must be called before prepare_parameters(%r) (src/head_main.py:259)' % mode)
            fresh = {}
            add_head_state(fresh, mode)
            add_head_state(fresh, mode)
            self._sd.update(fresh)
            self._trainable = 'head'
            self._materialise()
            handed = [k for k in self._sd if k.startswith(('proj.', 'pred.')) and k.endswith(_PARAM_SUFFIX)]
            return [self._param_objs[k] if k in self._param_objs else torch.nn.Parameter(self._sd[k], requires_grad=True) for k in handed]
        if 'selfsup' in mode:
            raise NotImplementedError('prepare mode %r (joint meta + head training) is not used by the shipped scripts' % mode)
        if 'meta' in mode:
            self._trainable = 'meta'
            if self.prepare_mode is None or 'selfsup' not in self.prepare_mode:
                self.prepare_mode = mode
            add_head_state(self._sd, mode)
            self._materialise()
            return list(self._param_objs.values())
        raise NotImplementedError('prepare mode %r' % mode)

    def compute_loss(self, input_rgb=None, output_depth=None, validity_map=None, ground_truth=None, l1_weight=1.0, l2_weight=1.0,
                     loss_type='pretrain'):
        """src/msg_chn_model_adapt.py:203-264: masked L2 against the ground truth on output_depth[0] (evaluated by the engine on the
        prediction of its last stage-1 forward)"""
        out0 = output_depth[0] if isinstance(output_depth, (list, tuple)) else output_depth
        eng = self._engine_for(out0)
        loss = _L2LossFn.apply(eng, out0, ground_truth.contiguous(), float(self.max_predict_depth))
        return loss, {'loss': loss}

    def train(self):
        self.training = True

    def eval(self):
        self.training = False

    def state_dict(self):
        return OrderedDict((k, (v.detach() if isinstance(v, torch.Tensor) else v)) for k, v in self._sd.items())

    def load_state_dict(self, sd, strict=True):
        missing = [k for k in self._sd if k not in sd]
        unexpected = [k for k in sd if k not in self._sd]
        if strict and (missing or unexpected):
            raise RuntimeError('Error(s) in loading state_dict: missing %s, unexpected %s' % (missing[:5], unexpected[:5]))
        for k in self._sd:
            if k in sd:
                src = sd[k]
                if tuple(src.shape) != tuple(self._sd[k].shape):
                    raise RuntimeError('size mismatch for %s: %s vs %s' % (k, tuple(src.shape), tuple(self._sd[k].shape)))
                self._sd[k].copy_(src.to(self._sd[k].device, self._sd[k].dtype))
        for e in self._engines.values():
            e.rebind()

    # -- checkpoints: same files as the reference (src/msg_chn_model_adapt.py:482-545) ---------------------------------------
    _ADAM_STEP_WORD = 7        # AdamHyper.step: the int after seven floats (csrc/small_kernels.cuh)

    def adam_step_count(self):
        """number of optimiser steps the fused Adam has taken (device-resident counter shared by the engines of all shapes)"""
        return int(self._adam_hyper.view(torch.int32)[self._ADAM_STEP_WORD].item())

    def _optimizer_names(self):
        """state-dict keys of the tensors the reference hands to torch.optim.Adam in this stage, in its order"""
        if self._trainable == 'head':
            return [k for k in self._sd if k.startswith(('proj.', 'pred.')) and k.endswith(_PARAM_SUFFIX)]
        return list(self._adapt_names)

    def load_adam_state(self, opt_sd):
        """torch.optim.Adam state dict (as written by the reference's save_model) -> the fused Adam's flat moment buffers and step
        counter, so that `tta_step` continues the checkpointed run exactly as `optimizer.step()` would"""
        ids = [i for g in opt_sd['param_groups'] for i in g['params']]
        names = self._optimizer_names()
        if len(ids) != len(names):
            raise RuntimeError('optimizer state covers %d tensors, this stage hands %d to Adam' % (len(ids), len(names)))
        step = 0
        for i, k in zip(ids, names):
            if k not in self._m_views:          # stage 2: proj.* is handed to Adam but never receives a gradient (no state, never stepped)
                if opt_sd['state'].get(i) is not None:
                    raise RuntimeError('optimizer state holds moments for %s, which the native stage-2 step does not train' % k)
                continue
            st = opt_sd['state'].get(i)
            if st is None:                      # tensor never stepped
                self._m_views[k].zero_(); self._v_views[k].zero_()
                continue
            if tuple(st['exp_avg'].shape) != tuple(self._m_views[k].shape):
                raise RuntimeError('optimizer state %d has shape %s, adapted tensor %s has %s' % (
                    i, tuple(st['exp_avg'].shape), k, tuple(self._m_views[k].shape)))
            self._m_views[k].copy_(st['exp_avg'].to(self.device, torch.float32))
            self._v_views[k].copy_(st['exp_avg_sq'].to(self.device, torch.float32))
            step = max(step, int(st['step']))
        self._adam_hyper.view(torch.int32)[self._ADAM_STEP_WORD] = step

    def adam_state_dict(self, lr=0.0, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        """the fused Adam's state in torch.optim.Adam's own state_dict format (built by a real torch.optim.Adam, so every key the
        installed torch expects is there)"""
        # the parameter list the reference's optimiser was built over: the adapted tensors, or proj.* + pred.* for stage 2 (src/head_main.py:268)
        params = [self._param_objs[k] if k in self._param_objs else torch.nn.Parameter(self._sd[k], requires_grad=True)
                  for k in self._optimizer_names()]
        opt = torch.optim.Adam(params, lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
        step = self.adam_step_count()
        if step > 0:
            for k, p in self._param_objs.items():
                opt.state[p] = {'step': torch.tensor(float(step)), 'exp_avg': self._m_views[k].clone(), 'exp_avg_sq': self._v_views[k].clone()}
        return opt.state_dict()

    def restore_model(self, restore_path, optimizer=None):
        ckpt = torch.load(restore_path, map_location=self.device, weights_only=False)
        self.load_state_dict(ckpt['net'])
        if 'optimizer' in ckpt:
            if optimizer is not None:
                optimizer.load_state_dict(ckpt['optimizer'])
            if self._param_objs:
                self.load_adam_state(ckpt['optimizer'])      # the fused path (tta_step) continues from the same moments
        return optimizer, ckpt.get('train_step', 0)

    def save_model(self, checkpoint_path, step, optimizer, meanvar=None):
        """optimizer = the driver's torch.optim.Adam, or None when the fused `tta_step` path was used (its state is then written in
        torch.optim.Adam's format, so the reference -- or this class -- restores it into a torch optimiser)"""
        ckpt = {'net': OrderedDict((k, v.clone()) for k, v in self.state_dict().items()),
                'optimizer': optimizer.state_dict() if optimizer is not None else self.adam_state_dict(),
                'train_step': step}
        torch.save(ckpt, checkpoint_path)

    def convert_syncbn(self, apex=False):
        # single process per model: BatchNorm statistics are local (the reference's SyncBN is numerically plain BN at world size 1)
        return None

    def distributed_data_parallel(self, rank=0):
        return None

    def data_parallel(self):
        return None

    def to(self, device):
        self.device = torch.device(device)
        if self.prepare_mode is not None:
            self._materialise()


class ExternalModel_Adapt(object):
    """src/external_model_adapt.py:29-660, restricted to the TTA hot path (MSG-CHN and NLSPN back-ends; 'adapt' losses)."""

    def __init__(self, model_name, min_predict_depth, max_predict_depth, max_input_depth=None, offset=False, from_scratch=False,
                 dataset_name=None, device=torch.device('cuda')):
        self.model_name = model_name
        self.dataset_name = dataset_name
        self.device = torch.device(device)
        self.max_predict_depth = max_predict_depth
        self.max_input_depth = max_input_depth
        if model_name == 'msg_chn':
            self.model = MsgChnModel_Adapt(device=self.device, max_predict_depth=max_predict_depth)
        elif model_name == 'nlspn':
            from .nlspn_model_adapt import NLSPNModel_Adapt
            self.model = NLSPNModel_Adapt(device=self.device, max_depth=max_predict_depth, offset=offset, dataset_name=dataset_name,
                                          from_scratch=from_scratch)
        elif 'costdcnet' in model_name:
            raise NotImplementedError('%s has no native back-end (needs MinkowskiEngine; DESIGN.md, out of scope)' % model_name)
        else:
            raise ValueError('Unsupported depth completion model: {}'.format(model_name))

    def forward(self, image, sparse_depth, crop_mask=None, intrinsics=None, loss_type='pretrain'):
        if self.max_input_depth is not None:
            sparse_depth = torch.clamp(sparse_depth, 0, self.max_input_depth)     # src/external_model_adapt.py:103-108
        return self.model.forward(image=image, sparse_depth=sparse_depth, intrinsics=intrinsics, crop_mask=crop_mask,
                                  loss_type=loss_type)

    def compute_loss(self, input_rgb, output_depth=None, output_depth_ref=None, ground_truth=None, intrinsincs=None,
                     sparse_depth=None, reference_depth=None, validity_map=None, embedding=None, reference=None, epoch=0,
                     max_input_depth=None, max_predict_depth=100.0, w_loss_sparse_depth=0.0, w_loss_smoothness=0.0,
                     w_loss_robust=1.0, w_loss_cos=1.0, dataset_name=None, loss_type='pretrain'):
        if 'adapt' in loss_type and not any(s in loss_type for s in ('prepare', 'cotta', 'init', '_bn')):
            return self.adapt_loss(input_rgb=input_rgb, output_depth=output_depth, sparse_depth=sparse_depth,
                                   validity_map=validity_map, embedding=embedding, reference=reference,
                                   w_loss_sparse_depth=w_loss_sparse_depth, w_loss_smoothness=w_loss_smoothness,
                                   w_loss_cos=w_loss_cos)
        if 'prepare' in loss_type:                                  # src/external_model_adapt.py:155-158
            return self.prepare_loss(embedding=embedding, reference=reference)
        if self.model_name == 'msg_chn' and ('init' in loss_type or loss_type == 'pretrain') and ground_truth is not None:   # :174-180, :225-230
            if w_loss_smoothness != 0.0:
                raise NotImplementedError('supervised loss with a smoothness term (src/external_model_adapt.py:232-234)')
            return self.model.compute_loss(input_rgb=input_rgb, output_depth=output_depth, validity_map=validity_map,
                                           ground_truth=ground_truth, loss_type=loss_type)
        raise NotImplementedError('loss_type %r is outside the TTA hot path (DESIGN.md, scope table)' % loss_type)

    def prepare_loss(self, embedding, reference):
        """src/external_model_adapt.py:524-540 -- cosine distance between the stage-2 forward's emb and ref"""
        if self.model_name != 'msg_chn':
            raise NotImplementedError('stage-2 head training is implemented for msg_chn')
        eng = self.model._engines.get(getattr(self.model, '_last_key', None))
        if eng is None:
            raise RuntimeError('prepare_loss called before a stage-2 forward')
        loss = _CosLossFn.apply(eng, embedding, reference)
        return loss, {'loss': loss}

    def prepare_parameters(self, mode=''):
        return self.model.prepare_parameters(mode)

    def init_step(self, image_raw, sparse_depth, ground_truth, learning_rate, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, graph=False):
        """One whole stage-1 step (src/init_main.py:482-522: forward 'init_meta...', supervised loss, backward, Adam) in one library
        call; `last_losses()['loss']` reads the loss."""
        eng = self._prep_engine(image_raw, 'meta', (learning_rate, betas, eps, weight_decay))
        eng.init_step(image_raw, sparse_depth, ground_truth.contiguous(), self.max_input_depth, self.max_predict_depth,
                      self.model.img_scale, self.model.img_shift, graph=graph)
        self._last_engine = eng

    def head_step(self, image_raw, sparse_depth, learning_rate, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, graph=False):
        """One whole stage-2 step (src/head_main.py:437-480) in one library call."""
        if self.model_name == 'nlspn':                    # orchestrated from Python over the C ABI (nlspn_prepare.NlspnHeadTrainer)
            if getattr(self.model, 'img_scale', None) is None:
                raise RuntimeError('NLSPN head_step: call set_image_normalization(scale, shift) first (ImageNet statistics folded into the stem)')
            self._last_engine = self.model.head_step(image_raw.contiguous(), sparse_depth.contiguous(), learning_rate, betas, eps, weight_decay,
                                                     max_input_depth=self.max_input_depth, img_scale=self.model.img_scale,
                                                     img_shift=self.model.img_shift, graph=graph)
            return
        eng = self._prep_engine(image_raw, 'head', (learning_rate, betas, eps, weight_decay))
        eng.head_step(image_raw, sparse_depth, self.max_input_depth, self.model.img_scale, self.model.img_shift, graph=graph)
        self._last_engine = eng

    def _prep_engine(self, image_raw, trainable, hyper):
        if self.model_name != 'msg_chn':
            raise NotImplementedError('the source-domain preparation steps are implemented for msg_chn')
        if self.model._trainable != trainable:
            raise RuntimeError('call prepare_parameters(...) for the %s stage first' % trainable)
        eng = self.model._engine_for(image_raw)
        if getattr(eng, '_hyper', None) != hyper:
            eng.set_adam(hyper[0], hyper[1], hyper[2], hyper[3], step_count=-1)
            eng._hyper = hyper
        return eng

    def adapt_loss(self, input_rgb, output_depth, sparse_depth, validity_map, embedding, reference, w_loss_sparse_depth=1.0,
                   w_loss_smoothness=1.0, w_loss_cos=1.0):
        """src/external_model_adapt.py:371-441 (the clamp of :191-193 is applied inside the loss kernel)."""
        eng = self.model._engine_for(input_rgb)
        if self.model_name == 'nlspn':
            from .nlspn_model_adapt import _NlspnLossFn as loss_fn
        else:
            loss_fn = _LossFn
        loss, parts = loss_fn.apply(eng, output_depth, embedding, reference, input_rgb.contiguous(), sparse_depth.contiguous(),
                                    validity_map.contiguous(), self.max_input_depth, float(w_loss_sparse_depth),
                                    float(w_loss_smoothness), float(w_loss_cos))
        info = {'loss': loss.detach(), 'loss_sparse_depth': parts[0], 'loss_smooth': parts[1], 'loss_cos': parts[2]}
        return loss, info

    # -- the fused fast path (extension) ---------------------------------------------------------------------
    def set_image_normalization(self, scale, shift):
        """network input = raw_image * scale[c] + shift[c]  (src/transforms.py:669-712; (1/255, 0) for range [0,1])."""
        self.model.img_scale, self.model.img_shift = tuple(scale), tuple(shift)

    def tta_step(self, image_raw, sparse_depth, learning_rate, w_loss_sparse_depth=1.0, w_loss_smoothness=1.0, w_loss_cos=1.0,
                 betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, graph=False):
        """One whole adaptation step (src/tta_main.py:583-633) in a single library call; returns nothing -- read
        `last_losses()` when the values are needed (that read synchronises)."""
        eng = self.model._engine_for(image_raw)
        if self.model_name == 'nlspn':
            if getattr(self.model, 'img_scale', None) is None:
                # the network must see the NORMALISED image and the smoothness loss the raw one (src/tta_main.py:595-620): without the folded
                # normalisation the fused step would feed the raw image to both
                raise RuntimeError('NLSPN tta_step: call set_image_normalization(scale, shift) first (ImageNet statistics folded into the stem)')
            comm = getattr(self.model, '_comm', None)
            if comm is not None:             # shared-model mode: every rank must step on the same (N, H, W) (SyncBatchNorm count)
                from .sharding import check_same_shape
                check_same_shape(comm, (image_raw.shape[0], image_raw.shape[2], image_raw.shape[3]))
            eng.set_image_normalization(self.model.img_scale, self.model.img_shift)
            eng.tta_step(image_raw, image_raw, sparse_depth, learning_rate, w_loss_sparse_depth, w_loss_smoothness, w_loss_cos,
                         self.max_input_depth, graph=graph, betas=betas, eps=eps, weight_decay=weight_decay)
            self._last_engine = eng
            return
        hyper = (learning_rate, betas, eps, weight_decay)
        if getattr(eng, '_hyper', None) != hyper:
            eng.set_adam(learning_rate, betas, eps, weight_decay, step_count=-1)
            eng._hyper = hyper
        eng.tta_step(image_raw, sparse_depth, self.max_input_depth, w_loss_sparse_depth, w_loss_smoothness, w_loss_cos,
                     self.model.img_scale, self.model.img_shift, graph=graph)
        self._last_engine = eng

    def last_losses(self):
        if hasattr(self._last_engine, 'read_loss'):       # NLSPN stage-2 trainer: one scalar
            return {'loss': self._last_engine.read_loss()}
        return self._last_engine.read_losses()

    def last_losses_device(self):
        """device tensor (fp32 [5]: loss, loss_sparse_depth, loss_smooth, loss_cos, effective w_cos) of the last step: lets a driver
        copy it to pinned memory asynchronously and look at it one step later instead of stalling the stream every step"""
        e = self._last_engine
        if self.model_name == 'nlspn':
            return e.loss_ws[:20].view(torch.float32)
        return e.tensor('losses').view(-1)[:5]

    def last_output(self):
        e = self._last_engine
        if self.model_name == 'nlspn':
            return e.B['output']
        return e.tensor('output').view(e.n, 1, e.h, e.w)

    # -- plumbing identical to the reference ---------------------------------------------------------------------
    def parameters(self):
        return self.model.parameters()

    def _prepare_head(self, mode=''):
        self.model._prepare_head(mode=mode)

    def adapt_parameters(self, mode=''):
        return self.model.adapt_parameters(mode=mode)

    def train(self, meta=False, prepare=False):
        self.model.train()

    def eval(self):
        self.model.eval()

    def to(self, device):
        self.device = torch.device(device)
        self.model.to(device)

    def data_parallel(self):
        self.model.data_parallel()

    def distributed_data_parallel(self, rank):
        self.model.distributed_data_parallel(rank)

    def restore_model(self, restore_path, optimizer=None, learning_schedule=None, learning_rates=None, n_step_per_epoch=None):
        return self.model.restore_model(restore_path=restore_path, optimizer=optimizer)

    def save_model(self, checkpoint_path, step, optimizer, meanvar=None):
        self.model.save_model(checkpoint_path, step, optimizer, meanvar)

    def convert_syncbn(self, apex=False):
        self.model.convert_syncbn(apex)

    def state_dict(self):
        return self.model.state_dict()

    def load_state_dict(self, sd, strict=True):
        self.model.load_state_dict(sd, strict)
