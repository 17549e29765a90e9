"""Host-side mirror of the reference's NLSPN wrapper (src/nlspn_model_adapt.py:30-486, class NLSPNModel_Adapt) on top of the
native engine (nlspn_engine.py): same method names, argument meaning and error types for the TTA hot path --

    model._prepare_head(mode) -> restore_model / load_state_dict -> adapt_parameters('meta_bn') -> torch.optim.Adam(params)
    per frame: forward(image, sparse_depth, loss_type='adapt_...') -> (output_depth, emb, ref); compute_loss(...) -> (loss, info);
               loss.backward(); optimizer.step()                                            (src/tta_main.py:309-354, 583-633)

`forward` returns tensors attached to a custom autograd.Function; `loss.backward()` runs the native backward and leaves `.grad` on
the 88 adapted nn.Parameters (views of the engine's flat buffer), so the driver's own three lines work unchanged.
Outside the hot path (DESIGN.md): adapt modes other than 'meta_bn', prepare modes other than '...meta...seq...1layer...ema',
the eval-time CPU hole filling (`inpainting`, src/nlspn_model_adapt.py:124-127, skimage) -- these raise NotImplementedError or
are skipped as documented.  No CPU / PyTorch fallback."""
import math
from collections import OrderedDict

import torch

from .nlspn_engine import NlspnEngine, adapt_parameter_names, RESNET34_LAYERS


def build_nlspn_state(prepare_mode, seed=None):
    """Freshly initialised state with the key set and shapes of the reference's `NLSPNModel_Adapt.state_dict()` after
    `_prepare_head(prepare_mode)` (external_src/NLSPN/src/model/nlspnmodel_adapt.py:384-448, 1338-1374); values follow the
    reference's initialisers in distribution (Kaiming-normal convs, unit BatchNorm, U(+-1/sqrt(fan_in)) Linear layers), the real
    values come from `restore_model`."""
    if not ('meta' in prepare_mode and 'seq' in prepare_mode and '1layer' in prepare_mode and 'selfsup' in prepare_mode and 'ema' in prepare_mode):
        raise NotImplementedError('NLSPN native back-end: prepare_mode %r (only meta_selfsup_seq_1layer_ema is on the TTA hot path)' % prepare_mode)
    g = torch.Generator()
    g.manual_seed(0 if seed is None else seed)
    sd = OrderedDict()

    def conv(name, cout, cin, k=3, bias=False, transposed=False):
        shape = (cin, cout, k, k) if transposed else (cout, cin, k, k)
        sd[name + '.weight'] = torch.randn(shape, generator=g) * math.sqrt(2.0 / (cout * k * k))
        if bias:
            sd[name + '.bias'] = torch.zeros(cout)

    def bn(name, c):
        sd[name + '.weight'] = torch.ones(c)
        sd[name + '.bias'] = torch.zeros(c)
        sd[name + '.running_mean'] = torch.zeros(c)
        sd[name + '.running_var'] = torch.ones(c)
        sd[name + '.num_batches_tracked'] = torch.tensor(0, dtype=torch.long)

    def linear(name, cout, cin):
        b = 1.0 / math.sqrt(cin)
        sd[name + '.weight'] = (torch.rand((cout, cin), generator=g) * 2 - 1) * b
        sd[name + '.bias'] = (torch.rand((cout,), generator=g) * 2 - 1) * b

    def mlp(name, dim, out, hidden):
        linear(name + '.0', hidden, dim)
        bn(name + '.1', hidden)
        linear(name + '.3', out, hidden)

    conv('conv1_rgb.0', 48, 3, bias=True)
    conv('conv1_dep.0', 16, 1, bias=True)
    for name, cin, cout, blocks, stride in RESNET34_LAYERS:
        for b in range(blocks):
            p = '%s.%d' % (name, b)
            conv(p + '.conv1', cout, cin if b == 0 else cout)
            bn(p + '.bn1', cout)
            conv(p + '.conv2', cout, cout)
            bn(p + '.bn2', cout)
            if b == 0 and stride != 1:
                conv(p + '.downsample.0', cout, cin, k=1)
                bn(p + '.downsample.1', cout)
    conv('conv6.0', 512, 512)
    bn('conv6.1', 512)
    for name, cin, cout in (('dec5', 512, 256), ('dec4', 768, 128), ('dec3', 384, 64), ('dec2', 192, 64)):
        conv(name + '.0', cout, cin, transposed=True)
        bn(name + '.1', cout)
    for br, c1, c0_in, c0_out in (('id', 64, 128, 1), ('gd', 64, 128, 8), ('cf', 32, 96, 1)):
        conv(br + '_dec1.0', c1, 128)
        bn(br + '_dec1.1', c1)
        conv(br + '_dec0.0', c0_out, c0_in, bias=True)
    sd['prop_layer.aff_scale_const'] = torch.full((1,), 0.5 * 8)
    sd['prop_layer.w'] = torch.ones((1, 1, 3, 3))
    sd['prop_layer.b'] = torch.zeros(1)
    sd['prop_layer.w_conf'] = torch.ones((1, 1, 1, 1))
    sd['prop_layer.conv_offset_aff.weight'] = torch.zeros((24, 8, 3, 3))          # nlspnmodel_adapt.py:223-224
    sd['prop_layer.conv_offset_aff.bias'] = torch.zeros(24)
    mlp('proj', 512, 1024, 1024)
    for k in [k for k in sd if k.startswith('proj.')]:
        sd['proj_t.' + k[5:]] = sd[k].clone()
    mlp('pred', 1024, 1024, 1024)
    conv('conv1_rgb_meta', 48, 48, bias=True)
    return sd


class _NlspnForwardFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, wrapper, image, sparse_depth, *params):
        eng = wrapper._engine_for(image)
        eng.repack_adapted()                     # the optimizer may have stepped the fp32 masters since the last call
        out, emb, ref = eng.forward(image, sparse_depth, training=True)
        ctx.wrapper, ctx.eng = wrapper, eng
        emb_v, ref_v = emb.view(-1, 1024), ref.view(-1, 1024)
        if not eng.syncbn:
            ctx.mark_non_differentiable(emb_v)   # emb = pred(proj(fe6_zero.detach())): without convert_syncbn no adapted tensor is on its path
        return out.clone(), emb_v, ref_v

    @staticmethod
    def backward(ctx, g_out, g_emb, g_ref):
        eng, wrapper = ctx.eng, ctx.wrapper
        go = eng.buf('g.out', (eng.N, 1, eng.H, eng.W), torch.float32)
        gr = eng.buf('g.ref', (eng.R, 1024))
        if g_out is not None and g_out.data_ptr() != go.data_ptr():
            go.view(-1).copy_(g_out.reshape(-1))
        if g_ref is not None and g_ref.data_ptr() != gr.data_ptr():
            gr.view(-1).copy_(g_ref.reshape(-1))
        if eng.syncbn:
            ge = eng.buf('g.emb', (eng.R, 1024))
            if g_emb is None:
                ge.zero_()
            elif g_emb.data_ptr() != ge.data_ptr():
                ge.view(-1).copy_(g_emb.reshape(-1))
        eng.network_backward()
        return (None, None, None) + tuple(eng.grads[k].clone() for k in wrapper._adapt_names)


class _NlspnLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, eng, output_depth, embedding, reference, image_raw, sparse_depth, validity_map, cap, w_sd, w_sm, w_cos):
        eng.loss(image_raw, sparse_depth, validity_map, cap, w_sd, w_sm, w_cos)
        ctx.eng = eng
        scal = eng.loss_ws[:16].view(torch.float32)
        loss, parts = scal[0].clone(), scal[1:4].clone()
        ctx.mark_non_differentiable(parts)
        return loss, parts

    @staticmethod
    def backward(ctx, g_loss, g_parts):
        eng = ctx.eng
        eng.loss_backward(float(g_loss))
        return (None, eng.B['g.out'], eng.B['g.emb'] if eng.syncbn else None, eng.B['g.ref'], None, None, None, None, None, None, None)


class NLSPNModel_Adapt(object):
    """src/nlspn_model_adapt.py:30-486 -- NLSPN wrapper (constructor arguments as in the reference)."""

    def __init__(self, device=torch.device('cuda'), max_depth=100.0, inpainting=False, use_pretrained=False, dataset_name=None,
                 from_scratch=False, offset=False):
        self.device = torch.device(device)
        self.max_depth = max_depth
        self.legacy = bool(offset)               # src/nlspn_model_adapt.py:62: args.legacy = offset
        self.prop_time = 18
        self.training = True
        self.warn_on_holes = True               # eval forward: one device->host read to report holes the reference would inpaint (False: skip the check)
        self.prepare_mode = None
        self.adapt = False
        self._sd = None
        self._engines = {}
        self._base = None
        self._adapt_names = []
        self._param_objs = OrderedDict()
        self._syncbn = False                     # set by convert_syncbn()
        self._comm = None                        # shared-model mode (sharding.enable_shared_model): every engine joins it

    # -- construction ---------------------------------------------------------------------------------------------------------------
    def _prepare_head(self, mode):
        self.prepare_mode = mode
        self._sd = build_nlspn_state(mode)
        self._reset_engines()

    def _reset_engines(self):
        if self.device.type != 'cuda':
            raise RuntimeError('the TTA step runs on CUDA only (no CPU fallback); got device %s' % self.device)
        self._engines, self._base = {}, None
        self._adapt_names = adapt_parameter_names(self._sd, self._syncbn)
        self._param_objs = OrderedDict()

    def _engine_for(self, image):
        if self.prepare_mode is None:
            raise RuntimeError('_prepare_head(mode) must be called before forward (src/tta_main.py:322)')
        key = (image.shape[0], image.shape[2], image.shape[3])
        eng = self._engines.get(key)
        if eng is None:
            n, h, w = key
            eng = NlspnEngine(self._sd, n, h, w, self.device, prop_time=self.prop_time, legacy=self.legacy, share_from=self._base,
                              syncbn=self._syncbn)
            if self._base is None:
                self._base = eng
                self._sd = eng.sd                      # device tensors; adapted entries are views of the engine's flat buffer
                self._param_objs = OrderedDict((k, torch.nn.Parameter(eng.params[k], requires_grad=True)) for k in self._adapt_names)
            self._engines[key] = eng
        if self._comm is not None and eng._comm is not self._comm:
            eng.set_comm(self._comm)
        return eng

    def _refuse_shared(self, what):
        if self._comm is not None:
            raise RuntimeError('NLSPN %s on a shared model (sharding.enable_shared_model): this path has no SyncBatchNorm / gradient '
                               'all-reduce form and would mix local and global semantics; use sharding.shared_model_step' % what)

    def _materialise(self, n=1, h=32, w=32):
        """parameters exist only once an engine does: create the smallest one if the driver asks for them before the first frame"""
        if self._base is None:
            self._engine_for(torch.empty((n, 3, h, w), device='meta'))
        return self._base

    # -- reference API ----------------------------------------------------------------------------------------------------------------
    def forward(self, image, sparse_depth, intrinsics=None, crop_mask=None, loss_type=None):
        if loss_type is None:
            raise TypeError("argument of type 'NoneType' is not iterable")      # the reference evaluates `'time' in loss_type`
        image, sparse_depth = image.contiguous(), sparse_depth.contiguous()
        if 'head' in loss_type or 'init_meta' in loss_type:
            # the preparation forwards (nlspnmodel_adapt.py:511-585) return embeddings / a supervised prediction, not this path's eval depth
            raise NotImplementedError('NLSPN native back-end: forward(loss_type=%r) -- stage 2 runs as the fused `head_step` '
                                      '(nlspn_prepare.NlspnHeadTrainer), stage 1 is not built' % (loss_type,))
        if self.training and 'adapt' in loss_type:
            self._refuse_shared('autograd adaptation forward')
            self._materialise(image.shape[0], image.shape[2], image.shape[3])
            return _NlspnForwardFn.apply(self, image, sparse_depth, *self._param_objs.values())
        eng = self._engine_for(image)
        eng.repack_adapted()
        with torch.no_grad():
            out = eng.forward(image, sparse_depth, training=False)
        # the reference fills holes (pixels that are exactly 0) with skimage's inpaint_biharmonic on the CPU here
        # (src/nlspn_model_adapt.py:124-127 -> src/data_utils.py:327-354) and returns the map untouched when there is none.  The solver is
        # not reproduced: a prediction without holes is identical to the reference's, one WITH holes is reported instead of passing silently
        out = out.clone()
        if self.warn_on_holes and 'head' not in loss_type:
            holes = int((out == 0).sum())
            if holes:
                import warnings
                warnings.warn('NLSPN eval forward: %d of %d predicted depths are exactly 0; the reference would fill them with '
                              'skimage.restoration.inpaint_biharmonic (src/data_utils.py:327-354), this path returns them as they are'
                              % (holes, out.numel()), RuntimeWarning)
        return out

    def parameters(self):
        self._materialise()
        return list(self._param_objs.values())

    def adapt_parameters(self, mode=None):
        """src/nlspn_model_adapt.py:287-340.  'meta_bn': the meta conv + every BatchNorm2d affine pair, batch statistics everywhere."""
        if mode != 'meta_bn':
            raise NotImplementedError('NLSPN native back-end: adapt mode %r (the TTA scripts use meta_bn, bash/adapt/adapt_nlspn_*.sh)' % (mode,))
        self._materialise()
        self.adapt = True
        return torch.nn.ParameterList(list(self._param_objs.values()))

    def prepare_parameters(self, mode=''):
        """src/nlspn_model_adapt.py:242-285.  'head...' (src/head_main.py:268 passes 'head_selfsup_ema'): proj / proj_t / pred are re-created
        from torch's global generator exactly as the reference's `_prepare_head(mode)` does, and the parameters of proj and pred are returned
        (proj_t is the EMA copy) in the reference, which hands them to torch.optim.Adam.  Here the whole step incl. Adam is the library call
        `head_step` (the trained tensors live in its flat buffer, created when the first frame fixes the input shape), so the returned list
        is empty; the trained tensors are read through `state_dict()` / `save_model`.  Other modes raise."""
        if 'head' not in mode:
            raise NotImplementedError('NLSPN native back-end: prepare_parameters(%r) (stage 2, "head...", is implemented)' % (mode,))
        if self._sd is None:
            raise RuntimeError('_prepare_head(mode) and restore_model(...) come first (src/head_main.py:259-266)')
        from .nlspn_prepare import fresh_head_state
        sd = OrderedDict((k, v.detach().clone().cpu()) for k, v in self.state_dict().items())
        sd.update(fresh_head_state())
        self._sd = sd
        self._reset_engines()
        self._trainable, self._head_trainer, self._head_key = 'head', None, None
        return []

    def _head_trainer_for(self, image):
        if getattr(self, '_trainable', None) != 'head':
            raise RuntimeError("call prepare_parameters('head_selfsup_ema') first")
        key = (image.shape[0], image.shape[2], image.shape[3])
        if self._head_trainer is None:
            from .nlspn_prepare import NlspnHeadTrainer
            n, h, w = key
            eng = NlspnEngine(self._sd, n, h, w, self.device, prop_time=self.prop_time, legacy=self.legacy, syncbn=False)
            self._base, self._engines[key], self._sd = eng, eng, eng.sd
            self._head_trainer, self._head_key = NlspnHeadTrainer(eng), key
        elif key != self._head_key:
            raise NotImplementedError('stage-2 training keeps one input shape (the reference crops every batch to n_height x n_width)')
        return self._head_trainer

    def head_step(self, image, sparse_depth, learning_rate, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, max_input_depth=None,
                  img_scale=None, img_shift=None, graph=False):
        """One whole stage-2 step (src/head_main.py:437-480) through the library; `image` is the network input unless a normalisation is folded
        into the stem (img_scale / img_shift)."""
        self._refuse_shared('head_step (stage 2)')
        tr = self._head_trainer_for(image)
        tr.eng.set_image_normalization(img_scale, img_shift)
        tr.head_step(image, sparse_depth, learning_rate, betas, eps, weight_decay, max_input_depth=max_input_depth, graph=graph)
        return tr

    def train(self):
        self.training = True

    def eval(self):
        self.training = False

    def to(self, device):
        device = torch.device(device)
        if device != self.device:
            self.device = device
            if self._sd is not None:
                self._sd = OrderedDict((k, v.detach().clone()) for k, v in self.state_dict().items())
                self._reset_engines()

    def data_parallel(self):
        pass

    def distributed_data_parallel(self, rank):
        pass                                      # one adapting model per GPU: nothing to wrap (DESIGN.md section 5)

    def convert_syncbn(self, apex=False):
        """src/nlspn_model_adapt.py:477-486.  One model per process, so the statistics stay local -- but the conversion also decides what
        adapt_parameters('meta_bn') returns afterwards: SyncBatchNorm.convert_sync_batchnorm turns the heads' BatchNorm1d layers into
        SyncBatchNorm instances as well, which :329-337 then matches (affine pairs adapted, running statistics None).  The reference
        driver always converts before it asks for the parameters (src/tta_main.py:327-339)."""
        if not self._syncbn:
            self._syncbn = True
            if self._sd is not None:
                sd = self.state_dict()
                self._sd = OrderedDict((k, v.detach().clone()) for k, v in sd.items())
                self._reset_engines()

    def state_dict(self):
        return OrderedDict((k, (v.data if isinstance(v, torch.nn.Parameter) else v)) for k, v in self._sd.items())

    def load_state_dict(self, sd, strict=True):
        if self._sd is None:
            raise RuntimeError('_prepare_head(mode) must be called before loading a checkpoint (src/tta_main.py:322-323)')
        missing = [k for k in self._sd if k not in sd]
        unexpected = [k for k in sd if k not in self._sd]
        if strict and (missing or unexpected):
            raise RuntimeError('Error(s) in loading state_dict: missing %s unexpected %s' % (missing[:4], unexpected[:4]))
        new = OrderedDict()
        for k, v in self._sd.items():
            src = sd.get(k, v)
            if tuple(src.shape) != tuple(v.shape):
                raise RuntimeError('size mismatch for %s: %s vs %s' % (k, tuple(src.shape), tuple(v.shape)))
            new[k] = src.detach().clone().to(v.dtype)
        self._sd = new
        self._reset_engines()

    def restore_model(self, restore_path, optimizer=None, learning_schedule=None, learning_rates=None, n_step_per_epoch=None):
        ckpt = torch.load(restore_path, map_location='cpu')
        self.load_state_dict(ckpt['net'] if 'net' in ckpt else ckpt)
        return optimizer

    def save_model(self, checkpoint_path, step, optimizer, meanvar=None):
        ckpt = {'net': OrderedDict((k, v.detach().cpu().clone()) for k, v in self.state_dict().items()), 'train_step': step}
        if optimizer is not None:
            ckpt['optimizer'] = optimizer.state_dict()
        torch.save(ckpt, checkpoint_path)
