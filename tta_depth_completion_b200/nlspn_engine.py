"""B200-native NLSPN ProxyTTA step (SURVEY.md section 8 row a18 on top of a19-a21): the graph of
external_src/NLSPN/src/model/nlspnmodel_adapt.py:850-944 (`_rgbd_meta_contrast`, mode [adapt, seq, reverse, ema]) with
`adapt_parameters('meta_bn')` semantics (src/nlspn_model_adapt.py:322-337: the 48->48 meta conv and every BatchNorm2d affine
pair are adapted, every BatchNorm2d uses batch statistics), the three TTA losses, the backward pass those 88 tensors need and
one fused Adam over them.  Host orchestration is Python (the reference's is); every operator is a CUDA kernel of
libptta_b200.so: tcgen05 implicit-GEMM convolutions (csrc/conv_gen.cuh), channel-generic BatchNorm / activation kernels
(csrc/nlspn_net.cuh), the propagation kernels (csrc/nlspn_prop.cuh), tcgen05 GEMMs for the heads.  No PyTorch compute on the
path (torch provides memory and streams) and no fallback.

Layout: feature maps NHWC bf16 with channel counts padded to multiples of 64; single-channel maps fp32 planar.
`fe1 = cat(conv1_rgb_meta(conv1_rgb(x)), conv1_dep(d))` is produced by ONE 64->64 convolution (identity centre tap for the 16
depth channels); `id_dec1 | gd_dec1 | cf_dec1` are one 128->192 convolution; `id_dec0 | gd_dec0 | cf_dec0` one 16-output
convolution with an fp32 planar epilogue.  Skip concatenations are never materialised (two TMA sources per convolution)."""
import ctypes

import torch

from . import _lib
from ._lib import check, ptr, c_void_p
from .convg import ConvG, FWD, DGRAD

RESNET34_LAYERS = (('conv2', 64, 64, 3, 1), ('conv3', 64, 128, 4, 2), ('conv4', 128, 256, 6, 2), ('conv5', 256, 512, 3, 2))
ACT_NONE, ACT_RELU, ACT_LEAKY = 0, 1, 2
BN_EPS = 1e-5


def _stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def adapt_parameter_names(sd, syncbn=True):
    """src/nlspn_model_adapt.py:322-337 ('meta_bn'): parameters whose name contains 'meta', then weight/bias of every BatchNorm2d /
    SyncBatchNorm in module order.  syncbn = True is the driver's sequence (src/tta_main.py:327-339: convert_syncbn() BEFORE
    adapt_parameters): SyncBatchNorm.convert_sync_batchnorm also converts the BatchNorm1d layers of the three heads, so their affine pairs
    are adapted too (94 tensors; the `'pred' not in np and 'proj' not in np` test of :335 sees the local names 'weight' / 'bias' and excludes
    nothing) and their running statistics are set to None.  syncbn = False: adapt_parameters without convert_syncbn (88 tensors)."""
    names = [k for k in sd if 'meta' in k and k.rsplit('.', 1)[-1] in ('weight', 'bias')]
    for k in sd:
        if k.endswith('.running_mean') and (syncbn or not k.startswith(('proj', 'pred'))):
            base = k[:-len('.running_mean')]
            names += [base + '.weight', base + '.bias']
    return names


class NlspnEngine:
    def __init__(self, state_dict, n, h, w, device, prop_time=18, legacy=True, share_from=None, syncbn=True):
        if h % 16 or w % 16:
            raise NotImplementedError('NLSPN engine: H and W must be multiples of 16 (got %dx%d)' % (h, w))
        _lib.lib()
        self.dev = torch.device(device)
        self.N, self.H, self.W = n, h, w
        self.prop_time, self.legacy = prop_time, legacy
        self.syncbn = syncbn if share_from is None else share_from.syncbn      # heads' BatchNorm1d adapted, no running statistics
        self.launches = 0
        self.B = {}            # named activation / gradient buffers
        if share_from is not None:
            # another input shape of the same model: parameters, packed operands and optimiser state are shared
            o = share_from
            self.sd, self.adapt_names, self.layout, self.params, self.grads = o.sd, o.adapt_names, o.layout, o.params, o.grads
            self.flat_p, self.flat_g, self.flat_m, self.flat_v = o.flat_p, o.flat_g, o.flat_m, o.flat_v
            self.fused_bn_w, self.fused_bn_b = o.fused_bn_w, o.fused_bn_b
            self.C, self.w_dec1, self.w_dec0, self.b_dec0, self.head_w = o.C, o.w_dec1, o.w_dec0, o.b_dec0, o.head_w
            self.bn_state = {}
            sd = self.sd
        else:
            sd = {k: v.detach().to(self.dev).contiguous() for k, v in state_dict.items()}
            self.sd = sd
            self._build_flat(sd)
            self._build_convs()
            self._build_heads()
        blocks = _lib.lib().ptta_nl_reduce_blocks(1 << 30, 64)
        self.partial = torch.empty(2 * 1024 * blocks, dtype=torch.float32, device=self.dev)
        self.partial_z = torch.empty_like(self.partial)      # reduction scratch of the zero-image branch (runs on its own stream)
        self.side_stream = torch.cuda.Stream(self.dev)
        self.two_streams = True
        # option: real + zero-image encoder passes as ONE batch-2N pass (per-half BatchNorm statistics; half the launches, twice the
        # tiles per conv launch).  Measured at 1x352x1216: 8.86 ms/step against 8.54 ms for the two-stream form, which also overlaps the
        # zero-image branch with the decoder and the propagation -- so it is off by default
        self.merge_branches = False
        self.coef = torch.empty(3 * 1024, dtype=torch.float32, device=self.dev)
        self.scratch_c = torch.empty(1024, dtype=torch.float32, device=self.dev)
        self.R = n * (h // 16) * (w // 16)
        self.loss_ws = torch.zeros(_lib.lib().ptta_tta_loss_workspace_bytes(n, h, w, self.R), dtype=torch.uint8, device=self.dev)
        self.wgrad_ws = torch.empty(_lib.lib().ptta_nl_wgrad48_workspace_bytes() // 4, dtype=torch.float32, device=self.dev)
        self.step_count = 0
        self.img_scale = self.img_shift = None
        self.aff_scale = float(sd['prop_layer.aff_scale_const'])
        self.adam_hyper = torch.tensor([0.0, 0.9, 0.999, 1e-8, 0.0], dtype=torch.float64, device=self.dev)
        self._adam_host = None
        self.adam_step_dev = share_from.adam_step_dev if share_from is not None else torch.zeros(1, dtype=torch.int32, device=self.dev)
        self._graph, self._graph_key, self._seen_key = None, None, None
        # shared-model mode (set_comm): exchanges of the running step body, in issue order
        self._comm, self._syncing, self._next_xid, self._exchange_at_world1 = None, False, 0, False
        if share_from is not None and share_from._comm is not None:
            self.set_comm(share_from._comm, share_from._exchange_at_world1)

    # ---- shared-model mode ----------------------------------------------------------------------------------------------------------
    def set_comm(self, comm, exchange_at_world1=False):
        """Join the peer communicator of the shared-model mode (sharding.PeerCommunicator; None: leave it).  With comm.world > 1 the
        TRAINING step takes every train-mode BatchNorm's statistics over all ranks (SyncBatchNorm: forward sums and backward sums
        exchanged inside the finalize kernels) and mean-all-reduces the flat gradient buffer inside the Adam kernel, so every rank applies
        the same update.  The eval forward keeps local statistics (SyncBatchNorm does not synchronise in eval mode).  The step then runs
        on ONE stream: the exchanging kernels spin until every rank has arrived, so all their blocks must be resident, and every rank
        must issue its exchanges in the same order.
        exchange_at_world1: a one-rank communicator runs the exchanging kernels too (otherwise world 1 is the plain step).  With one rank
        the rank-order sums are 0 + the local sums and the count is rows x 1, so the step computes what the plain step computes; this
        runs the rendezvous, the epoch advance and the slot parities on a single GPU."""
        self._exchange_at_world1 = bool(exchange_at_world1)
        if comm is not None and (comm.world > 1 or self._exchange_at_world1):
            if self.merge_branches:
                raise NotImplementedError('NLSPN shared-model mode: merge_branches (batch-2N encoder) has no SyncBatchNorm form')
            if comm.grad_floats < self.flat_g.numel():
                raise RuntimeError('NLSPN shared-model mode: the communicator holds %d gradient floats, the model has %d'
                                   % (comm.grad_floats, self.flat_g.numel()))
        self._comm = comm
        self._graph, self._graph_key, self._seen_key = None, None, None

    def _shared(self):
        return self._comm is not None and (self._comm.world > 1 or self._exchange_at_world1)

    def _take_xid(self):
        """exchange ids in issue order, reset at the start of every step body (the same sequence on every rank; a captured graph keeps
        them, the tags come from the device-side epoch)"""
        xid = self._next_xid
        if xid >= _lib.lib().ptta_comm_max_exchanges():
            raise RuntimeError('NLSPN shared-model mode: more than %d peer exchanges in one step' % _lib.lib().ptta_comm_max_exchanges())
        self._next_xid += 1
        return xid

    # ---- parameters -------------------------------------------------------------------------------------------------------------
    def _build_flat(self, sd):
        """Adapted tensors live in ONE flat fp32 buffer (+ gradient, Adam moments); the state-dict entries become views.  The
        three head-decoder BatchNorms are laid out back to back (+32 pad) so the fused 192-channel BatchNorm reads them in place,
        the meta bias is followed by 16 zeros (bias of the 64-channel fused stem convolution)."""
        names = adapt_parameter_names(sd, self.syncbn)
        self.adapt_names = names
        order, special = [], {}
        fused = ['id_dec1.1', 'gd_dec1.1', 'cf_dec1.1']
        for k in names:
            if any(k.startswith(f + '.') for f in fused) or k == 'conv1_rgb_meta.bias':
                continue
            order.append((k, sd[k].numel()))
        layout, off = {}, 0
        for k, n in order:
            layout[k] = off
            off += n
        layout['conv1_rgb_meta.bias'] = off
        off += 64
        self.fused_bn_w = off
        for f in fused:
            layout[f + '.weight'] = off
            off += sd[f + '.weight'].numel()
        off += 32
        self.fused_bn_b = off
        for f in fused:
            layout[f + '.bias'] = off
            off += sd[f + '.bias'].numel()
        off += 32
        self.flat_p = torch.zeros(off, dtype=torch.float32, device=self.dev)
        self.flat_p[self.fused_bn_w + 160:self.fused_bn_w + 192] = 1.0
        self.flat_g = torch.zeros_like(self.flat_p)
        self.flat_m = torch.zeros_like(self.flat_p)
        self.flat_v = torch.zeros_like(self.flat_p)
        self.layout = layout
        self.params, self.grads = {}, {}
        for k in names:
            o, cnt = layout[k], sd[k].numel()
            view = self.flat_p[o:o + cnt].view(sd[k].shape)
            view.copy_(sd[k])
            sd[k] = view
            self.params[k] = view
            self.grads[k] = self.flat_g[o:o + cnt].view(sd[k].shape)

    def _p(self, key, count=None):
        """flat-buffer slice of an adapted tensor (count > numel includes the zero / one padding behind it)"""
        o = self.layout[key]
        n = self.sd[key].numel() if count is None else count
        return self.flat_p[o:o + n], self.flat_g[o:o + n]

    def _build_convs(self):
        sd, C = self.sd, {}
        C['meta'] = ConvG('s1', FWD, sd['conv1_rgb_meta.weight'], 64, 64, ident_from=48)
        C['meta'].bias = self._p('conv1_rgb_meta.bias', 64)[0]
        for name, cin, cout, blocks, stride in RESNET34_LAYERS:
            for b in range(blocks):
                p = '%s.%d' % (name, b)
                ci = cin if b == 0 else cout
                ds = (p + '.downsample.0.weight') in sd
                kind = 's2' if (b == 0 and stride == 2) else 's1'
                C[p + '.conv1'] = ConvG(kind, FWD, sd[p + '.conv1.weight'], ci, cout)
                C[p + '.conv2'] = ConvG('s1', FWD, sd[p + '.conv2.weight'], cout, cout)
                C[p + '.conv2.d'] = ConvG('s1', DGRAD, sd[p + '.conv2.weight'], cout, cout)
                if ds:
                    C[p + '.down'] = ConvG('p1s2', FWD, sd[p + '.downsample.0.weight'], ci, cout)
                    C[p + '.conv1.d'] = ConvG('s2', DGRAD, sd[p + '.conv1.weight'], ci, cout, weight_short=sd[p + '.downsample.0.weight'])
                else:
                    C[p + '.conv1.d'] = ConvG(kind, DGRAD, sd[p + '.conv1.weight'], ci, cout)
        C['conv6'] = ConvG('s2', FWD, sd['conv6.0.weight'], 512, 512)
        C['conv6.d'] = ConvG('s2', DGRAD, sd['conv6.0.weight'], 512, 512)
        for name, cin, cout in (('dec5', (512, 0), 256), ('dec4', (256, 512), 128), ('dec3', (128, 256), 64), ('dec2', (64, 128), 64)):
            C[name] = ConvG('t2', FWD, sd[name + '.0.weight'], cin if cin[1] else cin[0], cout)
            C[name + '.d'] = ConvG('t2', DGRAD, sd[name + '.0.weight'], cin[0] + cin[1], cout)
        # id_dec1 | gd_dec1 | cf_dec1 (+ 32 zero channels): Conv2d(128, 192)
        w1 = torch.zeros((192, 128, 3, 3), dtype=torch.float32, device=self.dev)
        w1[0:64] = sd['id_dec1.0.weight']; w1[64:128] = sd['gd_dec1.0.weight']; w1[128:160] = sd['cf_dec1.0.weight']
        self.w_dec1 = w1
        C['dec1'] = ConvG('s1', FWD, w1, (64, 64), 192)
        C['dec1.d'] = ConvG('s1', DGRAD, w1, 128, 192)
        # id_dec0 | gd_dec0 | cf_dec0: Conv2d(192 + 64, 10) on (F, fe1); input channel blocks: id_fd1 0..63, gd_fd1 64..127,
        # cf_fd1 128..159, fe1 192..255
        w0 = torch.zeros((10, 256, 3, 3), dtype=torch.float32, device=self.dev)
        w0[0, 0:64] = sd['id_dec0.0.weight'][0, 0:64]; w0[0, 192:256] = sd['id_dec0.0.weight'][0, 64:128]
        w0[1:9, 64:128] = sd['gd_dec0.0.weight'][:, 0:64]; w0[1:9, 192:256] = sd['gd_dec0.0.weight'][:, 64:128]
        w0[9, 128:160] = sd['cf_dec0.0.weight'][0, 0:32]; w0[9, 192:256] = sd['cf_dec0.0.weight'][0, 32:96]
        self.w_dec0 = w0
        self.b_dec0 = torch.cat((sd['id_dec0.0.bias'], sd['gd_dec0.0.bias'], sd['cf_dec0.0.bias'], torch.zeros(6, device=self.dev))).contiguous()
        C['dec0'] = ConvG('s1', FWD, w0, (192, 64), 16)
        C['dec0.d'] = ConvG('s1', DGRAD, w0, 256, 64)
        self.C = C
        self.bn_state = {}

    def _build_heads(self):
        sd = self.sd
        self.head_w = {}
        for name in ('proj', 'proj_t', 'pred'):
            for i in ('0', '3'):
                wt = sd['%s.%s.weight' % (name, i)]
                self.head_w['%s.%s' % (name, i)] = wt.to(torch.bfloat16).contiguous()
                self.head_w['%s.%s.T' % (name, i)] = wt.t().contiguous().to(torch.bfloat16).contiguous()

    def repack_adapted(self):
        """after an Adam step: the bf16 operand copies of the adapted conv"""
        self.C['meta'].repack()

    # ---- small helpers --------------------------------------------------------------------------------------------------------
    def buf(self, name, shape, dtype=torch.bfloat16):
        t = self.B.get(name)
        if t is None or tuple(t.shape) != tuple(shape) or t.dtype != dtype:
            t = torch.empty(shape, dtype=dtype, device=self.dev)
            self.B[name] = t
        return t

    def conv(self, key, x0, x1=None, out_name=None, hw=None):
        op = self.C[key]
        n = x0.shape[0]
        if op.role == FWD:
            shape = op.out_shape(n, x0.shape[1], x0.shape[2])
        else:
            shape = op.out_shape(n, hw[0], hw[1])
        out = self.buf(out_name, shape)
        op(x0, x1, out=out, hw=hw)
        self.launches += 1
        return out

    def bn_stats(self, bn, x, gamma, beta, running=None):
        rows, c = x.numel() // x.shape[-1], x.shape[-1]
        if getattr(self, 'bn_running', False):
            # eval-mode BatchNorm2d (stage 2 of the preparation, src/nlspn_model_adapt.py:360-368): scale / shift from the running
            # statistics, computed once per layer -- the encoder is frozen there
            key = bn.split('.', 1)[1]
            st = self.bn_eval_state.get(key) if hasattr(self, 'bn_eval_state') else None
            if st is None:
                if not hasattr(self, 'bn_eval_state'):
                    self.bn_eval_state = {}
                scale = gamma / torch.sqrt(self.sd[key + '.running_var'] + BN_EPS)
                st = {'scale': scale.contiguous(), 'shift': (beta - self.sd[key + '.running_mean'] * scale).contiguous()}
                self.bn_eval_state[key] = st
            return st
        st = self.bn_state.get(bn)
        if st is None:
            st = {k: torch.empty(c, dtype=torch.float32, device=self.dev) for k in ('mean', 'rstd', 'scale', 'shift')}
            self.bn_state[bn] = st
        rm, rv, nbt = running if running is not None else (None, None, None)
        partial = self.partial_z if bn.startswith('z.') else self.partial
        if self._syncing:
            check(_lib.lib().ptta_nl_bn_stats_comm(ptr(x), c, rows, c, ptr(gamma), ptr(beta), BN_EPS, ptr(partial), ptr(st['mean']), ptr(st['rstd']),
                                                   ptr(st['scale']), ptr(st['shift']), ptr(rm), ptr(rv), ptr(nbt), 0.1, self._comm.handle,
                                                   self._take_xid(), _stream()), 'nl_bn_stats_comm')
        else:
            check(_lib.lib().ptta_nl_bn_stats(ptr(x), c, rows, c, ptr(gamma), ptr(beta), BN_EPS, ptr(partial), ptr(st['mean']), ptr(st['rstd']),
                                              ptr(st['scale']), ptr(st['shift']), ptr(rm), ptr(rv), ptr(nbt), 0.1, _stream()), 'nl_bn_stats')
        self.launches += 2
        return st

    def bn_act(self, x, st, act, out_name, res=None, res_st=None):
        rows, c = x.numel() // x.shape[-1], x.shape[-1]
        y = self.buf(out_name, x.shape)
        check(_lib.lib().ptta_nl_bn_act(ptr(x), ptr(st['scale']), ptr(st['shift']), ptr(res), c, ptr(res_st['scale']) if res_st else None,
                                        ptr(res_st['shift']) if res_st else None, ptr(y), rows, c, act, _stream()), 'nl_bn_act')
        self.launches += 1
        return y

    def bn_layer(self, prefix, bn_key, raw, act, res=None, res_st=None):
        """train-mode BatchNorm2d `bn_key` (+ residual) + activation on the raw conv output"""
        gamma, beta = self.sd[bn_key + '.weight'], self.sd[bn_key + '.bias']
        st = self.bn_stats(prefix + bn_key, raw, gamma, beta)
        return self.bn_act(raw, st, act, prefix + bn_key + '.act', res, res_st), st

    def bn_backward(self, prefix, bn_key, dy_a, ld_a, dy_b, ld_b, y, act, x, out_name, gskip_name=None, gamma=None, grads=True):
        """returns (dx wrt the raw conv output, gskip); writes d gamma / d beta into the flat gradient buffer"""
        rows, c = x.numel() // x.shape[-1], x.shape[-1]
        st = self.bn_state[prefix + bn_key]
        if gamma is None:
            gamma = self.sd[bn_key + '.weight']
        dg = db = None
        if grads:
            dg, db = self.grads[bn_key + '.weight'], self.grads[bn_key + '.bias']
        dx = self.buf(out_name, x.shape)
        gskip = self.buf(gskip_name, x.shape) if gskip_name else None
        self._bn_backward_call(dy_a, ld_a, dy_b, ld_b, y, act, x, st, gamma, dg, db, dx, gskip, rows, c)
        return dx, gskip

    def _bn_backward_call(self, dy_a, ld_a, dy_b, ld_b, y, act, x, st, gamma, dg, db, dx, gskip, rows, c):
        args = (ptr(dy_a), ld_a, ptr(dy_b), ld_b, ptr(y), act, ptr(x), ptr(st['mean']), ptr(st['rstd']), ptr(gamma), ptr(self.partial), ptr(dg), ptr(db),
                ptr(self.coef), ptr(dx), ptr(gskip), rows, c)
        if self._syncing:
            check(_lib.lib().ptta_nl_bn_backward_comm(*args, self._comm.handle, self._take_xid(), _stream()), 'nl_bn_backward_comm')
        else:
            check(_lib.lib().ptta_nl_bn_backward(*args, _stream()), 'nl_bn_backward')
        self.launches += 3

    # ---- forward ----------------------------------------------------------------------------------------------------------------
    def set_image_normalization(self, scale, shift):
        """network input = image * scale + shift per channel, applied inside the stem kernel (None: the caller passes the
        normalised image, as the reference's forward() expects)"""
        key = (None if scale is None else tuple(scale), None if shift is None else tuple(shift))
        if getattr(self, '_norm_key', ()) == key:
            return
        self._norm_key = key
        self.img_scale = None if scale is None else torch.tensor(scale, dtype=torch.float32, device=self.dev)
        self.img_shift = None if shift is None else torch.tensor(shift, dtype=torch.float32, device=self.dev)

    def encoder(self, pre, image, depth):
        """fe1 .. fe6 (nlspnmodel_adapt.py:866-880); `pre` prefixes the buffer names ('r.' real branch, 'z.' zero-image branch)"""
        sd, N, H, W = self.sd, self.N, self.H, self.W
        x1 = self.buf(pre + 'stem', (N, H, W, 64))
        check(_lib.lib().ptta_nl_stem(ptr(image), ptr(depth), ptr(sd['conv1_rgb.0.weight']), ptr(sd['conv1_rgb.0.bias']), ptr(sd['conv1_dep.0.weight']),
                                      ptr(sd['conv1_dep.0.bias']), ptr(self.img_scale), ptr(self.img_shift), ptr(x1), N, H, W, _stream()), 'nl_stem')
        self.launches += 1
        x = self.conv('meta', x1, out_name=pre + 'fe1')
        fe = [x]
        for name, cin, cout, blocks, stride in RESNET34_LAYERS:
            for b in range(blocks):
                p = '%s.%d' % (name, b)
                c1 = self.conv(p + '.conv1', x, out_name=pre + p + '.c1')
                a1, _ = self.bn_layer(pre, p + '.bn1', c1, ACT_RELU)
                c2 = self.conv(p + '.conv2', a1, out_name=pre + p + '.c2')
                if (p + '.down') in self.C:
                    cd = self.conv(p + '.down', x, out_name=pre + p + '.cd')
                    std = self.bn_stats(pre + p + '.downsample.1', cd, sd[p + '.downsample.1.weight'], sd[p + '.downsample.1.bias'])
                    x, _ = self.bn_layer(pre, p + '.bn2', c2, ACT_RELU, res=cd, res_st=std)
                else:
                    x, _ = self.bn_layer(pre, p + '.bn2', c2, ACT_RELU, res=x)
            fe.append(x)
        c6 = self.conv('conv6', x, out_name=pre + 'conv6.raw')
        fe6, _ = self.bn_layer(pre, 'conv6.1', c6, ACT_LEAKY)
        fe.append(fe6)
        return fe

    # ---- merged real | zero-image encoder -------------------------------------------------------------------------------------------
    def _bn_layer_grouped(self, key, raw, act, res=None, res_st=None):
        """train-mode BatchNorm of a merged batch: statistics per half (each half is its own forward pass in the reference)"""
        c = raw.shape[-1]
        rows_g = raw.numel() // c // 2
        st = self.bn_state.get('m.' + key)
        if st is None:
            st = {k: torch.empty(2 * c, dtype=torch.float32, device=self.dev) for k in ('mean', 'rstd', 'scale', 'shift')}
            self.bn_state['m.' + key] = st
            self.bn_state['r.' + key] = {k: v[:c] for k, v in st.items()}          # what the backward of the real half reads
        check(_lib.lib().ptta_nl_bn_stats_grouped(ptr(raw), c, rows_g, 2, c, ptr(self.sd[key + '.weight']), ptr(self.sd[key + '.bias']), BN_EPS,
                                                  ptr(self.partial), ptr(st['mean']), ptr(st['rstd']), ptr(st['scale']), ptr(st['shift']), _stream()),
              'nl_bn_stats_grouped')
        self.launches += 2
        if act is None:
            return None, st
        y = self.buf('m.' + key + '.act', raw.shape)
        check(_lib.lib().ptta_nl_bn_act_grouped(ptr(raw), ptr(st['scale']), ptr(st['shift']), ptr(res), c, ptr(res_st['scale']) if res_st else None,
                                                ptr(res_st['shift']) if res_st else None, ptr(y), rows_g, 2, c, act, _stream()), 'nl_bn_act_grouped')
        self.launches += 1
        return y, st

    def encoder_merged(self, image, depth):
        """both encoder passes of nlspnmodel_adapt.py:866-880 / 905-914 as one batch of 2N images (real first, zero-image second)"""
        sd, N, H, W = self.sd, self.N, self.H, self.W
        x1 = self.buf('m.stem', (2 * N, H, W, 64))
        check(_lib.lib().ptta_nl_stem_pair(ptr(image), ptr(depth), ptr(sd['conv1_rgb.0.weight']), ptr(sd['conv1_rgb.0.bias']),
                                           ptr(sd['conv1_dep.0.weight']), ptr(sd['conv1_dep.0.bias']), ptr(self.img_scale), ptr(self.img_shift), ptr(x1),
                                           N, H, W, _stream()), 'nl_stem_pair')
        self.launches += 1
        x = self.conv('meta', x1, out_name='m.fe1')
        fe = [x]
        for name, cin, cout, blocks, stride in RESNET34_LAYERS:
            for b in range(blocks):
                p = '%s.%d' % (name, b)
                c1 = self.conv(p + '.conv1', x, out_name='m.' + p + '.c1')
                a1, _ = self._bn_layer_grouped(p + '.bn1', c1, ACT_RELU)
                c2 = self.conv(p + '.conv2', a1, out_name='m.' + p + '.c2')
                if (p + '.down') in self.C:
                    cd = self.conv(p + '.down', x, out_name='m.' + p + '.cd')
                    _, std = self._bn_layer_grouped(p + '.downsample.1', cd, None)
                    x, _ = self._bn_layer_grouped(p + '.bn2', c2, ACT_RELU, res=cd, res_st=std)
                else:
                    x, _ = self._bn_layer_grouped(p + '.bn2', c2, ACT_RELU, res=x)
            fe.append(x)
        c6 = self.conv('conv6', x, out_name='m.conv6.raw')
        fe6, _ = self._bn_layer_grouped('conv6.1', c6, ACT_LEAKY)
        fe.append(fe6)
        # the backward pass and the decoder read the real half under the names of the unmerged path
        for k in [k for k in self.B if k.startswith('m.')]:
            self.B['r.' + k[2:]] = self.B[k][:N]
            self.B['z.' + k[2:]] = self.B[k][N:]
        return fe


    def _fused_dec1_params(self):
        w = self.flat_p[self.fused_bn_w:self.fused_bn_w + 192]
        b = self.flat_p[self.fused_bn_b:self.fused_bn_b + 192]
        return w, b

    def decoder(self, fe, depth):
        sd, N, H, W = self.sd, self.N, self.H, self.W
        fe1, fe2, fe3, fe4, fe5, fe6 = fe
        pre = 'r.'
        fd5, _ = self.bn_layer(pre, 'dec5.1', self.conv('dec5', fe6, out_name='r.dec5.raw'), ACT_LEAKY)
        fd4, _ = self.bn_layer(pre, 'dec4.1', self.conv('dec4', fd5, fe5, out_name='r.dec4.raw'), ACT_LEAKY)
        fd3, _ = self.bn_layer(pre, 'dec3.1', self.conv('dec3', fd4, fe4, out_name='r.dec3.raw'), ACT_LEAKY)
        fd2, _ = self.bn_layer(pre, 'dec2.1', self.conv('dec2', fd3, fe3, out_name='r.dec2.raw'), ACT_LEAKY)
        f_raw = self.conv('dec1', fd2, fe2, out_name='r.dec1.raw')
        gw, gb = self._fused_dec1_params()
        st = self.bn_stats('r.dec1', f_raw, gw, gb)
        F = self.bn_act(f_raw, st, ACT_LEAKY, 'r.dec1.act')
        # thin heads -> pred_init (LeakyReLU), guide (8), confidence (sigmoid)
        pred_init = self.buf('pred_init', (N, 1, H, W), torch.float32)
        guide = self.buf('guide', (N, 8, H, W), torch.float32)
        conf = self.buf('confidence', (N, 1, H, W), torch.float32)
        HW = H * W
        planes = (ctypes.c_void_p * 10)(pred_init.data_ptr(), *[guide.data_ptr() + 4 * k * HW for k in range(8)], conf.data_ptr())
        strides = (ctypes.c_longlong * 10)(HW, *([8 * HW] * 8), HW)
        acts = (ctypes.c_int * 10)(1, *([0] * 8), 2)
        op = self.C['dec0']
        check(_lib.lib().ptta_convg_run_thin(ptr(F), ptr(fe1), ptr(op.packed), ptr(self.b_dec0), planes, strides, acts, 10, N, H, W, 192, 64,
                                             _stream()), 'convg_run_thin')
        # prop_layer (nlspnmodel_adapt.py:340-373)
        oa = self.buf('offset_aff', (N, 24, H, W), torch.float32)
        check(_lib.lib().ptta_nl_conv8to24(ptr(guide), ptr(sd['prop_layer.conv_offset_aff.weight']), ptr(sd['prop_layer.conv_offset_aff.bias']),
                                           ptr(oa), N, H, W, 0, _stream()), 'nl_conv8to24')
        offset = self.buf('offset', (N, 18, H, W), torch.float32)
        aff = self.buf('aff', (N, 9, H, W), torch.float32)
        check(_lib.lib().ptta_nlspn_offset_affinity_forward(ptr(oa), ptr(conf), self.aff_scale, int(self.legacy), ptr(offset), ptr(aff), N, H, W,
                                                            _stream()), 'offset_affinity_forward')
        y = self.buf('y', (N, 1, H, W), torch.float32)
        saved = self.buf('prop_saved', (self.prop_time, N, H, W), torch.float32)
        check(_lib.lib().ptta_nlspn_propagate_forward(ptr(pred_init), ptr(offset), ptr(aff), ptr(depth), ptr(y), ptr(saved), None, N, H, W,
                                                      self.prop_time, _stream()), 'propagate_forward')
        out = self.buf('output', (N, 1, H, W), torch.float32)
        check(_lib.lib().ptta_nl_clamp0(ptr(y), ptr(out), y.numel(), _stream()), 'nl_clamp0')
        self.launches += 5 + self.prop_time
        return out

    def mlp(self, pre, name, x, train_running=True):
        """Linear -> BatchNorm1d (train: batch statistics + running-stat update) -> ReLU -> Linear  (nlspnmodel_adapt.py:1396-1402)"""
        sd = self.sd
        R = x.shape[0]
        h_raw = self.buf(pre + name + '.h_raw', (R, 1024))
        check(_lib.lib().ptta_gemm_bf16_tc(ptr(x), ptr(self.head_w[name + '.0']), ptr(h_raw), ptr(sd[name + '.0.bias']), R, 1024, x.shape[1],
                                           _stream()), 'gemm_tc')
        # after convert_syncbn + adapt_parameters('meta_bn') the heads' BatchNorm has running_mean = running_var = None: nothing to update
        running = (sd[name + '.1.running_mean'], sd[name + '.1.running_var'], sd[name + '.1.num_batches_tracked']) if (train_running and not self.syncbn) else None
        st = self.bn_stats(pre + name + '.1', h_raw, sd[name + '.1.weight'], sd[name + '.1.bias'], running)
        h_act = self.bn_act(h_raw, st, ACT_RELU, pre + name + '.h_act')
        out = self.buf(pre + name + '.out', (R, 1024))
        check(_lib.lib().ptta_gemm_bf16_tc(ptr(h_act), ptr(self.head_w[name + '.3']), ptr(out), ptr(sd[name + '.3.bias']), R, 1024, 1024, _stream()),
              'gemm_tc')
        self.launches += 2
        return out

    def forward(self, image, sparse_depth, training=True):
        """image: normalised fp32 NCHW; sparse_depth fp32 [N,1,H,W] (already clamped).  Returns (output, emb, ref) in training,
        output otherwise; all device tensors owned by the engine."""
        self._depth = sparse_depth
        if not training:
            fe = self.encoder('r.', image, sparse_depth)
            self.fe = fe
            return self.decoder(fe, sparse_depth)
        # the zero-image branch (nlspnmodel_adapt.py:905-914) and its heads depend only on the sparse depth and frozen / already
        # packed weights: they run on a second stream, concurrently with the real branch (fork / join through events, also inside a
        # CUDA-graph capture); their small layers fill the SMs the real branch's small layers leave idle
        main = torch.cuda.current_stream()
        # shared-model mode: one stream (the exchanging kernels of the two branches must not wait on each other across streams)
        side = self.side_stream if (self.two_streams and not self._syncing) else main
        if self._syncing and self.merge_branches:
            raise NotImplementedError('NLSPN shared-model mode: merge_branches (batch-2N encoder) has no SyncBatchNorm form')
        if self.merge_branches and image is not None:
            fe_m = self.encoder_merged(image, sparse_depth)
            fe = [t[:self.N] for t in fe_m]
            self.fe = fe
            z_zero = fe_m[-1][self.N:].reshape(self.R, 512)
            if side is not main:
                side.wait_stream(main)
            with torch.cuda.stream(side):                      # the heads of the zero rows run beside the decoder
                emb = self.mlp('z.', 'pred', self.mlp('z.', 'proj', z_zero))
            out = self.decoder(fe, sparse_depth)
            ref = self.mlp('r.', 'proj_t', fe[-1].reshape(self.R, 512))
            if side is not main:
                main.wait_stream(side)
            self.emb, self.ref = emb, ref
            return out, emb, ref
        if side is not main:
            side.wait_stream(main)
        with torch.cuda.stream(side):
            fe_z = self.encoder('z.', None, sparse_depth)
            emb = self.mlp('z.', 'pred', self.mlp('z.', 'proj', fe_z[-1].view(self.R, 512)))
        fe = self.encoder('r.', image, sparse_depth)
        self.fe = fe
        out = self.decoder(fe, sparse_depth)
        ref = self.mlp('r.', 'proj_t', fe[-1].view(self.R, 512))
        if side is not main:
            main.wait_stream(side)
        self.emb, self.ref = emb, ref
        return out, emb, ref

    # ---- losses -------------------------------------------------------------------------------------------------------------------
    def loss(self, image_raw, sparse, validity, cap, w_sd, w_sm, w_cos):
        self._loss_args = (image_raw, sparse, validity, float(cap if cap is not None else -1.0), float(w_sd), float(w_sm))
        check(_lib.lib().ptta_tta_loss_forward(ptr(self.B['output']), ptr(image_raw), ptr(sparse), ptr(validity), self._loss_args[3], ptr(self.emb),
                                               ptr(self.ref), self.R, 1024, w_sd, w_sm, w_cos, ptr(self.loss_ws), self.N, self.H, self.W, _stream()),
              'tta_loss_forward')
        self.launches += 3

    def read_losses(self):
        v = self.loss_ws[:20].view(torch.float32).cpu()
        return {'loss': float(v[0]), 'loss_sparse_depth': float(v[1]), 'loss_smooth': float(v[2]), 'loss_cos': float(v[3]), 'w_cos_eff': float(v[4])}

    # ---- backward -----------------------------------------------------------------------------------------------------------------
    def backward(self, gscale=1.0):
        self.loss_backward(gscale)
        self.network_backward()

    def loss_backward(self, gscale=1.0):
        """d loss / d output -> B['g.out'] (fp32 [N,1,H,W]) and d loss / d ref -> B['g.ref'] (bf16 [R,1024])"""
        L, N, H, W, B = _lib.lib(), self.N, self.H, self.W, self.B
        image_raw, sparse, validity, cap, w_sd, w_sm = self._loss_args
        g_out = self.buf('g.out', (N, 1, H, W), torch.float32)
        g_ref = self.buf('g.ref', (self.R, 1024))
        check(L.ptta_tta_loss_backward(ptr(B['output']), ptr(image_raw), ptr(sparse), ptr(validity), cap, ptr(self.emb), ptr(self.ref), self.R, 1024,
                                       w_sd, w_sm, ptr(self.loss_ws), gscale, ptr(g_out), ptr(g_ref), N, H, W, _stream()), 'tta_loss_backward')
        self.launches += 2
        if self.syncbn:          # emb = pred(proj(z_zero.detach())) reaches the adapted BatchNorm affine pairs of proj and pred
            g_emb = self.buf('g.emb', (self.R, 1024))
            check(L.ptta_tta_loss_backward_emb(ptr(self.emb), ptr(self.ref), self.R, 1024, ptr(self.loss_ws), gscale, ptr(g_emb), N, H, W, _stream()),
                  'tta_loss_backward_emb')
            self.launches += 1

    def network_backward(self):
        """from (B['g.out'], B['g.ref']) to the gradients of the 88 adapted tensors (flat_g)"""
        L, sd, N, H, W, B = _lib.lib(), self.sd, self.N, self.H, self.W, self.B
        fe1, fe2, fe3, fe4, fe5, fe6 = self.fe
        g_out = self.buf('g.out', (N, 1, H, W), torch.float32)
        g_ref = self.buf('g.ref', (self.R, 1024))
        g_y = self.buf('g.y', (N, 1, H, W), torch.float32)
        check(L.ptta_nl_mask_pos(ptr(g_out), ptr(B['y']), ptr(g_y), g_y.numel(), _stream()), 'nl_mask_pos')
        g_init = self.buf('g.pred_init', (N, 1, H, W), torch.float32)
        g_off = self.buf('g.offset', (N, 18, H, W), torch.float32)
        g_aff = self.buf('g.aff', (N, 9, H, W), torch.float32)
        scratch = self.buf('g.prop_scratch', (L.ptta_nlspn_backward_scratch_bytes(N, H, W) // 4,), torch.float32)
        check(L.ptta_nlspn_propagate_backward(ptr(g_y), ptr(B['offset']), ptr(B['aff']), ptr(self._depth), ptr(B['prop_saved']), ptr(g_init), ptr(g_off),
                                              ptr(g_aff), ptr(scratch), N, H, W, self.prop_time, _stream()), 'propagate_backward')
        g_oa = self.buf('g.offset_aff', (N, 24, H, W), torch.float32)
        g_conf = self.buf('g.conf', (N, 1, H, W), torch.float32)
        check(L.ptta_nlspn_offset_affinity_backward(ptr(B['offset_aff']), ptr(B['confidence']), self.aff_scale, int(self.legacy), ptr(g_off), ptr(g_aff),
                                                    ptr(g_oa), ptr(g_conf), N, H, W, _stream()), 'offset_affinity_backward')
        g_guide = self.buf('g.guide', (N, 8, H, W), torch.float32)
        check(L.ptta_nl_conv8to24(ptr(g_oa), ptr(sd['prop_layer.conv_offset_aff.weight']), None, ptr(g_guide), N, H, W, 1, _stream()), 'nl_conv8to24_t')
        T = self.buf('g.thin', (N, H, W, 64))
        check(L.ptta_nl_thin_grad_pack(ptr(g_init), ptr(B['pred_init']), ptr(g_guide), ptr(g_conf), ptr(B['confidence']), ptr(T), N, H, W, _stream()),
              'nl_thin_grad_pack')
        self.launches += 5 + self.prop_time
        # thin heads -> d(F | fe1)
        dcat1 = self.conv('dec0.d', T, out_name='g.cat1', hw=(H, W))                                   # [N,H,W,256]
        gw, _ = self._fused_dec1_params()
        dgw = self.flat_g[self.fused_bn_w:self.fused_bn_w + 192]
        dgb = self.flat_g[self.fused_bn_b:self.fused_bn_b + 192]
        st = self.bn_state['r.dec1']
        dF = self.buf('g.dec1.raw', (N, H, W, 192))
        rows = N * H * W
        self._bn_backward_call(dcat1, 256, None, 0, B['r.dec1.act'], ACT_LEAKY, B['r.dec1.raw'], st, gw, dgw, dgb, dF, None, rows, 192)
        dcat2 = self.conv('dec1.d', dF, out_name='g.cat2', hw=(H, W))                                  # [N,H,W,128] = d(fd2 | fe2)
        # decoder: dec2 .. dec5
        d2, _ = self.bn_backward('r.', 'dec2.1', dcat2, 128, None, 0, B['r.dec2.1.act'], ACT_LEAKY, B['r.dec2.raw'], 'g.dec2.raw')
        dcat3 = self.conv('dec2.d', d2, out_name='g.cat3', hw=(H // 2, W // 2))                       # [N,H/2,W/2,192] = d(fd3 | fe3)
        d3, _ = self.bn_backward('r.', 'dec3.1', dcat3, 192, None, 0, B['r.dec3.1.act'], ACT_LEAKY, B['r.dec3.raw'], 'g.dec3.raw')
        dcat4 = self.conv('dec3.d', d3, out_name='g.cat4', hw=(H // 4, W // 4))                       # [.,384] = d(fd4 | fe4)
        d4, _ = self.bn_backward('r.', 'dec4.1', dcat4, 384, None, 0, B['r.dec4.1.act'], ACT_LEAKY, B['r.dec4.raw'], 'g.dec4.raw')
        dcat5 = self.conv('dec4.d', d4, out_name='g.cat5', hw=(H // 8, W // 8))                       # [.,768] = d(fd5 | fe5)
        d5, _ = self.bn_backward('r.', 'dec5.1', dcat5, 768, None, 0, B['r.dec5.1.act'], ACT_LEAKY, B['r.dec5.raw'], 'g.dec5.raw')
        d_fe6_dec = self.conv('dec5.d', d5, out_name='g.fe6.dec', hw=(H // 16, W // 16))               # [.,512]
        # head: proj_t on the real rows (Linear, BatchNorm1d train, ReLU, Linear)
        R = self.R
        d_h = self.buf('g.proj_t.h', (R, 1024))
        check(L.ptta_gemm_bf16_tc(ptr(g_ref), ptr(self.head_w['proj_t.3.T']), ptr(d_h), None, R, 1024, 1024, _stream()), 'gemm_tc')
        d_hraw, _ = self.bn_backward('r.', 'proj_t.1', d_h, 1024, None, 0, B['r.proj_t.h_act'], ACT_RELU, B['r.proj_t.h_raw'], 'g.proj_t.h_raw',
                                     grads=self.syncbn)
        if self.syncbn:
            # emb = pred(proj(z_zero)), z_zero detached: gradients of pred.1 and proj.1 (weight, bias) only -- pred.3^T, BatchNorm backward,
            # pred.0^T, proj.3^T, BatchNorm backward; R = N H/16 W/16 rows of 1024, a few microseconds of GEMMs
            g_emb = B['g.emb']
            e_h = self.buf('g.pred.h', (R, 1024))
            check(L.ptta_gemm_bf16_tc(ptr(g_emb), ptr(self.head_w['pred.3.T']), ptr(e_h), None, R, 1024, 1024, _stream()), 'gemm_tc')
            e_hraw, _ = self.bn_backward('z.', 'pred.1', e_h, 1024, None, 0, B['z.pred.h_act'], ACT_RELU, B['z.pred.h_raw'], 'g.pred.h_raw')
            e_p = self.buf('g.proj.out', (R, 1024))
            check(L.ptta_gemm_bf16_tc(ptr(e_hraw), ptr(self.head_w['pred.0.T']), ptr(e_p), None, R, 1024, 1024, _stream()), 'gemm_tc')
            e_h1 = self.buf('g.proj.h', (R, 1024))
            check(L.ptta_gemm_bf16_tc(ptr(e_p), ptr(self.head_w['proj.3.T']), ptr(e_h1), None, R, 1024, 1024, _stream()), 'gemm_tc')
            self.bn_backward('z.', 'proj.1', e_h1, 1024, None, 0, B['z.proj.h_act'], ACT_RELU, B['z.proj.h_raw'], 'g.proj.h_raw')
            self.launches += 3
        d_fe6_head = self.buf('g.fe6.head', (R, 512))
        check(L.ptta_gemm_bf16_tc(ptr(d_hraw), ptr(self.head_w['proj_t.0.T']), ptr(d_fe6_head), None, R, 512, 1024, _stream()), 'gemm_tc')
        self.launches += 2
        # conv6
        d6, _ = self.bn_backward('r.', 'conv6.1', d_fe6_dec, 512, d_fe6_head, 512, fe6, ACT_LEAKY, B['r.conv6.raw'], 'g.conv6.raw')
        dy_a, ld_a = self.conv('conv6.d', d6, out_name='g.fe5.enc', hw=(H // 8, W // 8)), 512
        # encoder layers in reverse; the skip-concat slice of the decoder gradient joins at each layer output
        cat_slices = {'conv5': (dcat5, 256, 768), 'conv4': (dcat4, 128, 384), 'conv3': (dcat3, 64, 192), 'conv2': (dcat2, 64, 128)}
        sizes = {'conv2': (H, W), 'conv3': (H // 2, W // 2), 'conv4': (H // 4, W // 4), 'conv5': (H // 8, W // 8)}
        for name, cin, cout, blocks, stride in reversed(RESNET34_LAYERS):
            cat, coff, cld = cat_slices[name]
            dy_b, ld_b = cat.view(-1)[coff:], cld
            hh, ww = sizes[name]
            for b in reversed(range(blocks)):
                p = '%s.%d' % (name, b)
                out_act = B['r.' + p + '.bn2.act']
                has_down = (p + '.down') in self.C
                in_hw = (hh * 2, ww * 2) if (b == 0 and stride == 2) else (hh, ww)
                if has_down:
                    dc2, _ = self.bn_backward('r.', p + '.bn2', dy_a, ld_a, dy_b, ld_b, out_act, ACT_RELU, B['r.' + p + '.c2'], 'g.' + p + '.c2')
                    dcd, _ = self.bn_backward('r.', p + '.downsample.1', dy_a, ld_a, dy_b, ld_b, out_act, ACT_RELU, B['r.' + p + '.cd'], 'g.' + p + '.cd')
                    gskip = None
                else:
                    dc2, gskip = self.bn_backward('r.', p + '.bn2', dy_a, ld_a, dy_b, ld_b, out_act, ACT_RELU, B['r.' + p + '.c2'], 'g.' + p + '.c2',
                                                  gskip_name='g.' + p + '.skip')
                    dcd = None
                da1 = self.conv(p + '.conv2.d', dc2, out_name='g.' + p + '.a1', hw=(hh, ww))
                dc1, _ = self.bn_backward('r.', p + '.bn1', da1, cout, None, 0, B['r.' + p + '.bn1.act'], ACT_RELU, B['r.' + p + '.c1'], 'g.' + p + '.c1')
                dx = self.conv(p + '.conv1.d', dc1, dcd, out_name='g.' + p + '.x', hw=in_hw)
                dy_a, ld_a = dx, dx.shape[-1]
                dy_b, ld_b = (gskip, gskip.shape[-1]) if gskip is not None else (None, 0)
        # fe1 = meta conv output (no BN, no activation): three gradient sources
        d_fe1 = self.buf('g.fe1', (N, H, W, 64))
        check(L.ptta_nl_add3(ptr(dy_a), 64, ptr(dy_b), 64, c_void_p(dcat1.data_ptr() + 2 * 192), 256, ptr(d_fe1), rows, 64, _stream()), 'nl_add3')
        gw_meta = self.grads['conv1_rgb_meta.weight']
        check(L.ptta_nl_wgrad48(ptr(B['r.stem']), ptr(d_fe1), ptr(gw_meta), ptr(self.wgrad_ws), N, H, W, _stream()), 'nl_wgrad48')
        check(L.ptta_nl_col_sums(ptr(d_fe1), 64, rows, 64, ptr(self.partial), ptr(self.scratch_c), _stream()), 'nl_col_sums')
        self.grads['conv1_rgb_meta.bias'].copy_(self.scratch_c[:48])
        self.launches += 6

    # ---- optimiser + whole step ---------------------------------------------------------------------------------------------------
    def set_adam(self, lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        """hyper-parameters live on the device (the captured step reads them there); a change costs one small H2D copy"""
        host = (float(lr), float(betas[0]), float(betas[1]), float(eps), float(weight_decay))
        if host != self._adam_host:
            self.adam_hyper.copy_(torch.tensor(host, dtype=torch.float64))
            self._adam_host = host

    def adam_step(self):
        self.step_count += 1
        if self._syncing:
            # gradient mean all-reduce fused with the update; the averaged gradient is left in flat_g (DDP's .grad)
            check(_lib.lib().ptta_adam_flat_dev_comm(ptr(self.flat_p), ptr(self.flat_g), ptr(self.flat_m), ptr(self.flat_v), self.flat_p.numel(),
                                                     ptr(self.adam_hyper), ptr(self.adam_step_dev), self._comm.handle, self._take_xid(), _stream()),
                  'adam_flat_dev_comm')
        else:
            check(_lib.lib().ptta_adam_flat_dev(ptr(self.flat_p), ptr(self.flat_g), ptr(self.flat_m), ptr(self.flat_v), self.flat_p.numel(),
                                                ptr(self.adam_hyper), ptr(self.adam_step_dev), _stream()), 'adam_flat_dev')
        self.repack_adapted()
        self.launches += 3

    def tta_step(self, image_norm, image_raw, sparse_depth, lr, w_sd=1.0, w_sm=1.0, w_cos=0.1, cap=80.0, graph=False,
                 betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        """src/tta_main.py:583-633 for the NLSPN back-end: outlier removal, forward, losses, backward, Adam.
        image_norm: the image the network sees (normalised by the caller, or raw when set_image_normalization folds the
        normalisation into the stem), image_raw: the [0,255] image the smoothness loss sees.
        graph=True: the step is captured into a CUDA graph the second time it is called with the same input buffers and
        loss weights, and replayed from then on (the inputs are read from those buffers at every replay)."""
        self.set_adam(lr, betas, eps, weight_decay)
        if not graph:
            return self._step_body(image_norm, image_raw, sparse_depth, w_sd, w_sm, w_cos, cap)
        key = (image_norm.data_ptr(), image_raw.data_ptr(), sparse_depth.data_ptr(), float(w_sd), float(w_sm), float(w_cos), cap)
        if self._graph is not None and self._graph_key == key:
            self._graph.replay()
            self.step_count += 1
            return
        if self._seen_key != key:
            self._seen_key = key                               # first call: eager (allocates every buffer, sets kernel attributes)
            return self._step_body(image_norm, image_raw, sparse_depth, w_sd, w_sm, w_cos, cap)
        g = torch.cuda.CUDAGraph()
        l0 = self.launches
        torch.cuda.synchronize(self.dev)
        with torch.cuda.graph(g):
            self._step_body(image_norm, image_raw, sparse_depth, w_sd, w_sm, w_cos, cap)
        self.step_count -= 1                                   # capture does not execute
        self.launches_per_step = self.launches - l0
        self._graph, self._graph_key = g, key
        g.replay()
        self.step_count += 1

    def _step_body(self, image_norm, image_raw, sparse_depth, w_sd, w_sm, w_cos, cap):
        if not self._shared():
            return self._step_kernels(image_norm, image_raw, sparse_depth, w_sd, w_sm, w_cos, cap)
        self._syncing, self._next_xid = True, 0
        try:
            self._step_kernels(image_norm, image_raw, sparse_depth, w_sd, w_sm, w_cos, cap)
        finally:
            self._syncing = False
        check(_lib.lib().ptta_comm_advance(self._comm.handle, _stream()), 'comm_advance')       # the next step's exchanges use the next tag
        self.launches += 1
        self.exchanges_per_step = self._next_xid

    def _step_kernels(self, image_norm, image_raw, sparse_depth, w_sd, w_sm, w_cos, cap):
        N, H, W = self.N, self.H, self.W
        d_f = self.buf('filtered_depth', (N, 1, H, W), torch.float32)
        v_f = self.buf('filtered_validity', (N, 1, H, W), torch.float32)
        check(_lib.lib().ptta_outlier_removal(ptr(sparse_depth), ptr(d_f), ptr(v_f), N, H, W, 7, 1.5, _stream()), 'outlier_removal')
        d_c = self.buf('clamped_depth', (N, 1, H, W), torch.float32)
        hi = float(cap) if cap is not None else 3.0e38                # src/external_model_adapt.py:103-108
        check(_lib.lib().ptta_nl_clamp(ptr(d_f), ptr(d_c), 0.0, hi, d_f.numel(), _stream()), 'nl_clamp')
        self._depth = d_c
        self.forward(image_norm, d_c, training=True)
        self.loss(image_raw, d_f, v_f, cap, w_sd, w_sm, w_cos)
        self.backward()
        self.adam_step()
        self.launches += 2
