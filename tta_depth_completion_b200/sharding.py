"""Multi-GPU host logic for the TTA path (one process per GPU).

Default mode ("shards"): continual adaptation is a serial recurrence inside a sequence but sequences are independent,
so rank r adapts its own model copy on sequences r, r+W, r+2W, ... with NO data-path collective (the reference instead
runs shared-model DDP + SyncBN + one barrier per step: src/tta_main.py:101-111,354,804).

Optional mode ("shared"): every rank holds the same model and processes its own batch; the train-mode BatchNorm statistics are taken
over all ranks (SyncBatchNorm) and the adapted-parameter gradients (one flat fp32 buffer, 74 080 floats = 296 KB for MSG-CHN
`2layers`) are mean-all-reduced before the Adam step, so all replicas apply the identical update (the reference: SyncBN + DDP over all
1.53 M gradients, src/msg_chn_model_adapt.py:480,555-556).  Both exchanges are one-shot reads of NVLink peer memory inside the engine's own
kernels (csrc/peer_comm.cuh): the all-reduce is FUSED with the Adam update, the step stays one CUDA graph, no NCCL call on the path.
The NLSPN back-end has the same mode (its ~46 K-float flat gradient buffer, 125 exchanges per step; INTEGRATION.md section 2f)."""
import torch
import torch.distributed as dist


def shard_sequences(n_sequences, world_size, rank):
    """Sequence ids adapted by `rank` (strided like DistributedSampler, src/tta_main.py:17-21, without padding: a rank
    may get one sequence fewer)."""
    if not (0 <= rank < world_size):
        raise ValueError('rank %d outside world of %d' % (rank, world_size))
    return list(range(rank, n_sequences, world_size))


def shard_sizes(n_sequences, world_size):
    return [len(range(r, n_sequences, world_size)) for r in range(world_size)]


def allreduce_mean_(flat, group=None):
    """In-place mean all-reduce of one flat buffer (NCCL on CUDA tensors, gloo on CPU tensors)."""
    if not dist.is_available() or not dist.is_initialized() or dist.get_world_size(group) == 1:
        return flat
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    flat.div_(dist.get_world_size(group))
    return flat


class PeerCommunicator:
    """Peer-memory communicator of the shared-model mode (include/ptta_b200.h `ptta_comm_*`, csrc/peer_comm.cuh): one device block per
    rank, mapped into every peer of the node through CUDA IPC.  torch.distributed is used ONCE, to exchange the 64-byte IPC handles; the
    per-step exchanges (SyncBatchNorm sums, gradient all-reduce fused with Adam) then run inside the engine's kernels over NVLink."""

    def __init__(self, grad_floats, group=None, device=None):
        import ctypes
        from . import _lib
        from ._lib import check, c_void_p
        self.L = _lib.lib()
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.group, self.grad_floats = group, int(grad_floats)
        self.checked_shapes = set()          # input shapes all ranks were found to share (NLSPN: check_same_shape)
        if device is not None and torch.device(device).index is not None:
            torch.cuda.set_device(device)
        handle = c_void_p()
        check(self.L.ptta_comm_create(ctypes.byref(handle), self.rank, self.world, int(grad_floats)), 'comm_create')
        self.handle = handle
        nb = self.L.ptta_comm_handle_bytes()
        buf = ctypes.create_string_buffer(nb)
        check(self.L.ptta_comm_local_handle(self.handle, buf), 'comm_local_handle')
        if self.world > 1:
            handles = [None] * self.world
            dist.all_gather_object(handles, bytes(buf.raw), group=group)
            blob = ctypes.create_string_buffer(b''.join(handles), nb * self.world)
            check(self.L.ptta_comm_open_peers(self.handle, blob), 'comm_open_peers')
            dist.barrier(group)          # every rank has mapped every block before the first exchange

    def error(self):
        """0, or 1 + the id of the exchange that gave up waiting for a peer (the replicas are then out of step: stop)"""
        torch.cuda.synchronize()
        return int(self.L.ptta_comm_error(self.handle))

    def close(self):
        if getattr(self, 'handle', None):
            torch.cuda.synchronize()
            self.L.ptta_comm_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def enable_shared_model(model, group=None):
    """Switch a MSG-CHN or NLSPN `ExternalModel_Adapt` to the shared-model mode: every engine it creates from now on (and the ones it has)
    exchanges its train-mode BatchNorm sums and its adapted-parameter gradients with the other ranks through peer memory, so all ranks
    apply the identical update -- the reference's DDP + SyncBatchNorm semantics (src/msg_chn_model_adapt.py:480,555-556) without a
    collective call on the path.  Returns the communicator (keep it alive).

    NLSPN: convert_syncbn() must have been called (the reference driver always does, src/tta_main.py:327; without it the reference's
    BatchNorms would stay local).  The training step (shared_model_step, tta_step) then runs on one stream; the autograd path and the
    stage-2 head_step raise on a shared model."""
    if getattr(model, 'model_name', None) == 'nlspn':
        return _enable_shared_nlspn(model, group)
    wrapper = model.model
    comm = PeerCommunicator(wrapper._flat['grad'].numel(), group=group, device=wrapper.device)
    wrapper._comm = comm
    for eng in wrapper._engines.values():
        eng.set_comm(comm)
    return comm


def _enable_shared_nlspn(model, group):
    wrapper = model.model
    if not wrapper._syncbn:
        raise RuntimeError('NLSPN shared-model mode needs convert_syncbn() first: without it the reference\'s BatchNorms are local and '
                           'adapt_parameters(\'meta_bn\') hands a different tensor set to the optimiser')
    base = wrapper._materialise()
    comm = PeerCommunicator(base.flat_g.numel(), group=group, device=wrapper.device)
    wrapper._comm = comm
    for eng in wrapper._engines.values():
        eng.set_comm(comm)
    return comm


def check_same_shape(comm, shape):
    """Once per new input shape (called by the NLSPN tta_step of a shared model): every rank of the communicator must step on the same (N, H, W) -- the SyncBatchNorm count is local rows x
    world, and the ranks' exchange sequences must match.  One host all_gather_object; raises on a mismatch."""
    shape = tuple(int(v) for v in shape)
    if comm.world == 1 or shape in comm.checked_shapes:
        return
    shapes = [None] * comm.world
    dist.all_gather_object(shapes, shape, group=comm.group)
    if any(tuple(s) != shape for s in shapes):
        raise RuntimeError('shared-model mode: the ranks step on different input shapes %s (unequal per-rank batches are not supported)' % (shapes,))
    comm.checked_shapes.add(shape)


def shared_model_step(model, image_raw, sparse_depth, learning_rate, w_sd=1.0, w_sm=1.0, w_cos=0.1, group=None, graph=False):
    """One shared-model adaptation step.  With a peer communicator (enable_shared_model) this is the engine's ordinary fused step -- the
    exchanges happen inside its kernels and the step replays from a CUDA graph.  Without one (CPU tensors / gloo tests, or
    `PTTA_SHARED_NCCL=1`): local forward / loss / backward, mean all-reduce of the flat gradient buffer through torch.distributed,
    fused Adam -- local BatchNorm statistics, the round-1 form."""
    wrapper = model.model
    if getattr(model, 'model_name', None) == 'nlspn':
        # NLSPN: the engine's fused step with the exchanges inside its kernels (eager, or replayed from a CUDA graph)
        comm = getattr(wrapper, '_comm', None)
        if comm is None:
            raise RuntimeError('NLSPN shared_model_step: call sharding.enable_shared_model(model) first')
        model.tta_step(image_raw, sparse_depth, learning_rate, w_sd, w_sm, w_cos, graph=graph)
        return
    eng = wrapper._engine_for(image_raw)
    comm = getattr(wrapper, '_comm', None)
    if comm is not None:
        if getattr(eng, '_comm', None) is not comm:
            eng.set_comm(comm)
        model.tta_step(image_raw, sparse_depth, learning_rate, w_sd, w_sm, w_cos, graph=graph)
        return
    hyper = (learning_rate, (0.9, 0.999), 1e-8, 0.0)
    if getattr(eng, '_hyper', None) != hyper:
        eng.set_adam(learning_rate, step_count=-1)
        eng._hyper = hyper
    from . import ops
    d_f, v_f = ops.outlier_removal(sparse_depth.contiguous())
    eng.forward(image_raw, d_f, model.max_input_depth, True, wrapper.img_scale, wrapper.img_shift)
    eng.loss(image_raw, d_f, v_f, model.max_input_depth, w_sd, w_sm, w_cos)
    eng.backward(1.0)
    allreduce_mean_(wrapper._flat['grad'], group)
    eng.adam_step()
    model._last_engine = eng
