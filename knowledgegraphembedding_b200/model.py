"""Drop-in `KGEModel` for the RotatE toolkit (reference: codes/model.py:22-429), B200-native.

Same constructor, parameters, state_dict keys, `forward(sample, mode)`, the five public score methods and
the static `train_step` / `test_step` that `codes/run.py` calls (run.py:227-235, 311, 341-363) -- but every
arithmetic step runs in the hand-written sm_100a kernels of libkge_b200.so (include/kge_b200.h).  PyTorch is
used for device memory, streams, `nn.Module` bookkeeping and NCCL only.  There is no CPU / eager fallback:
calling the scoring paths with parameters that are not on a B200 raises.
"""
import collections
import ctypes
import itertools
import logging
import os

import numpy as np
import torch
import torch.nn as nn

from . import _lib
from .filter_index import FilterIndex, relation_table

_MODELS = ('TransE', 'DistMult', 'ComplEx', 'RotatE', 'pRotatE')


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _on_device(t, dev, dtype, stage=None, st=None):
    """t as a contiguous `dtype` tensor on `dev` (no torch dispatch at all when it already is: the staged batches are).
    A host tensor of the right dtype goes through `stage(key_numel)` -> persistent device buffer + one cudaMemcpyAsync
    (kge_copy_h2d) instead of a framework copy with a fresh allocation (model.py:263-266)."""
    if t.device == dev and t.dtype == dtype and t.is_contiguous():
        return t
    if stage is not None and t.device.type == 'cpu' and t.dtype == dtype and t.is_contiguous() and t.numel():
        buf = stage(t.numel())
        _lib.call("kge_copy_h2d", ctypes.c_void_p(buf.data_ptr()), ctypes.c_void_p(t.data_ptr()),
                  t.numel() * t.element_size(), st if st is not None else _stream(dev))
        return buf.view(t.shape)
    return t.to(device=dev, dtype=dtype, non_blocking=True).contiguous()


def _is_integer(a):
    """An integer (not bool) numpy array or torch tensor."""
    if isinstance(a, torch.Tensor):
        return not a.dtype.is_floating_point and not a.dtype.is_complex and a.dtype != torch.bool
    return np.issubdtype(a.dtype, np.integer)


def _dist():
    """(rank, world_size) of the data-parallel group, (0, 1) when torch.distributed is not initialised."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_bounds(total, rank, world, align=1):
    """Contiguous balanced slice [begin, end) of `total` items for `rank` (batch rows / entity ids); with `align`
    the interior boundaries fall on multiples of it (entity tiles)."""
    total, align = int(total), int(align)
    units = (total + align - 1) // align
    base, rem = divmod(units, int(world))
    begin = rank * base + min(rank, rem)
    end = begin + base + (1 if rank < rem else 0)
    return min(begin * align, total), min(end * align, total)


# A train batch cut down to this rank's positive rows (multi-GPU): only the shard crosses PCIe.  `weight` stays whole
# (B floats) because the loss is normalised by the global sum of weights (model.py:285-286).
_RowShard = collections.namedtuple('_RowShard', 'positive negative weight mode total row_begin')


def _shard_rows(batch):
    if isinstance(batch, _RowShard):
        return batch
    positive_sample, negative_sample, subsampling_weight, mode = batch
    total = positive_sample.shape[0]
    rank, world = _dist()
    lo, hi = shard_bounds(total, rank, world)
    if world > 1:
        positive_sample, negative_sample = positive_sample[lo:hi], negative_sample[lo:hi]
    return _RowShard(positive_sample, negative_sample, subsampling_weight, mode, total, lo)


class _ScoreFunction(torch.autograd.Function):
    """forward(sample, mode) with autograd: the backward is kge_score_backward (model.py:301 through :86-146)."""

    @staticmethod
    def forward(ctx, model, entity, relation, modulus, positive, negative, mode):
        B = positive.shape[0]
        N = 1 if mode == 'single' else negative.shape[1]
        score = torch.empty((B, N), dtype=torch.float32, device=entity.device)
        desc = model._descriptor(entity, relation, modulus)
        err = model._err_flag()
        _lib.call("kge_score_forward", ctypes.byref(desc), _lib.MODE_IDS[mode], _ptr(positive), _ptr(negative),
                  B, N, _ptr(score), _ptr(err), _stream(entity.device))
        ctx.model, ctx.mode = model, mode
        ctx.save_for_backward(entity, relation, modulus if modulus is not None else entity.new_empty(0),
                              positive, negative if negative is not None else positive.new_empty(0))
        return score

    @staticmethod
    def backward(ctx, dscore):
        entity, relation, modulus, positive, negative = ctx.saved_tensors
        model, mode = ctx.model, ctx.mode
        modulus = modulus if modulus.numel() else None
        negative = negative if negative.numel() else None
        B = positive.shape[0]
        N = 1 if mode == 'single' else negative.shape[1]
        dscore = dscore.contiguous().float()
        gE, gR = torch.zeros_like(entity), torch.zeros_like(relation)
        gM = torch.zeros_like(modulus) if modulus is not None else None
        desc = model._descriptor(entity, relation, modulus)
        wbytes = _lib.load().kge_train_workspace_bytes(ctypes.byref(desc), B, N) if mode != 'single' else 0
        wsp = torch.empty(wbytes, dtype=torch.uint8, device=entity.device) if wbytes else None
        _lib.call("kge_score_backward", ctypes.byref(desc), _lib.MODE_IDS[mode], _ptr(positive), _ptr(negative),
                  B, N, _ptr(dscore), _ptr(gE), _ptr(gR), _ptr(gM), _ptr(wsp), wbytes, None, _stream(entity.device))
        return None, gE, gR, gM, None, None, None


class KGEModel(nn.Module):
    def __init__(self, model_name, nentity, nrelation, hidden_dim, gamma,
                 double_entity_embedding=False, double_relation_embedding=False):
        super(KGEModel, self).__init__()
        self.model_name = model_name
        self.nentity = nentity
        self.nrelation = nrelation
        self.hidden_dim = hidden_dim
        self.epsilon = 2.0

        # registration order = the reference's (model.py:32-60), so optimizer param order is [E, R, (modulus)]
        self.gamma = nn.Parameter(torch.Tensor([gamma]), requires_grad=False)
        self.embedding_range = nn.Parameter(
            torch.Tensor([(self.gamma.item() + self.epsilon) / hidden_dim]), requires_grad=False)

        self.entity_dim = hidden_dim * 2 if double_entity_embedding else hidden_dim
        self.relation_dim = hidden_dim * 2 if double_relation_embedding else hidden_dim

        rho = self.embedding_range.item()
        self.entity_embedding = nn.Parameter(torch.zeros(nentity, self.entity_dim))
        nn.init.uniform_(tensor=self.entity_embedding, a=-rho, b=rho)
        self.relation_embedding = nn.Parameter(torch.zeros(nrelation, self.relation_dim))
        nn.init.uniform_(tensor=self.relation_embedding, a=-rho, b=rho)
        if model_name == 'pRotatE':
            self.modulus = nn.Parameter(torch.Tensor([[0.5 * rho]]))

        if model_name not in _MODELS:
            raise ValueError('model %s not supported' % model_name)
        if model_name == 'RotatE' and (not double_entity_embedding or double_relation_embedding):
            raise ValueError('RotatE should use --double_entity_embedding')
        if model_name == 'ComplEx' and (not double_entity_embedding or not double_relation_embedding):
            raise ValueError('ComplEx should use --double_entity_embedding and --double_relation_embedding')

        self._ws = {}           # lazily allocated device workspaces (not part of state_dict)
        self._filter_cache = None

    # ------------------------------------------------------------------------------------------ plumbing
    def _device(self):
        dev = self.entity_embedding.device
        if dev.type != 'cuda':
            raise RuntimeError('KGEModel (B200-native) computes only on a CUDA device: call .cuda() first; '
                               'there is no CPU fallback')
        _lib.require_device(dev.index if dev.index is not None else torch.cuda.current_device())
        return dev

    def _scalars(self):
        """(gamma.item(), embedding_range.item()) without a device sync per call (the reference syncs in every
        score function, model.py:172,209,...); refreshed when the parameters are modified in place."""
        key = (self.gamma._version, self.embedding_range._version, self.gamma.data_ptr())
        if self._ws.get('scalars_key') != key:
            self._ws['scalars_key'] = key
            self._ws['scalars'] = (self.gamma.item(), self.embedding_range.item())
        return self._ws['scalars']

    def _own_descriptor(self):
        """_descriptor() of the model's own tables, rebuilt only when a table moved (train_step's launch path)."""
        E, R = self.entity_embedding, self.relation_embedding
        key = (E.data_ptr(), R.data_ptr(), self.gamma._version, self.embedding_range._version)
        held = self._ws.get('own_desc')
        if held is None or held[0] != key:
            held = self._ws['own_desc'] = (key, self._descriptor())
        return held[1]

    def _descriptor(self, entity=None, relation=None, modulus=None, name=None):
        entity = self.entity_embedding if entity is None else entity
        relation = self.relation_embedding if relation is None else relation
        if modulus is None and hasattr(self, 'modulus') and name is None:
            modulus = self.modulus
        for t in (entity, relation):
            if t.dtype != torch.float32 or not t.is_contiguous():
                raise ValueError('embedding tables must be contiguous float32')
        dev = entity.device
        return _lib.KgeModelStruct(
            model=_lib.MODEL_IDS[name or self.model_name],
            device=dev.index if dev.index is not None else torch.cuda.current_device(),
            nentity=entity.shape[0], nrelation=relation.shape[0],
            hidden_dim=entity.shape[1] // 2 if (name or self.model_name) in ('RotatE', 'ComplEx') else entity.shape[1],
            entity_dim=entity.shape[1], relation_dim=relation.shape[1],
            gamma=self._scalars()[0], embedding_range=self._scalars()[1],
            entity=entity.data_ptr(), relation=relation.data_ptr(),
            modulus=modulus.data_ptr() if modulus is not None else None)

    def _buffer(self, key, numel, dtype, device):
        buf = self._ws.get(key)
        if buf is None or buf.numel() < numel or buf.device != device or buf.dtype != dtype:
            buf = torch.empty(max(int(numel), 1), dtype=dtype, device=device)
            self._ws[key] = buf
            self._ws.pop('grad_views', None)
            self._ws.pop('grad_views_small', None)
        return buf

    def _err_flag(self):
        """int32 device flag set by the kernels on an out-of-range id; it is slot 4 of the 8-float loss buffer so
        that train_step reads losses and flag back in one copy."""
        dev = self.entity_embedding.device
        flag = self._ws.get('err')
        if flag is None or flag.device != dev:
            out = torch.zeros(8, dtype=torch.float32, device=dev)
            self._ws['loss_out'] = out
            flag = out.view(torch.int32)[4:5]
            self._ws['err'] = flag
        return flag

    def _raise_if_bad_index(self):
        flag = self._ws.get('err')
        if flag is not None and int(flag.item()) != 0:
            flag.zero_()
            raise IndexError('index out of range in sample (entity/relation id outside the embedding table)')

    def _apply(self, fn, *args, **kwargs):      # .cuda()/.to(): workspaces belong to the old device
        self._release_shard()
        self._ws = {}
        return super(KGEModel, self)._apply(fn, *args, **kwargs)

    # ------------------------------------------------------------------------------------------ scoring
    def forward(self, sample, mode='single'):
        '''
        Score a batch of triples (reference: model.py:72-164).
        'single': sample is a LongTensor [B,3] -> [B,1].
        'head-batch' / 'tail-batch': sample = (positive [B,3], negative entities [B,N]) -> [B,N].
        '''
        dev = self._device()
        if mode == 'single':
            positive, negative = sample, None
        elif mode in ('head-batch', 'tail-batch'):
            positive, negative = sample
            negative = negative.to(device=dev, dtype=torch.int64).contiguous()
            if negative.dim() != 2 or negative.shape[0] != positive.shape[0]:
                raise ValueError('negative sample must be [batch, negative_sample_size]')
        else:
            raise ValueError('mode %s not supported' % mode)
        positive = positive.to(device=dev, dtype=torch.int64).contiguous()
        if positive.dim() != 2 or positive.shape[1] != 3:
            raise ValueError('positive sample must be [batch, 3]')
        if self.model_name not in _MODELS:
            raise ValueError('model %s not supported' % self.model_name)
        modulus = self.modulus if self.model_name == 'pRotatE' else None
        return _ScoreFunction.apply(self, self.entity_embedding, self.relation_embedding, modulus,
                                    positive, negative, mode)

    def _score_rows(self, name, head, relation, tail, mode):
        """Public score-function signature of the reference (model.py:166-249): gathered rows
        head/relation/tail [B, 1|N, D] -> [B, N].  The rows are stacked into temporary tables and sent
        through the same kernels, so the arithmetic is identical to forward()."""
        dev = self._device()
        B = head.shape[0]
        hb = mode == 'head-batch'               # every other mode string takes the else-branch, as in the reference
        cand, fixed = (head, tail) if hb else (tail, head)
        if fixed.shape[1] != 1 or relation.shape[1] != 1:
            raise ValueError('only the candidate side may have more than one row per batch element')
        N = cand.shape[1]
        table = torch.cat([fixed.reshape(B, -1), cand.reshape(B * N, -1)], dim=0).float().contiguous()
        rel = relation.reshape(B, -1).float().contiguous()
        ar = torch.arange(B, device=dev, dtype=torch.int64)
        positive = torch.stack([ar, ar, ar], dim=1)          # row b of the temporary tables is the fixed side
        negative = (B + torch.arange(B * N, device=dev, dtype=torch.int64)).reshape(B, N)
        modulus = self.modulus if name == 'pRotatE' else None
        return _ScoreFunction.apply(_NamedView(self, name), table, rel, modulus, positive, negative,
                                    'head-batch' if hb else 'tail-batch')

    def TransE(self, head, relation, tail, mode):
        return self._score_rows('TransE', head, relation, tail, mode)

    def DistMult(self, head, relation, tail, mode):
        return self._score_rows('DistMult', head, relation, tail, mode)

    def ComplEx(self, head, relation, tail, mode):
        return self._score_rows('ComplEx', head, relation, tail, mode)

    def RotatE(self, head, relation, tail, mode):
        return self._score_rows('RotatE', head, relation, tail, mode)

    def pRotatE(self, head, relation, tail, mode):
        return self._score_rows('pRotatE', head, relation, tail, mode)

    # ------------------------------------------------------------------------------------------ training
    def _trainable(self):
        ps = [self.entity_embedding, self.relation_embedding]
        if self.model_name == 'pRotatE':
            ps.append(self.modulus)
        return ps

    def _peer_exchange(self, floats):
        """The NVLink peer-memory exchange of this model's gradient workspace (peer.py), or None: single process,
        KGE_NO_PEER=1, or peer memory could not be set up (then every rank falls back to the NCCL all-reduce)."""
        rank, world = _dist()
        if world == 1 or os.environ.get('KGE_NO_PEER'):
            return None
        peer = self._ws.get('peer')
        if peer is False:
            return None
        dev = self.entity_embedding.device
        if peer is not None and (peer.capacity < floats or peer.device != dev or peer.world != world):
            torch.cuda.synchronize(dev)
            peer.close()
            peer = None
            self._ws.pop('grad_views', None)
        if peer is None:
            from .peer import PeerExchange
            try:
                peer = PeerExchange(dev, floats + 8192)       # slack: a larger ragged batch does not re-map
            except _lib.KgeError as exc:
                logging.warning('NVLink peer exchange disabled, using NCCL all-reduce: %s' % exc)
                self._ws['peer'] = False
                return None
            self._ws['peer'] = peer
        return peer

    def _grad_workspace(self, B, entity_grad=True):
        """One flat fp32 buffer [dE | dR | dModulus(4) | pos_row[B] | neg_row[B]] so that the multi-GPU
        exchange covers it in one piece (peer-visible memory when the NVLink exchange is active), plus the small
        scalar buffers.  With entity_grad=False (the entity table's Adam update is fused into the backward,
        kge_train_rows_adam) the dE part does not exist."""
        dev = self.entity_embedding.device
        nE, nR = self.entity_embedding.numel(), self.relation_embedding.numel()
        nE4, nR4 = (nE + 3) // 4 * 4, (nR + 3) // 4 * 4
        if not entity_grad:
            nE = nE4 = 0
        total = nE4 + nR4 + 4 + 2 * B
        peer = self._peer_exchange(total) if entity_grad else None
        cached = self._ws.get('grad_views' if entity_grad else 'grad_views_small')
        if cached is not None and cached[0] == (B, dev, peer is not None):
            return dict(cached[1])
        if peer is not None:
            flat = peer.workspace[:total]
        else:
            flat = self._buffer('grad_flat' if entity_grad else 'grad_small', total, torch.float32, dev)[:total]
        views = {
            'flat': flat,
            'gE': flat[:nE].view_as(self.entity_embedding) if entity_grad else None,
            'gR': flat[nE4:nE4 + nR].view_as(self.relation_embedding),
            'gM': flat[nE4 + nR4:nE4 + nR4 + 1].view(1, 1),
            'pos_row': flat[nE4 + nR4 + 4:nE4 + nR4 + 4 + B],
            'neg_row': flat[nE4 + nR4 + 4 + B:total],
            'param_floats': nE4 + nR4 + 4,
            'rows_sum': self._buffer('rows_sum', 2 * B, torch.float32, dev)[:2 * B],
            'peer': peer,
            'wsum': self._buffer('wsum', 1, torch.float32, dev),
            'reg': self._buffer('reg_partials', 148 * 8, torch.float64, dev),
        }
        # slicing costs ~10 us per view: once per batch size
        self._ws['grad_views' if entity_grad else 'grad_views_small'] = ((B, dev, peer is not None), views)
        return dict(views)

    def _gather_moments(self, optimizer):
        """Peer-exchange steps keep exp_avg / exp_avg_sq current only on the rank that owns each slice; make them whole
        on every rank (collective: every rank calls it at the same point, e.g. run.py:106 optimizer.state_dict())."""
        sliced = getattr(optimizer, '_kge_sliced_moments', None)
        if not sliced:
            return
        from .peer import gather_moment_ranges
        params = self._trainable()
        pairs = [(optimizer.state[p]['exp_avg'], optimizer.state[p]['exp_avg_sq']) for p in params if len(optimizer.state[p])]
        gather_moment_ranges(pairs, list(sliced)[:len(pairs)])
        optimizer._kge_sliced_moments = None

    def _own_moments(self, optimizer, layout):
        """Record which rank keeps which element ranges of exp_avg / exp_avg_sq current (peer.moment_ranges /
        entity_ranges, one tuple per trainable parameter); a change of ownership gathers the moments first, and
        optimizer.state_dict() (run.py:106) gathers them through a pre-hook."""
        held = getattr(optimizer, '_kge_sliced_moments', None)
        if held is not None and held != layout:
            self._gather_moments(optimizer)
        if not getattr(optimizer, '_kge_hooked', False):
            optimizer.register_state_dict_pre_hook(lambda opt: self._gather_moments(opt))
            optimizer._kge_hooked = True
        optimizer._kge_sliced_moments = layout

    # ---- entity-sharded optimizer (multi-GPU; include/kge_b200.h `kge_train_rows_sharded`) ------------------------------
    def _release_shard(self):
        """Move the entity table out of the peer block of the entity-sharded step and unmap the block (device change,
        larger batch, end of life).  No exchange may be in flight: every step ends with a cross-GPU barrier."""
        held = self._ws.pop('shard', None)
        if held is None:
            return
        torch.cuda.synchronize(held['dev'])
        if self.entity_embedding.data_ptr() == held['e_view'].data_ptr():
            with torch.no_grad():
                self.entity_embedding.data = self.entity_embedding.data.clone()
        self._ws.pop('own_desc', None)
        held['peer'].close()

    def _shard_state(self, B, N, rank, world, dev):
        """Peer block of the entity-sharded step, [flags | dR dM row-losses | entity table | gather area], created on the
        first step (collective) and re-created when a larger batch arrives; the entity Parameter's storage is moved into
        it so that the owners of other entity ranges can store updated rows in place.  None: not available."""
        if os.environ.get('KGE_PEER_DENSE') or os.environ.get('KGE_NO_PEER') or os.environ.get('KGE_KEEP_GRADS') \
                or self._ws.get('peer') is False or self._ws.get('shard') is False:
            return None
        if self.nentity < world or self.entity_dim % 4:
            return None
        lib = _lib.load()
        rows_max = -(-int(B) // world)
        held = self._ws.get('shard')
        if held is not None and (held['rows_cap'] < rows_max or held['N'] != N or held['world'] != world or held['dev'] != dev):
            self._release_shard()
            held = None
        E, R = self.entity_embedding, self.relation_embedding
        if held is None:
            desc = self._own_descriptor()
            if not (lib.kge_train_plan(ctypes.byref(desc), rows_max, N) & _lib.PLAN_ENTITY_ADAM):
                return None
            from .peer import PeerExchange, _align256
            nR4 = (R.numel() + 3) // 4 * 4
            small = nR4 + 4 + 2 * rows_max * world + 64
            e_bytes = _align256(E.numel() * 4)
            g_bytes = int(lib.kge_train_gather_bytes(ctypes.byref(desc), world, rows_max, N))
            try:
                peer = PeerExchange(dev, small, extra_bytes=e_bytes + g_bytes)
            except _lib.KgeError as exc:
                logging.warning('entity-sharded optimizer disabled (no peer memory): %s' % exc)
                self._ws['shard'] = False
                return None
            wbytes = int(lib.kge_train_shard_workspace_bytes(ctypes.byref(desc), world, rows_max, N))
            held = self._ws['shard'] = {
                'peer': peer, 'rows_cap': rows_max, 'N': N, 'world': world, 'dev': dev,
                'gather_offset': peer.extra_offset + e_bytes,
                'e_view': peer.extra[:E.numel() * 4].view(torch.float32).view(E.shape),
                'wsp': torch.empty(wbytes, dtype=torch.uint8, device=dev), 'wbytes': wbytes, 'views': {},
                'reg_scratch': torch.zeros(148, dtype=torch.float64, device=dev),
            }
        if E.data_ptr() != held['e_view'].data_ptr():
            with torch.no_grad():
                held['e_view'].copy_(E.data)
                E.data = held['e_view']
            self._ws.pop('own_desc', None)
        return held

    def _train_step_sharded(self, held, optimizer, positive, negative, weight, B, rows, N, row_begin, mode_id, loss_kind,
                            alpha, reg, st):
        """One train step with the entity-sharded optimizer (see include/kge_b200.h): row kernel with mirrored outputs ->
        barrier -> owner's sort + entity-major backward + fused Adam with NVLink parameter stores; the relation table
        (and modulus) and the loss rows go through the small dense exchange on a second stream; barrier.  Returns the
        loss buffer.  Everything that does not change from step to step is cached per batch size, and the optimizer
        bookkeeping runs on the host while the row kernel is already in flight."""
        model = self
        dev = held['dev']
        peer = held['peer']
        world = peer.world
        E, R = model.entity_embedding, model.relation_embedding
        err = model._err_flag()
        desc = model._own_descriptor()
        params = model._trainable()
        ws = held['views'].get(B)
        if ws is None:
            from .peer import entity_ranges, moment_ranges
            nR = R.numel()
            nR4 = (nR + 3) // 4 * 4
            total = nR4 + 4 + 2 * B
            flat = peer.workspace[:total]
            rows_of = [hi - lo for lo, hi in (shard_bounds(B, r, world) for r in range(world))]
            has_mod = model.model_name == 'pRotatE'
            small = moment_ranges([0] + ([nR4] if has_mod else []), [p.numel() for p in params[1:]], [(0, (nR4 + 4) // 4)], world)
            ws = held['views'][B] = {
                'flat': flat, 'gR': flat[:nR].view_as(R), 'gM': flat[nR4:nR4 + 1].view(1, 1) if has_mod else None,
                'pos_row': flat[nR4 + 4:nR4 + 4 + B], 'neg_row': flat[nR4 + 4 + B:total], 'param_floats': nR4 + 4,
                'rows_sum': model._buffer('rows_sum', 2 * B, torch.float32, dev)[:2 * B],
                'wsum': model._buffer('wsum', 1, torch.float32, dev),
                'reg': model._buffer('reg_partials', 148 * 8, torch.float64, dev),
                'shard': peer.shard(held['gather_offset'], held['rows_cap'], rows_of),
                'layout': (entity_ranges(model.nentity, model.entity_dim, world),) + small,
            }
            ws['ptrs'] = {k: _ptr(ws[k]) for k in ('flat', 'gR', 'gM', 'wsum', 'reg')}
        out = model._ws['loss_out']
        events = model._ws.get('kernel_events')
        xevents = model._ws.get('exchange_events')
        pt = ws['ptrs']
        wsum_ptr = pt['wsum'] if weight is not None else None

        main = torch.cuda.current_stream(dev)
        side = model._ws.get('exchange_stream')          # id mirror next to the row kernel; relation-table exchange next
        if side is None:                                 # to the entity pass
            side = model._ws['exchange_stream'] = torch.cuda.Stream(dev)
        side_ptr = ctypes.c_void_p(side.cuda_stream)
        # ---- launches that need nothing from the optimizer: the row kernel is in flight before the host bookkeeping ----
        _lib.call("kge_zero", pt['flat'], ws['flat'].numel() * 4, st)
        if weight is not None:
            _lib.call("kge_weight_sum", _ptr(weight), B, pt['wsum'], st)
        if reg != 0.0:               # value of the L3 term from the replicated tables, before any owner updates them
            tensors = (_lib.KgeAdamTensor * 2)(_lib.KgeAdamTensor(E.data_ptr(), None, None, None, E.numel(), 1, 1),
                                               _lib.KgeAdamTensor(R.data_ptr(), None, None, None, R.numel(), 1, 1))
            _lib.call("kge_l3_partials", tensors, 2, pt['reg'], ws['reg'].numel(), st)
        if events is not None:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
        _lib.call("kge_train_rows_sharded", ctypes.byref(desc), mode_id, loss_kind, alpha, _ptr(positive), _ptr(negative),
                  _ptr(weight[row_begin:]) if weight is not None else None, wsum_ptr, B, rows, N,
                  _ptr(ws['neg_row'][row_begin:]), _ptr(ws['pos_row'][row_begin:]), pt['gR'], pt['gM'],
                  ctypes.byref(ws['shard']), _ptr(err), st, side_ptr)
        peer.barrier(2, err, st, exchange_err=True)      # every rank's rows are in every block; errors are shared

        # ---- torch.optim.Adam bookkeeping (host only; state created lazily exactly like torch/optim/adam.py) ----------
        model._own_moments(optimizer, ws['layout'])
        model._ws['exchange_regions'] = 1
        group = optimizer.param_groups[0]
        hyper = (float(group['lr']), float(group['betas'][0]), float(group['betas'][1]), float(group['eps']))
        grads = [None, ws['gR'], ws['gM']]
        entries = []
        for i, p in enumerate(params):
            state = optimizer.state[p]
            if len(state) == 0:
                state['step'] = torch.tensor(0.0, dtype=torch.float32)
                state['exp_avg'] = torch.zeros_like(p, memory_format=torch.preserve_format)
                state['exp_avg_sq'] = torch.zeros_like(p, memory_format=torch.preserve_format)
            state['step'] += 1
            g = grads[i]
            entries.append((p.data_ptr(), g.data_ptr() if g is not None else None, state['exp_avg'].data_ptr(),
                            state['exp_avg_sq'].data_ptr(), p.numel(), int(state['step'].item()),
                            1 if (reg != 0.0 and i < 2) else 0))

        # the relation table's (small, dense) exchange runs on a second stream under the owners' entity pass
        side.wait_stream(main)
        peer.reduce_adam(entries[1:], hyper, ws['param_floats'], (0, ws['param_floats'] // 4), ws['param_floats'], 2 * B,
                         ws['rows_sum'], err, side_ptr, l3=reg)
        e0 = entries[0]
        ea = _lib.KgeEntityAdam(exp_avg=e0[2], exp_avg_sq=e0[3], step=e0[5], lr=hyper[0], beta1=hyper[1], beta2=hyper[2],
                                eps=hyper[3], l3_coefficient=reg,
                                reg_partials=held['reg_scratch'].data_ptr() if reg != 0.0 else None, n_reg_partials=148)
        _lib.call("kge_train_entity_sharded", ctypes.byref(desc), mode_id, N, ctypes.byref(ws['shard']), _ptr(held['wsp']),
                  held['wbytes'], ctypes.byref(ea), _ptr(err), st)
        peer.barrier(3, err, st, phase=1)                # my parameter stores are issued (arrival only)
        if events is not None:
            ev1.record()
            events.append((ev0, ev1))
        if xevents is not None:
            xev0, xev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            xev0.record()
        main.wait_stream(side)
        _lib.call("kge_loss_finalize", _ptr(ws['rows_sum'][:B]), _ptr(ws['rows_sum'][B:]), _ptr(weight), wsum_ptr, B, reg,
                  pt['reg'] if reg != 0.0 else None, ws['reg'].numel() if reg != 0.0 else 0, _ptr(out), st)
        peer.barrier(3, err, st, phase=2)                # every owner's parameter rows have landed in every table
        if xevents is not None:
            xev1.record()
            xevents.append((xev0, xev1))
        for p in params:
            p.grad = None
        model._ws['update_cancelled_on_error'] = False
        return out

    @staticmethod
    def _fusable_adam(model, optimizer):
        if type(optimizer) is not torch.optim.Adam or len(optimizer.param_groups) != 1:
            return False
        g = optimizer.param_groups[0]
        if g.get('amsgrad') or g.get('maximize') or g.get('weight_decay', 0) != 0 or g.get('capturable') \
                or g.get('differentiable') or g.get('decoupled_weight_decay'):
            return False
        if isinstance(g['lr'], torch.Tensor) or any(isinstance(b, torch.Tensor) for b in g['betas']):
            return False
        want = model._trainable()
        have = [p for p in g['params'] if p.requires_grad]       # run.py:266 filters; tolerate unfiltered lists
        return len(have) == len(want) and all(a is b for a, b in zip(have, want))

    @staticmethod
    def train_step(model, optimizer, train_iterator, args):
        '''
        A single train step (reference: model.py:251-312): next batch -> negative scores ->
        self-adversarial / uniform loss -> positive scores -> weighted loss (+ L3) -> backward -> Adam.
        Returns the same log dict of python floats.
        '''
        if not model.training:
            model.train()
        if KGEModel._fusable_adam(model, optimizer):
            for p in model._trainable():          # optimizer.zero_grad(set_to_none=True) for exactly these parameters
                p.grad = None
        else:
            optimizer.zero_grad()
        # exactly one batch per call, pulled at the call (model.py:261).  (Round 1 pulled the batch of step i+1 ahead and
        # copied it on a side stream; with the staging copies of train_step_async that measured SLOWER -- 0.97 vs 0.75 ms
        # per step on B200 -- and changed the iterator contract, so it is gone.)
        out = model.train_step_async(optimizer, next(train_iterator), args)
        reg = float(getattr(args, 'regularization', 0.0))
        # the step's single device->host sync (model.py:305-310 has 3-4): 32 bytes into a pinned buffer
        host = model._ws.get('loss_host')
        if host is None:
            host = model._ws['loss_host'] = torch.empty(8, dtype=torch.float32).pin_memory()
        _lib.call("kge_copy_d2h_sync", ctypes.c_void_p(host.data_ptr()), ctypes.c_void_p(out.data_ptr()), 32,
                  _stream(out.device))
        code = int(host.view(torch.int32)[4])
        out = host.tolist()
        if code != 0:
            model._err_flag().zero_()
            if code == 2:
                raise _lib.KgeError('NVLink peer exchange timed out: a rank died or the ranks fell out of step')
            if model._ws.get('update_cancelled_on_error'):
                # the optimizer kernels saw the flag and left parameters and moments untouched (the reference raises
                # in index_select before backward): undo the host-side step counters too
                for p in model._trainable():
                    if len(optimizer.state[p]):
                        optimizer.state[p]['step'] -= 1
            raise IndexError('index out of range in sample (entity/relation id outside the embedding table)')
        regularization_log = {'regularization': out[3]} if reg != 0.0 else {}
        log = {
            **regularization_log,
            'positive_sample_loss': out[0],
            'negative_sample_loss': out[1],
            'loss': out[2]
        }
        return log

    def _exchange_slices(self, B, world, N):
        """How many regions the multi-GPU exchange of one step is cut into (KGE_PEER_SLICES, default 1 = no slicing).
        With n > 1 the exchange of a finished entity range runs on a second stream under the entity-major backward of
        the next range.  Measured on B200 (FB15k shapes): the exposed exchange shrinks (0.41 -> 0.27 ms at 8 GPUs, n=3)
        but the backward slows by as much (0.73 -> 0.88 ms: both kernels fight for L2 and issue slots), 1.22 vs 1.19 ms
        per step -- so it stays opt-in.  The answer must be the same on every rank, so it is derived from the global
        batch only: slicing needs the entity-major backward (csrc/kge_train.cu takes it when a rank's rows x N >=
        6 x nentity) on the rank with the fewest rows."""
        n = int(os.environ.get('KGE_PEER_SLICES', '1'))
        if n <= 1 or self.entity_dim % 4 or (B // world) * N < 6 * self.nentity or self.nentity < 4 * n:
            return 1
        return min(n, 8)

    def _train_plan(self, rows, N):
        """(workspace bytes, kge_train_plan bits) for `rows` local positive rows x N candidates, cached per shape."""
        desc = self._own_descriptor()
        wkey = (rows, N, desc.entity_dim, desc.nentity, desc.entity, desc.relation)
        held = self._ws.get('train_ws_bytes')
        if held is None or held[0] != wkey:
            lib = _lib.load()
            held = self._ws['train_ws_bytes'] = (wkey, lib.kge_train_workspace_bytes(ctypes.byref(desc), rows, N),
                                                 lib.kge_train_plan(ctypes.byref(desc), rows, N))
        return held[1], held[2]

    def train_step_async(self, optimizer, batch, args):
        """Everything train_step does on the device, without the final read-back: returns the device buffer
        [positive_sample_loss, negative_sample_loss, loss, regularization, err_flag(int32 bits), ...]."""
        model = self
        dev = model._device()
        st = _stream(dev)

        if batch[3] not in ('head-batch', 'tail-batch'):
            raise ValueError('mode %s not supported' % batch[3])
        # multi-GPU: this rank's positive rows only (the H2D copy and the kernels see rows [row_begin, row_end) of B)
        positive_sample, negative_sample, subsampling_weight, mode, B, row_begin = _shard_rows(batch)
        # host batches are staged into persistent device buffers; the host tensors stay referenced until the next step
        # (a pinned source must outlive its asynchronous copy)
        model._ws['staged_host_batch'] = (positive_sample, negative_sample, subsampling_weight)
        positive = _on_device(positive_sample, dev, torch.int64,
                              lambda n: model._buffer('stage_pos', n, torch.int64, dev)[:n], st)
        fused_adam = KGEModel._fusable_adam(model, optimizer)
        # Zero-copy negatives (KGE_ZERO_COPY=1, off by default): a pinned host batch is not copied when the single-read row
        # kernel will run -- it reads each candidate id exactly once, through windows prefetched 24 candidates (and a whole
        # row) ahead, and leaves the int32 copy that the counting sort needs on the device.  Measured on B200 (cfg 3):
        # 0.745 vs 0.728 ms per end-to-end step with the staging copy -- the strided 8-byte window loads become 262 k
        # separate PCIe reads, slower than one 2 MB DMA -- so the staging copy stays the default.
        negative = None
        if (os.environ.get('KGE_ZERO_COPY') == '1' and negative_sample.device.type == 'cpu'
                and negative_sample.dtype == torch.int64 and negative_sample.dim() == 2
                and negative_sample.numel() and negative_sample.is_contiguous() and negative_sample.is_pinned()):
            plan0 = model._train_plan(negative_sample.shape[0], negative_sample.shape[1])[1]
            if (plan0 & _lib.PLAN_SINGLE_READ) or ((plan0 & _lib.PLAN_ENTITY_ADAM) and fused_adam
                                                   and not os.environ.get('KGE_KEEP_GRADS')):
                negative = negative_sample           # host pointer == device pointer (unified addressing)
        if negative is None:
            negative = _on_device(negative_sample, dev, torch.int64,
                                  lambda n: model._buffer('stage_neg', n, torch.int64, dev)[:n], st)
        rows, N = negative.shape
        uni = bool(getattr(args, 'uni_weight', False))
        weight = None if uni else _on_device(subsampling_weight, dev, torch.float32,
                                             lambda n: model._buffer('stage_w', n, torch.float32, dev)[:n], st)
        reg = float(getattr(args, 'regularization', 0.0))
        adversarial = bool(args.negative_adversarial_sampling)
        alpha = float(args.adversarial_temperature) if adversarial else 1.0
        loss_kind = _lib.LOSS_NEG_ADVERSARIAL if adversarial else _lib.LOSS_NEG_UNIFORM
        mode_id = _lib.MODE_IDS[mode]

        err = model._err_flag()
        rank, world = _dist()
        if world > 1 and fused_adam:
            # multi-GPU default: entity-sharded optimizer (owner computes; no dense gradient, no exchange kernel)
            held = model._shard_state(B, N, rank, world, dev)
            if held is not None:
                return model._train_step_sharded(held, optimizer, positive, negative, weight, B, rows, N, row_begin,
                                                 mode_id, loss_kind, alpha, reg, st)
        desc = model._own_descriptor()
        # which kernels run for this shape (cached per shape): the single-read path can also apply the entity table's
        # Adam update inside the backward -- on one device, with a stock Adam, unless the caller wants p.grad
        wbytes, plan = model._train_plan(rows, N)
        fuse_entity = bool(fused_adam and world == 1 and rows == B and (plan & _lib.PLAN_ENTITY_ADAM)
                           and not os.environ.get('KGE_KEEP_GRADS'))
        ws = model._grad_workspace(B, entity_grad=not fuse_entity)
        ws['out'] = model._ws['loss_out']
        events = model._ws.get('kernel_events')       # bench.py: CUDA events around the dominant kernel
        xevents = model._ws.get('exchange_events')    # bench.py: CUDA events around the exposed exchange + optimizer
        params = model._trainable()
        grads = [ws['gE'], ws['gR']] + ([ws['gM']] if model.model_name == 'pRotatE' else [])
        gM = ws['gM'] if model.model_name == 'pRotatE' else None

        def adam_entries():
            """torch.optim.Adam bookkeeping (host only; state created lazily exactly like torch/optim/adam.py
            _init_group).  Called after the local kernels are in flight so that it does not delay them."""
            group = optimizer.param_groups[0]
            hyper = (float(group['lr']), float(group['betas'][0]), float(group['betas'][1]), float(group['eps']))
            entries = []
            for i, (p, g) in enumerate(zip(params, grads)):
                state = optimizer.state[p]
                if len(state) == 0:
                    state['step'] = torch.tensor(0.0, dtype=torch.float32)
                    state['exp_avg'] = torch.zeros_like(p, memory_format=torch.preserve_format)
                    state['exp_avg_sq'] = torch.zeros_like(p, memory_format=torch.preserve_format)
                state['step'] += 1
                entries.append((p.data_ptr(), g.data_ptr() if g is not None else None, state['exp_avg'].data_ptr(),
                                state['exp_avg_sq'].data_ptr(), p.numel(), int(state['step'].item()),
                                1 if (reg != 0.0 and i < 2) else 0))
            return entries, hyper

        # ---- multi-GPU plan: NVLink peer-memory exchange (csrc/kge_peer.cu) when it is set up and Adam is fused,
        # otherwise one NCCL all-reduce of the workspace followed by the replicated optimizer
        peer = ws['peer'] if (world > 1 and fused_adam) else None
        regions = entity_slices = None
        if peer is not None:
            from .peer import exchange_regions
            regions, entity_slices = exchange_regions(ws['param_floats'], model.nentity, model.entity_dim,
                                                      model._exchange_slices(B, world, N))
            from .peer import moment_ranges
            offsets = [(g.data_ptr() - ws['flat'].data_ptr()) // 4 for g in grads]
            model._own_moments(optimizer, moment_ranges(offsets, [p.numel() for p in params], regions, world))
            model._ws['exchange_regions'] = len(regions)
        elif world > 1 and getattr(optimizer, '_kge_sliced_moments', None):
            model._gather_moments(optimizer)

        # ---- local kernels ---------------------------------------------------------------------------------------
        _lib.call("kge_zero", _ptr(ws['flat']), ws['flat'].numel() * 4, st)
        if weight is not None:
            _lib.call("kge_weight_sum", _ptr(weight), B, _ptr(ws['wsum']), st)
        # the row arrays passed down start at this rank's first row: [positive, negative] hold the shard only,
        # weight / row losses are offset views of the whole-batch buffers
        common = (_ptr(positive), _ptr(negative), _ptr(weight[row_begin:]) if weight is not None else None,
                  _ptr(ws['wsum']) if weight is not None else None, B, 0, rows, N)
        neg_row, pos_row = ws['neg_row'][row_begin:], ws['pos_row'][row_begin:]
        wsp = model._buffer('train_ws', wbytes, torch.uint8, dev)
        if events is not None:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
        pos_rows, neg_rows = ws['pos_row'], ws['neg_row']
        model._ws['update_cancelled_on_error'] = fused_adam and peer is None and world == 1
        if fuse_entity:
            # one device: negatives + positive triple + backward, with torch.optim.Adam for the entity table applied
            # inside the entity-major pass (no dense entity gradient); R (and modulus) follow through kge_adam_step
            entries, hyper = adam_entries()
            e0 = entries[0]
            ea = _lib.KgeEntityAdam(exp_avg=e0[2], exp_avg_sq=e0[3], step=e0[5], lr=hyper[0], beta1=hyper[1],
                                    beta2=hyper[2], eps=hyper[3], l3_coefficient=reg,
                                    reg_partials=ws['reg'].data_ptr() if reg != 0.0 else None, n_reg_partials=148)
            _lib.call("kge_train_rows_adam", ctypes.byref(desc), mode_id, loss_kind, alpha, *common[:5], rows, N,
                      _ptr(neg_row), _ptr(pos_row), _ptr(ws['gR']), _ptr(gM), _ptr(wsp), wbytes, _ptr(err),
                      ctypes.byref(ea), st)
            entries = entries[1:]
            if events is not None:
                ev1.record()
                events.append((ev0, ev1))
            if xevents is not None:
                xev0, xev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                xev0.record()
        elif peer is None or len(regions) == 1:
            if rows:                                  # (a rank can be left without rows by a short last batch)
                _lib.call("kge_train_rows", ctypes.byref(desc), mode_id, loss_kind, alpha, *common,
                          _ptr(neg_row), _ptr(pos_row), _ptr(ws['gE']), _ptr(ws['gR']), _ptr(gM), None, _ptr(wsp),
                          wbytes, _ptr(err), st)      # negatives and the positive triple of every row, one call
            if events is not None:
                ev1.record()
                events.append((ev0, ev1))
            if xevents is not None:
                xev0, xev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                xev0.record()
            if fused_adam:
                entries, hyper = adam_entries()
            if peer is not None:
                if reg != 0.0:                       # value of the L3 term from the replicated pre-update tables
                    tensors = (_lib.KgeAdamTensor * len(entries))(*[_lib.KgeAdamTensor(*c) for c in entries])
                    _lib.call("kge_l3_partials", tensors, len(entries), _ptr(ws['reg']), ws['reg'].numel(), st)
                peer.reduce_adam(entries, hyper, ws['param_floats'], regions[0], ws['param_floats'], 2 * B,
                                 ws['rows_sum'], err, st, l3=reg)
            elif world > 1:
                torch.distributed.all_reduce(ws['flat'])     # [dE|dR|dM|row losses] in one piece
        else:
            # sliced: row pass + counting sort, then per entity range the entity-major backward on this stream and, as
            # soon as a range is final, its exchange (reduce-scatter + Adam + broadcast) on a second stream -- the
            # NVLink traffic of slice k runs under the computation of slice k+1
            pending = ctypes.c_int32(0)
            if rows:
                _lib.call("kge_train_rows_begin", ctypes.byref(desc), mode_id, loss_kind, alpha, *common,
                          _ptr(neg_row), _ptr(pos_row), _ptr(ws['gE']), _ptr(ws['gR']), _ptr(gM), _ptr(wsp),
                          wbytes, _ptr(err), ctypes.byref(pending), st)
            entries, hyper = adam_entries()
            if reg != 0.0:
                tensors = (_lib.KgeAdamTensor * len(entries))(*[_lib.KgeAdamTensor(*c) for c in entries])
                _lib.call("kge_l3_partials", tensors, len(entries), _ptr(ws['reg']), ws['reg'].numel(), st)
            main = torch.cuda.current_stream(dev)
            side = model._ws.get('exchange_stream')
            if side is None:
                side = model._ws['exchange_stream'] = torch.cuda.Stream(dev)
            side_ptr = ctypes.c_void_p(side.cuda_stream)
            last = len(regions) - 1
            for k, (region, (eb, ee)) in enumerate(zip(regions, entity_slices)):
                if pending.value:
                    _lib.call("kge_train_entity_pass", ctypes.byref(desc), mode_id, _ptr(wsp), rows, N, eb, ee, k,
                              _ptr(ws['gE']), _ptr(gM), st)
                if k == last:
                    if events is not None:
                        ev1.record()
                        events.append((ev0, ev1))
                    if xevents is not None:
                        xev0, xev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        xev0.record()
                side.wait_stream(main)
                peer.reduce_adam(entries, hyper, ws['param_floats'], region, ws['param_floats'],
                                 2 * B if k == last else 0, ws['rows_sum'], err, side_ptr, l3=reg)
            main.wait_stream(side)
        if peer is not None:
            pos_rows, neg_rows = ws['rows_sum'][:B], ws['rows_sum'][B:]

        # ---- optimizer ---------------------------------------------------------------------------------------------
        if fused_adam:
            if peer is None:
                # with the fused entity pass the first 148 partial sums of |x|^3 are the entity kernel's
                rp = ws['reg'][148:] if fuse_entity else ws['reg']
                tensors = (_lib.KgeAdamTensor * len(entries))(*[_lib.KgeAdamTensor(*c) for c in entries])
                _lib.call("kge_adam_step", tensors, len(entries), *hyper, reg,
                          _ptr(rp) if reg != 0.0 else None, rp.numel(), _ptr(err) if world == 1 else None, st)
            reg_partials = ws['reg'] if reg != 0.0 else None
            for p, g in zip(params, grads):
                p.grad = g if peer is None else None    # peer path: the workspace slots now carry parameter values;
                #                                         fused entity pass: entity_embedding.grad stays None
        else:
            # any other optimizer object: hand it our gradients and let it do its own update
            reg_partials = None
            if reg != 0.0:
                with torch.no_grad():
                    parts = ws['reg']
                    parts.zero_()
                    for i, (p, g) in enumerate(zip(params[:2], grads[:2])):
                        parts[i] = p.detach().abs().pow(3).sum(dtype=torch.float64)
                        g.add_(3.0 * reg * p.detach() * p.detach().abs())
                reg_partials = parts
            for p, g in zip(params, grads):
                p.grad = g
            optimizer.step()

        if xevents is not None:
            xev1.record()
            xevents.append((xev0, xev1))
        _lib.call("kge_loss_finalize", _ptr(pos_rows), _ptr(neg_rows), _ptr(weight),
                  _ptr(ws['wsum']) if weight is not None else None, B, reg,
                  _ptr(reg_partials) if reg_partials is not None else None,
                  reg_partials.numel() if reg_partials is not None else 0, _ptr(ws['out']), st)
        return ws['out']

    # ------------------------------------------------------------------------------------------ evaluation
    # largest key space (nentity * nrelation) for the device-built direct-address filter index: 2^27 keys = 0.5 GB of
    # int32 offsets per mode; beyond it (or with KGE_FILTER_HOST_INDEX=1) the host-built sorted-key index is used
    _DENSE_FILTER_KEYS = 1 << 27

    def _filter_index(self, all_true_triples, nentity, nrelation):
        """Cache entry for one `all_true_triples` list.  It holds the list itself (an id() alone can be reused by a later
        temporary such as train+valid+test) and is keyed on identity + length; a list mutated in place to the same length
        must be passed as a new object."""
        key = (len(all_true_triples), nentity, nrelation)
        held = self._filter_cache
        if held is None or held['list'] is not all_true_triples or held['key'] != key:
            self._filter_cache = held = {'list': all_true_triples, 'key': key, 'host': None, 'triples': {}, 'tables': {}}
        return held

    def _filter_tables(self, held, mode, dev, st):
        """The index of all true triples, resident on the device (once per list, mode and device):
        ('dense', offsets int32 [nentity*nrelation+1], entities int32) built ON the device by counting sort
        (kge_eval_filter_index_build), or ('sorted', keys, offsets, entities, nkeys) from the host-side FilterIndex."""
        tab = held['tables'].get((mode, dev))
        if tab is not None:
            return tab
        n, nentity, nrelation = held['key']
        if nentity * nrelation <= self._DENSE_FILTER_KEYS and not os.environ.get('KGE_FILTER_HOST_INDEX'):
            tri = held['triples'].get(dev)
            if tri is None:
                lst = held['list']
                try:          # python list of 3-tuples -> int64 [n,3]: the one host pass over the list (0.09 s per 483 k)
                    arr = np.fromiter(itertools.chain.from_iterable(lst), dtype=np.int64, count=3 * n)
                except (TypeError, ValueError):
                    arr = np.asarray(lst, dtype=np.int64).reshape(-1)
                if arr.size != 3 * n or (n and (len(lst[0]) != 3 or len(lst[-1]) != 3)):
                    raise ValueError('all_true_triples must be a list of (head, relation, tail)')
                tri = held['triples'][dev] = torch.from_numpy(arr).to(dev)
            lib = _lib.load()
            nkeys = nentity * nrelation
            offsets = torch.empty(nkeys + 1, dtype=torch.int32, device=dev)
            entities = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
            sbytes = int(lib.kge_eval_filter_index_scratch_bytes(nentity, nrelation))
            scratch = torch.empty(sbytes, dtype=torch.uint8, device=dev)
            _lib.call("kge_eval_filter_index_build", _ptr(tri), n, _lib.MODE_IDS[mode], nentity, nrelation, _ptr(offsets),
                      _ptr(entities), _ptr(scratch), sbytes, None, st)      # (scratch: stream-ordered reuse by the allocator)
            tab = ('dense', offsets, entities)
        else:
            if held['host'] is None:
                held['host'] = FilterIndex(held['list'], nentity, nrelation)
            keys, offsets, values = held['host'].table(mode)
            tab = ('sorted', torch.from_numpy(np.ascontiguousarray(keys)).to(dev),
                   torch.from_numpy(np.ascontiguousarray(offsets)).to(dev),
                   torch.from_numpy(np.ascontiguousarray(values)).to(dev) if values.size else
                   torch.zeros(1, dtype=torch.int32, device=dev), int(keys.size))
        held['tables'][(mode, dev)] = tab
        return tab

    def filtered_ranks(self, test_triples, all_true_triples, mode, query_chunk=4096, return_scores=False, exact=False,
                       return_approx=False):
        """Filtered rank of every test triple in `mode` (model.py:382-418 without the sort): int64 [len].
        Entities are sharded across the ranks of an initialised process group; the integer counts are
        all-reduced (bit-exact)."""
        counts, scores, approx = self._entity_rank_counts(test_triples, all_true_triples, mode, query_chunk, exact,
                                                          False, return_scores, return_approx)
        ranks = counts + 1
        if return_approx:
            return ranks, approx
        return (ranks, scores) if return_scores else ranks

    RANK_STATS = 6          # KGE_RANK_STATS of include/kge_b200.h

    def rank_statistics(self, test_triples, all_true_triples, mode, query_chunk=4096, exact=False):
        """Raw and tie-aware rank statistics of every test triple in `mode`: int64 numpy [len, 6], per query the number
        of candidate entities j != the positive with
          [0] j not filtered, s_j > s_pos          [3] s_j > s_pos
          [1] j not filtered, s_j == s_pos, j < pos  [4] s_j == s_pos, j < pos
          [2] j not filtered, s_j == s_pos, j > pos  [5] s_j == s_pos, j > pos
        where j is filtered when it completes the query into a triple of all_true_triples and s is the exact score of
        filtered_ranks (NaN is never greater or equal, -0.0 == +0.0).  1 + [0] + [1] is filtered_ranks' rank (for
        |s_pos| < 2^24, where its filter bias s_pos - 1 stays below s_pos) and
        1 + [3] + [4] the raw rank; ranks_from_statistics turns the table into optimistic, pessimistic or realistic
        ranks.  The path is filtered_ranks' (exact=True or KGE_EVAL_SIMT=1: the exact tile kernel); with an initialised
        process group every rank counts over its entity slice and the tallies are all-reduced (a collective: call it on
        every rank)."""
        return self._entity_rank_counts(test_triples, all_true_triples, mode, query_chunk, exact, True)[0]

    def _entity_rank_counts(self, test_triples, all_true_triples, mode, query_chunk, exact, stats,
                            return_scores=False, return_approx=False, path=None):
        """The query loop of filtered_ranks (stats=False: int64 counts [len]) and rank_statistics (stats=True: int64
        [len, 6]), with the [len, nentity] score dumps of filtered_ranks (None when not asked for).  path (a _PathQueries
        of path_rank_statistics): its answer sets and folded vectors replace the filter bitmap and the query vectors of
        each chunk; test_triples then only carries the positives, and the answer counts are left in path.answer_counts."""
        dev = self._device()
        st = _stream(dev)
        nentity, nrelation = self.entity_embedding.shape[0], self.relation_embedding.shape[0]
        cached = self._ws.get('queries_np')                  # test_step ranks the same list in both modes
        if path is not None:
            queries_all = np.asarray(test_triples, dtype=np.int64).reshape(-1, 3)
            queries_dev = torch.from_numpy(queries_all).to(dev, non_blocking=True)
        elif cached is not None and cached[0] is test_triples and cached[1] == len(test_triples) and cached[3].device == dev:
            queries_all, queries_dev = cached[2], cached[3]
        else:
            queries_all = np.asarray(test_triples, dtype=np.int64).reshape(-1, 3)
            queries_dev = torch.from_numpy(queries_all).to(dev, non_blocking=True)      # one H2D for the whole list
            self._ws['queries_np'] = (test_triples, len(test_triples), queries_all, queries_dev)
        if mode not in ('head-batch', 'tail-batch'):
            raise ValueError('negative batch mode %s not supported' % mode)       # dataloader.py:147
        if path is None:
            ftab = self._filter_tables(self._filter_index(all_true_triples, nentity, nrelation), mode, dev, st)
        rank, world = _dist()
        ent_begin, ent_end = shard_bounds(nentity, rank, world, align=128)
        desc = self._descriptor()
        err = self._err_flag()
        words = (nentity + 31) // 32
        phase = None
        if self.model_name == 'pRotatE':
            phase = self._buffer('phase_table', self.entity_embedding.numel(), torch.float32, dev)
            _lib.call("kge_eval_phase_table", ctypes.byref(desc), _ptr(phase), st)
        # DistMult / ComplEx: the all-entity scores are a dense contraction -> tcgen05 path (exact SIMT re-score of
        # the ambiguous band keeps the counts identical); KGE_EVAL_SIMT=1 forces the exact tile kernel
        exact = exact or return_scores or bool(os.environ.get("KGE_EVAL_SIMT"))
        gemm = bool(_lib.load().kge_eval_gemm_supported(ctypes.byref(desc))) and not exact
        two_stage = not exact and ((self.model_name == 'RotatE' and self.entity_dim % 8 == 0) or
                                   (self.model_name == 'pRotatE' and self.entity_dim % 4 == 0))
        nchunks = (queries_all.shape[0] + query_chunk - 1) // query_chunk
        # one int32 buffer [rank counts | per-chunk (ambiguous pairs, overflow flag) | path answer counts]: a single
        # all-reduce and a single read-back per call
        nq_all = queries_all.shape[0]
        ncol = self.RANK_STATS if stats else 1
        namb = 2 * max(nchunks, 1)
        tally = torch.zeros(nq_all * ncol + namb + (nq_all if path is not None else 0), dtype=torch.int32, device=dev)
        amb_counts = tally[nq_all * ncol:nq_all * ncol + namb].view(-1, 2) if (gemm or two_stage) else None
        if gemm:
            nE = self.entity_embedding.numel()
            ehi = self._buffer('gemm_ehi', nE, torch.float32, dev)
            elo = self._buffer('gemm_elo', nE, torch.float32, dev)
            enorm = self._buffer('gemm_enorm', nentity, torch.float32, dev)
            _lib.call("kge_eval_gemm_split", _ptr(self.entity_embedding), nentity, self.entity_dim, _ptr(ehi), _ptr(elo),
                      _ptr(enorm), st)
        counts_all = tally[:nq_all * ncol]
        scores = torch.empty((queries_all.shape[0], nentity), dtype=torch.float32, device=dev) if return_scores else None
        # tests: the approximations of the tcgen05 path or of the two-stage fast pass (to pin their error bands against
        # exact scores)
        approx = torch.zeros((queries_all.shape[0], nentity), dtype=torch.float32, device=dev) \
            if (return_approx and (gemm or two_stage)) else None
        m = _lib.MODE_IDS[mode]
        for ci, lo in enumerate(range(0, queries_all.shape[0], query_chunk)):
            queries = queries_dev[lo:lo + query_chunk]
            Q = queries.shape[0]
            bits = self._buffer('filter_bits', Q * words, torch.int32, dev)
            qvec = self._buffer('qvec', Q * self.entity_dim, torch.float32, dev)
            pos = self._buffer('pos_score', Q, torch.float32, dev)
            counts = counts_all[lo * ncol:(lo + Q) * ncol]
            if path is not None:                            # answer sets + folded paths (rank 0 counts the answers)
                answers = tally[nq_all * ncol + namb + lo:] if rank == 0 else None
                self._path_chunk(path, lo, Q, m, desc, bits, qvec, answers, err, st)
            # filter bitmap of the chunk, looked up on the device in the resident index (dataloader.py:134-154)
            elif ftab[0] == 'dense':
                _lib.call("kge_eval_filter_bits_lookup_dense", _ptr(ftab[1]), _ptr(ftab[2]), _ptr(queries), Q, m, nentity,
                          nrelation, _ptr(bits), st)
            else:
                _lib.call("kge_eval_filter_bits_lookup", _ptr(ftab[1]), _ptr(ftab[2]), _ptr(ftab[3]), ftab[4],
                          _ptr(queries), Q, m, nentity, nrelation, _ptr(bits), st)
            if path is None:
                _lib.call("kge_eval_query_vectors", ctypes.byref(desc), m, _ptr(queries), Q, _ptr(qvec), _ptr(err), st)
            _lib.call("kge_eval_positive_scores", ctypes.byref(desc), m, _ptr(qvec), _ptr(queries), Q, _ptr(phase),
                      _ptr(pos), st)
            events = self._ws.get('eval_events')            # bench.py: CUDA events around the dominant kernel
            if events is not None:
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record()
            if gemm:
                qhi = self._buffer('gemm_qhi', Q * self.entity_dim, torch.float32, dev)
                qlo = self._buffer('gemm_qlo', Q * self.entity_dim, torch.float32, dev)
                qnorm = self._buffer('gemm_qnorm', Q, torch.float32, dev)
                cap = int(os.environ.get('KGE_EVAL_AMB_CAP', Q * 1024))
                amb = self._buffer('gemm_amb', cap * 2, torch.int32, dev)
                _lib.call("kge_eval_gemm_split", _ptr(qvec), Q, self.entity_dim, _ptr(qhi), _ptr(qlo), _ptr(qnorm), st)
                gemm_args = (ctypes.byref(desc), m, _ptr(qvec), _ptr(qhi), _ptr(qlo), _ptr(qnorm), _ptr(queries), Q,
                             _ptr(pos), _ptr(bits), _ptr(ehi), _ptr(elo), _ptr(enorm), ent_begin, ent_end, _ptr(counts),
                             _ptr(amb), cap, _ptr(amb_counts[ci]))
                if stats:
                    _lib.call("kge_eval_gemm_count_rank_stats", *gemm_args, st)
                else:
                    _lib.call("kge_eval_gemm_count_ranks", *gemm_args,
                              _ptr(approx[lo:lo + Q]) if approx is not None else None, st)
            elif two_stage:
                cap = int(os.environ.get('KGE_EVAL_AMB_CAP', Q * 256))
                amb = self._buffer('gemm_amb', cap * 2, torch.int32, dev)
                two_stage_args = (ctypes.byref(desc), m, _ptr(qvec), _ptr(queries), Q, _ptr(phase), _ptr(pos), _ptr(bits),
                                  ent_begin, ent_end, _ptr(counts), _ptr(amb), cap, _ptr(amb_counts[ci]))
                if stats:
                    _lib.call("kge_eval_count_rank_stats_two_stage", *two_stage_args, st)
                else:
                    _lib.call("kge_eval_count_ranks_two_stage_approx", *two_stage_args,
                              _ptr(approx[lo:lo + Q]) if approx is not None else None, st)
            else:
                exact_args = (ctypes.byref(desc), m, _ptr(qvec), _ptr(queries), Q, _ptr(phase), _ptr(pos), _ptr(bits),
                              ent_begin, ent_end, _ptr(counts))
                if stats:
                    _lib.call("kge_eval_count_rank_stats", *exact_args, st)
                else:
                    _lib.call("kge_eval_count_ranks", *exact_args,
                              _ptr(scores[lo:lo + Q]) if scores is not None else None, st)
            if events is not None:
                ev1.record()
                events.append((ev0, ev1))
        if world > 1:
            torch.distributed.all_reduce(tally)              # integer sums over the entity shards: bit-exact; an
            #                                                  overflow flag on any rank re-runs the chunk everywhere
        host = tally.cpu().numpy()                           # the call's one host sync
        counts = host[:nq_all * ncol].astype(np.int64)
        if stats:
            counts = counts.reshape(nq_all, ncol)
        if path is not None:
            path.answer_counts = host[nq_all * ncol + namb:].astype(np.int64)
        if amb_counts is not None:
            amb_host = host[nq_all * ncol:nq_all * ncol + namb].reshape(-1, 2)
            self._ws['gemm_last_ambiguous' if gemm else 'two_stage_last_ambiguous'] = int(amb_host[:, 0].sum())
            for ci in np.nonzero(amb_host[:, 1])[0]:         # ambiguous list overflowed: exact kernel for that chunk
                lo = int(ci) * query_chunk
                if path is not None:
                    counts[lo:lo + query_chunk] = self._entity_rank_counts(
                        queries_all[lo:lo + query_chunk], None, mode, query_chunk, True, stats,
                        path=path.slice(lo, lo + query_chunk))[0]
                    continue
                chunk = [tuple(int(v) for v in row) for row in queries_all[lo:lo + query_chunk]]
                counts[lo:lo + query_chunk] = self._entity_rank_counts(chunk, all_true_triples, mode, query_chunk, True,
                                                                       stats)[0]
        self._raise_if_bad_index()
        return counts, scores, approx

    # device bytes of the exclusion bitmap of one query chunk (nentity / 8 per query): at 2.5 M entities a 4096-query
    # chunk would need 1.3 GB, so candidate_rank_statistics shrinks its chunk to stay within this
    _CAND_BITS_BUDGET = 1 << 28

    def candidate_rank_statistics(self, queries, candidates, mode, exclude_triples=None, query_chunk=4096,
                                  return_scores=False):
        """Rank statistics of every query against its own list of candidate entities (sampled evaluation, as in OGB's
        ogbl-wikikg2 / ogbl-biokg evaluators): int64 numpy [Q, 6] with the columns of rank_statistics, counted over the
        listed entries instead of all entities.

        queries: (h, r, t) tuples or an int64 array / tensor [Q, 3] (the layout of test_triples); the positive is the
        entity in the predicted slot ('head-batch': h, 'tail-batch': t).  candidates: int64 array / tensor [Q, C] (any
        device) or a list of equal-length lists of entity ids for the predicted slot; -1 is padding and may appear
        anywhere in a row, so ragged lists work.  Any other id outside [0, nentity) raises IndexError.  Per query, over
        the listed entries j (counted as often as they are listed; an entry naming the positive itself is skipped):
          [0] j not excluded, s_j > s_pos          [3] s_j > s_pos
          [1] j not excluded, s_j == s_pos, j < pos  [4] s_j == s_pos, j < pos
          [2] j not excluded, s_j == s_pos, j > pos  [5] s_j == s_pos, j > pos
        where j is excluded when it completes the query into a triple of exclude_triples (the filter of filtered_ranks)
        and s is the canonical exact score of filtered_ranks (NaN is never greater or equal, -0.0 == +0.0).
        ranks_from_statistics and metrics_from_ranks take the table unchanged; ranks_from_statistics(stats,
        filtered=False, ties='realistic') is OGB's rank 1 + #{neg > pos} + #{neg == pos} / 2, with two differences from
        OGB's evaluator: a negative that names the positive counts as a tie there and is skipped here, and OGB's scores
        come from torch, so near-ties may order differently.

        return_scores: also a float32 tensor [Q, C] on the model's device with the canonical score of every listed entry
        (s_pos, bit for bit, where an entry names the positive) and -inf at padding.  With an initialised process group
        every rank counts its slice of the candidate columns and the tallies are all-reduced (a collective: call it on
        every rank); return_scores then raises ValueError."""
        if mode not in ('head-batch', 'tail-batch'):
            raise ValueError('negative batch mode %s not supported' % mode)
        if isinstance(query_chunk, bool) or int(query_chunk) != query_chunk or int(query_chunk) < 1:
            raise ValueError('query_chunk must be a positive integer, got %r' % (query_chunk,))
        q_in = queries.detach() if isinstance(queries, torch.Tensor) else np.asarray(queries)
        if q_in.ndim != 2 or q_in.shape[1] != 3 or not _is_integer(q_in):
            raise ValueError('queries must be (h, r, t) triples: an integer array [Q, 3], got %s %s'
                             % (q_in.dtype, tuple(q_in.shape)))
        if isinstance(candidates, torch.Tensor):
            c_in = candidates.detach()
        else:
            try:
                c_in = np.asarray(candidates)
            except ValueError:                     # ragged nested lists
                raise ValueError('candidates must be an integer array [Q, C] (pad short lists with -1)') from None
        if c_in.ndim != 2 or c_in.shape[0] != q_in.shape[0] or not _is_integer(c_in):
            raise ValueError('candidates must be an integer array [Q, C] (pad short lists with -1) with Q = %d, got '
                             '%s %s' % (q_in.shape[0], c_in.dtype, tuple(c_in.shape)))
        rank, world = _dist()
        if return_scores and world > 1:
            raise ValueError('return_scores is single-process only: each rank scores a slice of the candidate columns')
        dev = self._device()
        st = _stream(dev)
        nq, ncand = int(c_in.shape[0]), int(c_in.shape[1])
        stats = torch.zeros(max(nq * self.RANK_STATS, 1), dtype=torch.int32, device=dev)
        scores = torch.empty((nq, ncand), dtype=torch.float32, device=dev) if return_scores else None
        if nq == 0 or ncand == 0:
            out = np.zeros((nq, self.RANK_STATS), dtype=np.int64)
            return (out, scores) if return_scores else out
        queries_dev = torch.as_tensor(q_in).to(device=dev, dtype=torch.int64, non_blocking=True).contiguous()
        cand_dev = torch.as_tensor(c_in).to(device=dev, dtype=torch.int64, non_blocking=True).contiguous()
        nentity, nrelation = self.entity_embedding.shape[0], self.relation_embedding.shape[0]
        words = (nentity + 31) // 32
        ftab = None
        chunk = int(query_chunk)
        if exclude_triples is not None:
            ftab = self._filter_tables(self._filter_index(exclude_triples, nentity, nrelation), mode, dev, st)
            chunk = max(1, min(chunk, self._CAND_BITS_BUDGET // (4 * words)))
        col_begin, col_end = shard_bounds(ncand, rank, world)
        desc = self._descriptor()
        err = self._err_flag()
        phase = None
        if self.model_name == 'pRotatE':
            phase = self._buffer('phase_table', self.entity_embedding.numel(), torch.float32, dev)
            _lib.call("kge_eval_phase_table", ctypes.byref(desc), _ptr(phase), st)
        m = _lib.MODE_IDS[mode]
        for lo in range(0, nq, chunk):
            q = queries_dev[lo:lo + chunk]
            Q = q.shape[0]
            bits = None
            if ftab is not None:
                bits = self._buffer('cand_bits', Q * words, torch.int32, dev)
                if ftab[0] == 'dense':
                    _lib.call("kge_eval_filter_bits_lookup_dense", _ptr(ftab[1]), _ptr(ftab[2]), _ptr(q), Q, m, nentity,
                              nrelation, _ptr(bits), st)
                else:
                    _lib.call("kge_eval_filter_bits_lookup", _ptr(ftab[1]), _ptr(ftab[2]), _ptr(ftab[3]), ftab[4],
                              _ptr(q), Q, m, nentity, nrelation, _ptr(bits), st)
            qvec = self._buffer('cand_qvec', Q * self.entity_dim, torch.float32, dev)
            pos = self._buffer('cand_pos_score', Q, torch.float32, dev)
            _lib.call("kge_eval_query_vectors", ctypes.byref(desc), m, _ptr(q), Q, _ptr(qvec), _ptr(err), st)
            _lib.call("kge_eval_positive_scores", ctypes.byref(desc), m, _ptr(qvec), _ptr(q), Q, _ptr(phase), _ptr(pos),
                      st)
            events = self._ws.get('candidate_events')        # tools/candidate_rate.py: CUDA events around the kernel
            if events is not None:
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record()
            _lib.call("kge_eval_candidate_rank_stats", ctypes.byref(desc), m, _ptr(qvec), _ptr(q), Q, _ptr(phase),
                      _ptr(pos), _ptr(cand_dev[lo:lo + Q]), ncand, col_begin, col_end, _ptr(bits),
                      _ptr(stats[lo * self.RANK_STATS:(lo + Q) * self.RANK_STATS]),
                      _ptr(scores[lo:lo + Q]) if scores is not None else None, _ptr(err), st)
            if events is not None:
                ev1.record()
                events.append((ev0, ev1))
        if world > 1:
            import torch.distributed as dist
            if dist.get_backend() == 'gloo':
                stats = stats.cpu()
            dist.all_reduce(stats)                           # integer sums over the column slices: bit-exact
        out = stats.cpu().numpy()[:nq * self.RANK_STATS].astype(np.int64).reshape(nq, self.RANK_STATS)   # one host sync
        self._raise_if_bad_index()
        return (out, scores) if return_scores else out

    TOPK_MAX = 256          # KGE_TOPK_MAX of include/kge_b200.h

    def predict_topk(self, queries, mode, k=10, exclude_triples=None):
        """Link prediction: the k most plausible entities for every query, best first.

        queries: (h, r, t) tuples or an int64 array [Q, 3] (the layout of test_triples); mode 'head-batch' predicts h,
        'tail-batch' predicts t, and the value in the predicted slot is ignored.  exclude_triples: optional list of true
        triples; every entity that completes a query into one of them is left out (the entity named in the predicted
        slot included).  Returns (ids int64 [Q, k], scores float32 [Q, k]) on the model's device, ordered by score
        descending, then entity id ascending; slots beyond the entities left hold id -1 and score -inf.  The scores are
        the exact ones of the filtered ranking (DESIGN.md section 3.8), for every model.  With an initialised process
        group every rank selects over its entity slice and the lists are merged (a collective: call it on every rank)."""
        if mode not in ('head-batch', 'tail-batch'):
            raise ValueError('negative batch mode %s not supported' % mode)
        if isinstance(k, bool) or int(k) != k or not 1 <= int(k) <= self.TOPK_MAX:
            raise ValueError('k must be an integer in [1, %d], got %r' % (self.TOPK_MAX, k))
        k = int(k)
        dev = self._device()
        st = _stream(dev)
        head = mode == 'head-batch'
        if isinstance(queries, torch.Tensor):
            queries_dev = queries.detach().to(device=dev, dtype=torch.int64).reshape(-1, 3).clone()
            queries_dev[:, 0 if head else 2] = 0
        else:
            arr = np.array(queries, dtype=np.int64).reshape(-1, 3)
            arr[:, 0 if head else 2] = 0         # unused; an out-of-range value would set the bad-index flag
            queries_dev = torch.from_numpy(arr).to(dev, non_blocking=True)
        return self._topk_chunks(queries_dev, mode, k, exclude_triples)

    def _topk_chunks(self, queries_dev, mode, k, exclude_triples, path=None, chunk=4096):
        """The chunk loop of predict_topk; path (a _PathQueries of predict_path_topk): its folded vectors and, with
        exclude_triples, its answer sets replace the query vectors and the exclusion bitmap of each chunk."""
        dev = self._device()
        st = _stream(dev)
        nq = queries_dev.shape[0]
        ids = torch.empty((nq, k), dtype=torch.int64, device=dev)
        scores = torch.empty((nq, k), dtype=torch.float32, device=dev)
        if nq == 0:
            return ids, scores
        nentity, nrelation = self.entity_embedding.shape[0], self.relation_embedding.shape[0]
        ftab = None
        if exclude_triples is not None and path is None:
            ftab = self._filter_tables(self._filter_index(exclude_triples, nentity, nrelation), mode, dev, st)
        rank, world = _dist()
        ent_begin, ent_end = shard_bounds(nentity, rank, world, align=128)
        desc = self._descriptor()
        err = self._err_flag()
        lib = _lib.load()
        words = (nentity + 31) // 32
        phase = None
        if self.model_name == 'pRotatE':
            phase = self._buffer('phase_table', self.entity_embedding.numel(), torch.float32, dev)
            _lib.call("kge_eval_phase_table", ctypes.byref(desc), _ptr(phase), st)
        m = _lib.MODE_IDS[mode]
        # the keys of this rank's slice, merged over the ranks below (one device: merged and decoded per chunk)
        local = torch.empty((nq, k), dtype=torch.int64, device=dev) if world > 1 else None
        for lo in range(0, nq, chunk):
            q = queries_dev[lo:lo + chunk]
            Q = q.shape[0]
            bits = None
            if path is not None:
                bits = self._buffer('topk_bits', Q * words, torch.int32, dev) if exclude_triples is not None else None
                qvec = self._buffer('topk_qvec', Q * self.entity_dim, torch.float32, dev)
                self._path_chunk(path, lo, Q, m, desc, bits, qvec, None, err, st)
            elif ftab is not None:
                bits = self._buffer('topk_bits', Q * words, torch.int32, dev)
                if ftab[0] == 'dense':
                    _lib.call("kge_eval_filter_bits_lookup_dense", _ptr(ftab[1]), _ptr(ftab[2]), _ptr(q), Q, m, nentity,
                              nrelation, _ptr(bits), st)
                else:
                    _lib.call("kge_eval_filter_bits_lookup", _ptr(ftab[1]), _ptr(ftab[2]), _ptr(ftab[3]), ftab[4],
                              _ptr(q), Q, m, nentity, nrelation, _ptr(bits), st)
            if path is None:
                qvec = self._buffer('topk_qvec', Q * self.entity_dim, torch.float32, dev)
                _lib.call("kge_eval_query_vectors", ctypes.byref(desc), m, _ptr(q), Q, _ptr(qvec), _ptr(err), st)
            sbytes = int(lib.kge_eval_topk_scratch_bytes(ctypes.byref(desc), Q, ent_begin, ent_end, k))
            _lib.check(min(sbytes, 0))
            scratch = self._buffer('topk_scratch', sbytes, torch.uint8, dev)
            keys = local[lo:lo + Q] if local is not None else self._buffer('topk_keys', Q * k, torch.int64, dev)
            events = self._ws.get('topk_events')             # tools/topk_rate.py: CUDA events around select + merge
            if events is not None:
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record()
            _lib.call("kge_eval_topk", ctypes.byref(desc), m, _ptr(qvec), Q, _ptr(phase), _ptr(bits), ent_begin,
                      ent_end, k, _ptr(keys), _ptr(scratch), sbytes, st)
            if local is None:
                _lib.call("kge_eval_topk_merge", _ptr(keys), Q, 1, k, None, _ptr(ids[lo:lo + Q]),
                          _ptr(scores[lo:lo + Q]), st)
            if events is not None:
                ev1.record()
                events.append((ev0, ev1))
        if local is not None:
            import torch.distributed as dist
            gloo = dist.get_backend() == 'gloo'          # gloo gathers host tensors only
            mine = local.cpu() if gloo else local
            parts = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(parts, mine)
            lists = torch.stack(parts, dim=1).to(dev).contiguous()          # [Q, world, k]
            _lib.call("kge_eval_topk_merge", _ptr(lists), nq, world, k, None, _ptr(ids), _ptr(scores), st)
        self._raise_if_bad_index()                        # the call's one host sync
        return ids, scores

    # ------------------------------------------------------------------------------------------ path queries
    def path_rank_statistics(self, anchors, paths, answers, all_true_triples, mode, query_chunk=4096, exact=False,
                             return_answer_counts=False):
        """Rank statistics of path queries (Guu et al. 2015; the 1p/2p/3p projection chains of complex-query benchmarks):
        int64 numpy [Q, 6] with the columns, tie rule and NaN / -0.0 handling of rank_statistics, where a candidate is
        filtered when it is in the query's answer set.

        anchors: int [Q] entity ids.  paths: int [Q, L] hop ids: r in [0, nrelation) follows relation r, r + nrelation
        follows it inverted, -1 pads a row after its last hop (every row has at least one hop).  answers: int [Q], the
        entity ranked.  mode 'tail-batch' asks (a, r1/.../rL, ?), the entities reached from a along the path; 'head-batch'
        asks (?, r1/.../rL, a), the entities x with x -r1-> ... -rL-> a.  The path is folded into one query vector
        (DESIGN.md section 3.13; one hop forward gives rank_statistics' numbers bit for bit) and the answer set is the
        breadth-first traversal of the path in all_true_triples, on the device.  The counting path is rank_statistics'
        (exact=True: the exact tile kernel).  return_answer_counts: also int64 [Q], the size of every answer set (the mean
        quantile of Guu et al. needs it).  A bad anchor, hop id, padding or answer raises IndexError.  With an initialised
        process group every rank counts over its entity slice and the tallies are all-reduced (a collective: call it on
        every rank)."""
        if isinstance(query_chunk, bool) or int(query_chunk) != query_chunk or int(query_chunk) < 1:
            raise ValueError('query_chunk must be a positive integer, got %r' % (query_chunk,))
        path, queries = self._path_queries(anchors, paths, mode, all_true_triples, answers)
        # two [chunk, nentity / 32] bitmaps (ping-pong of the traversal) stay within _CAND_BITS_BUDGET
        chunk = max(1, min(int(query_chunk), self._CAND_BITS_BUDGET // (8 * ((self.nentity + 31) // 32))))
        stats = self._entity_rank_counts(queries, None, mode, chunk, exact, True, path=path)[0]
        return (stats, path.answer_counts) if return_answer_counts else stats

    def predict_path_topk(self, anchors, paths, mode, k=10, exclude_triples=None):
        """The k most plausible answers of every path query, best first: (ids int64 [Q, k], scores float32 [Q, k]) on the
        model's device, with the order, scores and empty slots of predict_topk.  anchors, paths and mode as in
        path_rank_statistics; exclude_triples: optional list of true triples whose answer set along each path is left
        out.  A bad anchor, hop id or padding raises IndexError.  With an initialised process group every rank selects
        over its entity slice and the lists are merged (a collective: call it on every rank)."""
        if isinstance(k, bool) or int(k) != k or not 1 <= int(k) <= self.TOPK_MAX:
            raise ValueError('k must be an integer in [1, %d], got %r' % (self.TOPK_MAX, k))
        path, _ = self._path_queries(anchors, paths, mode, exclude_triples)
        chunk = 4096
        if exclude_triples is not None:
            chunk = max(1, min(chunk, self._CAND_BITS_BUDGET // (8 * ((self.nentity + 31) // 32))))
        return self._topk_chunks(path.anchors, mode, int(k), exclude_triples, path=path, chunk=chunk)

    def _path_queries(self, anchors, paths, mode, triples, answers=None):
        """(_PathQueries on the device, queries [Q, 3] int64 numpy with the answers in the mode's positive column or None)
        from the user's arrays; the filter indexes of `triples` the traversal reads are made resident."""
        if mode not in ('head-batch', 'tail-batch'):
            raise ValueError('negative batch mode %s not supported' % mode)
        host = [np.asarray(x.detach().cpu() if isinstance(x, torch.Tensor) else x) for x in (anchors, paths)]
        a, p = host
        if a.ndim != 1 or p.ndim != 2 or p.shape[0] != a.shape[0] or p.shape[1] < 1 or \
                (a.size and not _is_integer(a)) or (p.size and not _is_integer(p)):
            raise ValueError('anchors must be integer ids [Q] and paths integer hop ids [Q, L >= 1], got %s %s and %s %s'
                             % (a.dtype, tuple(a.shape), p.dtype, tuple(p.shape)))
        a, p = a.astype(np.int64), np.ascontiguousarray(p, dtype=np.int64)
        nentity, nrelation = self.entity_embedding.shape[0], self.relation_embedding.shape[0]
        queries = None
        if answers is not None:
            t = np.asarray(answers.detach().cpu() if isinstance(answers, torch.Tensor) else answers)
            if t.shape != a.shape or (t.size and not _is_integer(t)):
                raise ValueError('answers must be integer ids [%d], got %s %s' % (a.shape[0], t.dtype, tuple(t.shape)))
            if t.size and (t.min() < 0 or t.max() >= nentity):
                raise IndexError('answer id outside the entity table')
            queries = np.zeros((a.shape[0], 3), dtype=np.int64)
            queries[:, 0 if mode == 'head-batch' else 2] = t
        dev = self._device()
        st = _stream(dev)
        tables = None
        if triples is not None:
            held = self._filter_index(triples, nentity, nrelation)
            forward, inverse = bool(((p >= 0) & (p < nrelation)).any()), bool((p >= nrelation).any())
            if mode == 'head-batch':
                forward, inverse = inverse, forward          # as index readers: head-batch walks the path backwards
            tables = (self._filter_tables(held, 'tail-batch', dev, st) if forward else None,
                      self._filter_tables(held, 'head-batch', dev, st) if inverse else None)
        return _PathQueries(torch.from_numpy(a).to(dev), torch.from_numpy(p).to(dev), tables), queries

    def _path_chunk(self, path, lo, Q, m, desc, bits, qvec, answer_counts, err, st):
        """Queries [lo, lo + Q) of `path`: their folded vectors into qvec and, when bits is given, their answer sets into
        bits (answer_counts: int32 [Q] set sizes, or None)."""
        anchors, paths = path.anchors[lo:lo + Q], path.paths[lo:lo + Q]
        L = paths.shape[1]
        _lib.call("kge_eval_path_query_vectors", ctypes.byref(desc), m, _ptr(anchors), _ptr(paths), Q, L, _ptr(qvec),
                  _ptr(err), st)
        if bits is None:
            return
        nentity, nrelation = self.entity_embedding.shape[0], self.relation_embedding.shape[0]
        pong = self._buffer('path_pong', Q * ((nentity + 31) // 32), torch.int32, bits.device)
        tail, head = path.tables
        layouts = {t[0] for t in (tail, head) if t is not None}
        if layouts == {'sorted'}:
            name = "kge_eval_path_bits"
            index = [v for t in (tail, head) for v in ((_ptr(t[1]), _ptr(t[2]), _ptr(t[3]), t[4]) if t else (None,) * 3 + (0,))]
        elif layouts <= {'dense'}:
            name = "kge_eval_path_bits_dense"
            index = [_ptr(t[i]) if t else None for t in (tail, head) for i in (1, 2)]
        else:        # KGE_FILTER_HOST_INDEX changed between two calls on the same list
            raise ValueError('the two filter indexes of this triple list have different layouts; pass a new list object')
        _lib.call(name, *index, _ptr(anchors), _ptr(paths), Q, L, m, nentity, nrelation, _ptr(bits), _ptr(pong),
                  _ptr(answer_counts), st)

    # ------------------------------------------------------------------------------------------ relation prediction
    def _relation_filter_table(self, held, dev):
        """The relation index h*nentity+t -> relations of one true-triple list (filter_index.relation_table), resident on
        the device: built on the first relation request and kept in the list's _filter_cache entry next to the entity
        tables, which never pay for it."""
        tab = held['tables'].get(('relation', dev))
        if tab is None:
            keys, offsets, values = relation_table(held['list'], held['key'][1])
            tab = (torch.from_numpy(keys).to(dev), torch.from_numpy(offsets).to(dev),
                   torch.from_numpy(values).to(dev) if values.size else torch.zeros(1, dtype=torch.int32, device=dev),
                   int(keys.size))
            held['tables'][('relation', dev)] = tab
        return tab

    def _relation_operands(self, desc, dev, st):
        """(relation operand table, phase table) of kge_eval_relation_*: the table for RotatE / pRotatE, the phase table
        for pRotatE, None otherwise.  (The phase table is the buffer of filtered_ranks / predict_topk: same size, same
        values.)"""
        rel_table = phase = None
        if self.model_name in ('RotatE', 'pRotatE'):
            rel_table = self._buffer('rel_operand', self.relation_embedding.shape[0] * self.entity_dim, torch.float32, dev)
            _lib.call("kge_eval_relation_table", ctypes.byref(desc), _ptr(rel_table), st)
        if self.model_name == 'pRotatE':
            phase = self._buffer('phase_table', self.entity_embedding.numel(), torch.float32, dev)
            _lib.call("kge_eval_phase_table", ctypes.byref(desc), _ptr(phase), st)
        return rel_table, phase

    def filtered_relation_ranks(self, test_triples, all_true_triples, query_chunk=4096, return_scores=False):
        """Filtered relation rank of every test triple (h, r, t) among all relations for the query (h, ?, t): int64 [len],
        1 + #{r' != r unfiltered: s(h,r',t) > s(h,r,t)} + #{r' < r unfiltered: equal score}, where r' is filtered when
        (h, r', t) is in all_true_triples.  s is the exact 'single'-mode score (DESIGN.md section 3.9); metrics_from_ranks
        turns the ranks into MRR / Hits@k.  return_scores: also the [len, nrelation] scores (a filtered column holds
        s(h,r,t) - 1).  With an initialised process group every rank counts over its relation slice and the counts are
        all-reduced (a collective: call it on every rank)."""
        dev = self._device()
        st = _stream(dev)
        nentity, nrelation = self.entity_embedding.shape[0], self.relation_embedding.shape[0]
        queries_all = np.asarray(test_triples, dtype=np.int64).reshape(-1, 3)
        nq = queries_all.shape[0]
        queries_dev = torch.from_numpy(queries_all).to(dev, non_blocking=True)
        ftab = self._relation_filter_table(self._filter_index(all_true_triples, nentity, nrelation), dev)
        rank, world = _dist()
        rel_begin, rel_end = shard_bounds(nrelation, rank, world, align=64)
        desc = self._descriptor()
        err = self._err_flag()
        rel_table, phase = self._relation_operands(desc, dev, st)
        words = (nrelation + 31) // 32
        counts_all = torch.zeros(max(nq, 1), dtype=torch.int32, device=dev)
        scores = torch.empty((nq, nrelation), dtype=torch.float32, device=dev) if return_scores else None
        tail = _lib.MODE_IDS['tail-batch']
        for lo in range(0, nq, query_chunk):
            queries = queries_dev[lo:lo + query_chunk]
            Q = queries.shape[0]
            bits = self._buffer('rel_filter_bits', Q * words, torch.int32, dev)
            qvec = self._buffer('rel_qvec', Q * self.entity_dim, torch.float32, dev)
            pos = self._buffer('rel_pos_score', Q, torch.float32, dev)
            _lib.call("kge_eval_relation_filter_bits", _ptr(ftab[0]), _ptr(ftab[1]), _ptr(ftab[2]), ftab[3],
                      _ptr(queries), Q, nentity, nrelation, _ptr(bits), st)
            # s(h, r, t) of the positive: the tail-batch query vector and positive score, the same fold, op and order
            _lib.call("kge_eval_query_vectors", ctypes.byref(desc), tail, _ptr(queries), Q, _ptr(qvec), _ptr(err), st)
            _lib.call("kge_eval_positive_scores", ctypes.byref(desc), tail, _ptr(qvec), _ptr(queries), Q, _ptr(phase),
                      _ptr(pos), st)
            events = self._ws.get('relation_events')         # tools/relation_rate.py: CUDA events around the kernel
            if events is not None:
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record()
            _lib.call("kge_eval_relation_count_ranks", ctypes.byref(desc), _ptr(queries), Q, _ptr(rel_table), _ptr(phase),
                      _ptr(pos), _ptr(bits), rel_begin, rel_end, _ptr(counts_all[lo:lo + Q]),
                      _ptr(scores[lo:lo + Q]) if scores is not None else None, st)
            if events is not None:
                ev1.record()
                events.append((ev0, ev1))
        if world > 1:
            import torch.distributed as dist
            if dist.get_backend() == 'gloo':
                counts_all = counts_all.cpu()
            dist.all_reduce(counts_all)                      # integer sums over the relation slices: bit-exact
        ranks = counts_all.cpu().numpy()[:nq].astype(np.int64) + 1      # the call's one host sync
        self._raise_if_bad_index()
        return (ranks, scores) if return_scores else ranks

    def predict_relations(self, queries, k=10, exclude_triples=None):
        """Relation prediction: the k most plausible relations r for every query (h, ?, t), best first.

        queries: (h, r, t) tuples or an int64 array [Q, 3] (the layout of test_triples); the relation slot is ignored.
        exclude_triples: optional list of true triples; every r with (h, r, t) in it is left out.  Returns (ids int64
        [Q, k], scores float32 [Q, k]) on the model's device, ordered as predict_topk's: score descending, then relation
        id ascending, NaN last; slots beyond the relations left hold id -1 and score -inf (k may exceed nrelation).  The
        scores are the exact ones of filtered_relation_ranks.  With an initialised process group every rank selects over
        its relation slice and the lists are merged (a collective: call it on every rank)."""
        if isinstance(k, bool) or int(k) != k or not 1 <= int(k) <= self.TOPK_MAX:
            raise ValueError('k must be an integer in [1, %d], got %r' % (self.TOPK_MAX, k))
        k = int(k)
        dev = self._device()
        st = _stream(dev)
        if isinstance(queries, torch.Tensor):
            queries_dev = queries.detach().to(device=dev, dtype=torch.int64).reshape(-1, 3).clone()
            queries_dev[:, 1] = 0
        else:
            arr = np.array(queries, dtype=np.int64).reshape(-1, 3)
            arr[:, 1] = 0
            queries_dev = torch.from_numpy(arr).to(dev, non_blocking=True)
        nq = queries_dev.shape[0]
        ids = torch.empty((nq, k), dtype=torch.int64, device=dev)
        scores = torch.empty((nq, k), dtype=torch.float32, device=dev)
        if nq == 0:
            return ids, scores
        nentity, nrelation = self.entity_embedding.shape[0], self.relation_embedding.shape[0]
        ftab = None
        if exclude_triples is not None:
            ftab = self._relation_filter_table(self._filter_index(exclude_triples, nentity, nrelation), dev)
        rank, world = _dist()
        rel_begin, rel_end = shard_bounds(nrelation, rank, world, align=64)
        desc = self._descriptor()
        err = self._err_flag()
        lib = _lib.load()
        rel_table, phase = self._relation_operands(desc, dev, st)
        words = (nrelation + 31) // 32
        local = torch.empty((nq, k), dtype=torch.int64, device=dev) if world > 1 else None
        chunk = 4096
        for lo in range(0, nq, chunk):
            q = queries_dev[lo:lo + chunk]
            Q = q.shape[0]
            bits = None
            if ftab is not None:
                bits = self._buffer('rel_topk_bits', Q * words, torch.int32, dev)
                _lib.call("kge_eval_relation_filter_bits", _ptr(ftab[0]), _ptr(ftab[1]), _ptr(ftab[2]), ftab[3], _ptr(q),
                          Q, nentity, nrelation, _ptr(bits), st)
            sbytes = int(lib.kge_eval_relation_topk_scratch_bytes(ctypes.byref(desc), Q, rel_begin, rel_end, k))
            _lib.check(min(sbytes, 0))
            scratch = self._buffer('rel_topk_scratch', sbytes, torch.uint8, dev)
            keys = local[lo:lo + Q] if local is not None else self._buffer('rel_topk_keys', Q * k, torch.int64, dev)
            events = self._ws.get('relation_topk_events')    # tools/relation_rate.py: CUDA events around select + merge
            if events is not None:
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record()
            _lib.call("kge_eval_relation_topk", ctypes.byref(desc), _ptr(q), Q, _ptr(rel_table), _ptr(phase), _ptr(bits),
                      rel_begin, rel_end, k, _ptr(keys), _ptr(scratch), sbytes, _ptr(err), st)
            if local is None:
                _lib.call("kge_eval_topk_merge", _ptr(keys), Q, 1, k, None, _ptr(ids[lo:lo + Q]),
                          _ptr(scores[lo:lo + Q]), st)
            if events is not None:
                ev1.record()
                events.append((ev0, ev1))
        if local is not None:
            import torch.distributed as dist
            gloo = dist.get_backend() == 'gloo'          # gloo gathers host tensors only
            mine = local.cpu() if gloo else local
            parts = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(parts, mine)
            lists = torch.stack(parts, dim=1).to(dev).contiguous()          # [Q, world, k]
            _lib.call("kge_eval_topk_merge", _ptr(lists), nq, world, k, None, _ptr(ids), _ptr(scores), st)
        self._raise_if_bad_index()                        # the call's one host sync
        return ids, scores

    # ------------------------------------------------------------------------------------------ similarity search
    def nearest_neighbors(self, items, table='entity', k=10, metric='cosine', exclude_self=True):
        """Similarity search: the k rows of the entity or relation table closest to each query, best first.

        table: 'entity' (rows of entity_embedding) or 'relation' (rows of relation_embedding).  A row is the stored row
        as one flat real vector: [re | im] together for double tables, and the stored phases, unscaled, for RotatE /
        pRotatE relations (phase wrap-around is not modelled).  items: 1-D integer row ids (list, array or tensor), or a
        2-D float array / tensor [Q, width] of free query vectors (any device).  metric, "larger is more similar":
        'dot' = acc(q x), 'cosine' = acc(q x) / (|q| |x|) with |v| = sqrt(acc(v v)), 'l2' = -sqrt(acc((q - x)^2)),
        'l1' = -acc(|q - x|), where acc is the canonical blocked float32 sum of DESIGN.md section 4, so the scores are
        bit-reproducible; a zero row under cosine scores NaN.  exclude_self: an id query leaves its own row out (rows
        with identical values stay); vector queries exclude nothing.  Returns (ids int64 [Q, k], scores float32 [Q, k])
        on the model's device, ordered as predict_topk's: score descending, then row id ascending, NaN last, -0.0 ==
        +0.0; slots beyond the rows left hold id -1 and score -inf.  An id outside the table raises IndexError.  With an
        initialised process group every rank selects over its row slice and the lists are merged (a collective: call it
        on every rank with the same items)."""
        if table not in ('entity', 'relation'):
            raise ValueError("table must be 'entity' or 'relation', got %r" % (table,))
        if metric not in _lib.SIM_IDS:
            raise ValueError('metric must be one of %s, got %r' % (', '.join(_lib.SIM_IDS), metric))
        if isinstance(k, bool) or int(k) != k or not 1 <= int(k) <= self.TOPK_MAX:
            raise ValueError('k must be an integer in [1, %d], got %r' % (self.TOPK_MAX, k))
        k = int(k)
        X = self.entity_embedding if table == 'entity' else self.relation_embedding
        rows, width = X.shape
        arr = items.detach() if isinstance(items, torch.Tensor) else np.ascontiguousarray(items)
        if arr.ndim == 1:
            if arr.shape[0] and not _is_integer(arr):
                raise ValueError('1-D items must be integer row ids, got dtype %s' % (arr.dtype,))
        elif arr.ndim == 2:
            if not (arr.dtype.is_floating_point if isinstance(arr, torch.Tensor)
                    else np.issubdtype(arr.dtype, np.floating)):
                raise ValueError('2-D items must be float query vectors [Q, %d], got dtype %s' % (width, arr.dtype))
            if arr.shape[1] != width:
                raise ValueError('query vectors of width %d, the %s table has width %d' % (arr.shape[1], table, width))
        else:
            raise ValueError('items must be 1-D row ids or 2-D query vectors, got %d dimensions' % arr.ndim)
        dev = self._device()
        st = _stream(dev)
        by_id = arr.ndim == 1
        if by_id:
            src = torch.as_tensor(arr) if arr.shape[0] else torch.empty(0, dtype=torch.int64)
            queries = src.to(device=dev, dtype=torch.int64).contiguous()
        else:
            queries = torch.as_tensor(arr).to(device=dev, dtype=torch.float32).contiguous()
        nq = queries.shape[0]
        ids = torch.empty((nq, k), dtype=torch.int64, device=dev)
        scores = torch.empty((nq, k), dtype=torch.float32, device=dev)
        if nq == 0:
            return ids, scores
        rank, world = _dist()
        row_begin, row_end = shard_bounds(rows, rank, world, align=128)
        desc = self._descriptor()
        err = self._err_flag()
        lib = _lib.load()
        tab = _lib.TABLE_ENTITY if table == 'entity' else _lib.TABLE_RELATION
        sim = _lib.SIM_IDS[metric]
        xnorm = None
        if metric == 'cosine':             # recomputed every call: training changes the tables, and it is one read
            xnorm = self._buffer('nn_xnorm', rows, torch.float32, dev)
            _lib.call("kge_similarity_norms", ctypes.byref(desc), tab, None, rows, _ptr(xnorm), st)
        # the keys of this rank's slice, merged over the ranks below (one device: merged and decoded per chunk)
        local = torch.empty((nq, k), dtype=torch.int64, device=dev) if world > 1 else None
        chunk = 4096
        for lo in range(0, nq, chunk):
            q = queries[lo:lo + chunk]
            Q = q.shape[0]
            self_ids = None
            if by_id:
                qvec = self._buffer('nn_qvec', Q * width, torch.float32, dev)
                _lib.call("kge_similarity_rows", ctypes.byref(desc), tab, _ptr(q), Q, _ptr(qvec), _ptr(err), st)
                self_ids = q if exclude_self else None
            else:
                qvec = q
            qnorm = None
            if metric == 'cosine':
                qnorm = self._buffer('nn_qnorm', Q, torch.float32, dev)
                _lib.call("kge_similarity_norms", ctypes.byref(desc), tab, _ptr(qvec), Q, _ptr(qnorm), st)
            sbytes = int(lib.kge_similarity_topk_scratch_bytes(ctypes.byref(desc), tab, Q, row_begin, row_end, k))
            _lib.check(min(sbytes, 0))
            scratch = self._buffer('nn_scratch', sbytes, torch.uint8, dev)
            keys = local[lo:lo + Q] if local is not None else self._buffer('nn_keys', Q * k, torch.int64, dev)
            events = self._ws.get('nn_events')               # tools/similarity_rate.py: CUDA events around select + merge
            if events is not None:
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record()
            _lib.call("kge_similarity_topk", ctypes.byref(desc), tab, sim, _ptr(qvec), _ptr(qnorm), _ptr(xnorm),
                      _ptr(self_ids), Q, row_begin, row_end, k, _ptr(keys), _ptr(scratch), sbytes, st)
            if local is None:
                _lib.call("kge_eval_topk_merge", _ptr(keys), Q, 1, k, None, _ptr(ids[lo:lo + Q]),
                          _ptr(scores[lo:lo + Q]), st)
            if events is not None:
                ev1.record()
                events.append((ev0, ev1))
        if local is not None:
            import torch.distributed as dist
            gloo = dist.get_backend() == 'gloo'          # gloo gathers host tensors only
            mine = local.cpu() if gloo else local
            parts = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(parts, mine)
            lists = torch.stack(parts, dim=1).to(dev).contiguous()          # [Q, world, k]
            _lib.call("kge_eval_topk_merge", _ptr(lists), nq, world, k, None, _ptr(ids), _ptr(scores), st)
        self._raise_if_bad_index()                        # the call's one host sync
        return ids, scores

    @staticmethod
    def test_step(model, test_triples, all_true_triples, args):
        '''
        Evaluate the model on test or valid datasets (reference: model.py:314-429).
        '''
        model.eval()

        if args.countries:
            # Countries S* are evaluated on AUC-PR (model.py:322-344); 5 regions x |test| scores, sklearn on host
            from sklearn.metrics import average_precision_score
            sample = list()
            y_true = list()
            for head, relation, tail in test_triples:
                for candidate_region in args.regions:
                    y_true.append(1 if candidate_region == tail else 0)
                    sample.append((head, relation, candidate_region))
            sample = torch.LongTensor(sample)
            with torch.no_grad():
                y_score = model(sample).squeeze(1).cpu().numpy()
            y_true = np.array(y_true)
            auc_pr = average_precision_score(y_true, y_score)
            return {'auc_pr': auc_pr}

        # filtered MRR / MR / HITS@1,3,10 (model.py:346-427)
        batch = max(1, int(getattr(args, 'test_batch_size', 1)))
        steps_per_mode = (len(test_triples) + batch - 1) // batch
        total_steps = 2 * steps_per_mode
        log_every = max(1, int(getattr(args, 'test_log_steps', 1000)))
        all_ranks = []
        step = 0
        with torch.no_grad():
            for mode in ('head-batch', 'tail-batch'):
                all_ranks.append(model.filtered_ranks(test_triples, all_true_triples, mode))
                for _ in range(steps_per_mode):          # same progress lines as model.py:420-423
                    if step % log_every == 0:
                        logging.info('Evaluating the model... (%d/%d)' % (step, total_steps))
                    step += 1
        return metrics_from_ranks(np.concatenate(all_ranks))


def ranks_from_statistics(stats, filtered=True, ties='stable'):
    """Ranks from the [len, 6] table of KGEModel.rank_statistics: the filtered (filtered=True) or raw ranks, with the
    positive placed among the candidates of equal score
      'optimistic'   first:              1 + greater
      'stable'       by entity id:       1 + greater + equal_before        (filtered: the rank of filtered_ranks)
      'pessimistic'  last:               1 + greater + equal_before + equal_after
      'realistic'    in the middle:      1 + greater + (equal_before + equal_after) / 2   (the expected rank under a random
                                         order of the ties)
    int64 [len], float64 for 'realistic'; metrics_from_ranks turns them into MRR / MR / HITS@k."""
    table = np.asarray(stats)
    if table.ndim != 2 or table.shape[1] != KGEModel.RANK_STATS or not np.issubdtype(table.dtype, np.integer):
        raise ValueError('stats must be an integer table [len, %d] (KGEModel.rank_statistics), got %s %s'
                         % (KGEModel.RANK_STATS, table.dtype, table.shape))
    g, eb, ea = (table[:, c].astype(np.int64) for c in ((0, 1, 2) if filtered else (3, 4, 5)))
    if ties == 'optimistic':
        return 1 + g
    if ties == 'stable':
        return 1 + g + eb
    if ties == 'pessimistic':
        return 1 + g + eb + ea
    if ties == 'realistic':
        return 1.0 + g + (eb + ea) / 2.0
    raise ValueError("ties must be 'optimistic', 'stable', 'pessimistic' or 'realistic', got %r" % (ties,))


def metrics_from_ranks(ranks):
    """model.py:412-427: per-query MRR / MR / HITS@1,3,10 (head-batch queries first, then tail-batch) averaged with
    python's `sum(list) / len(logs)`.  The same float64 values go through the same builtin sum() in the same order, so
    the metrics are bit-identical to the reference's loop over per-query dicts (also under CPython >= 3.12's compensated
    float sum) without building 2*|test| dicts."""
    ranking = np.asarray(ranks).astype(np.float64)
    per_query = {
        'MRR': 1.0 / ranking,
        'MR': ranking,
        'HITS@1': (ranking <= 1).astype(np.float64),
        'HITS@3': (ranking <= 3).astype(np.float64),
        'HITS@10': (ranking <= 10).astype(np.float64),
    }
    return {name: sum(values.tolist()) / len(ranking) for name, values in per_query.items()}


class _PathQueries:
    """Path queries on the device (anchors int64 [Q], hop ids int64 [Q, L]) and the resident filter indexes their answer
    sets are traversed in, (tail index, head index) with None for one no hop reads, or None without answer sets."""

    def __init__(self, anchors, paths, tables):
        self.anchors, self.paths, self.tables = anchors, paths, tables
        self.answer_counts = None            # int64 numpy [Q], left here by KGEModel._entity_rank_counts

    def slice(self, lo, hi):
        return _PathQueries(self.anchors[lo:hi], self.paths[lo:hi], self.tables)


class _NamedView:
    """Descriptor provider for the public score methods: same scalars as the owning model, another model name."""

    def __init__(self, owner, name):
        self.owner, self.name = owner, name

    def _descriptor(self, entity, relation, modulus):
        return self.owner._descriptor(entity, relation, modulus, name=self.name)

    def _err_flag(self):
        return self.owner._err_flag()
