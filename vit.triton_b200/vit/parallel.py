"""Batch-sharded data parallelism: one process per GPU, replicated weights, ONE collective per step.

The reference is single-GPU (no distributed code at all, SURVEY.md 2a).  Every image is independent
through the whole forward (vit/vit.py:240-247), so the batch shards with no data-path exchange; the
only collective is the all-gather of the pooled CLS embeddings ((B/G, D) per rank, a few hundred KB:
latency-bound over NVLink/NVSwitch).  On GPUs with peer access that step is ONE kernel of ours
(``PeerGather``: pool + P2P stores into every peer's gather buffer + flag exchange, no NCCL call);
``all_gather_rows`` over torch.distributed is the portable form (NCCL for ragged shards or when
symmetric memory is unavailable; the CPU tests drive the same wrapper over gloo).
"""
import ctypes
import os
import warnings
from typing import Optional, Tuple

import torch
import torch.distributed as dist


def shard_bounds(total: int, world_size: int, rank: int) -> Tuple[int, int]:
    """Contiguous [start, stop) of ``total`` items owned by ``rank``; the first ``total % world``
    ranks hold one extra item."""
    assert world_size > 0 and 0 <= rank < world_size, f"Invalid rank/world size: {rank}, {world_size}"
    base, extra = divmod(total, world_size)
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


def all_gather_rows(local: torch.Tensor, total_rows: int, group=None) -> torch.Tensor:
    """All-gather row shards laid out by ``shard_bounds`` into the full (total_rows, ...) tensor.
    Equal shards take the single-buffer path; ragged shards are padded to the largest one."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    lo, hi = shard_bounds(total_rows, world, rank)
    assert local.shape[0] == hi - lo, f"Rank {rank} should hold {hi - lo} rows, provided: {local.shape[0]}"
    local = local.contiguous()
    tail = tuple(local.shape[1:])
    if total_rows % world == 0:
        out = torch.empty((total_rows,) + tail, device=local.device, dtype=local.dtype)
        dist.all_gather_into_tensor(out, local, group=group)
        return out
    widest = (total_rows + world - 1) // world
    padded = torch.zeros((widest,) + tail, device=local.device, dtype=local.dtype)
    padded[:local.shape[0]] = local
    pieces = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(pieces, padded, group=group)
    rows = []
    for r, piece in enumerate(pieces):
        a, b = shard_bounds(total_rows, world, r)
        rows.append(piece[:b - a])
    return torch.cat(rows, dim=0)


class PeerGather:
    """Pool + all-gather as one kernel over NVLink peer memory (``vt_pool_cls_allgather``).

    Owns four symmetric gather buffers of (world * B_local, D) used in turn (step mod 4, see the protocol
    note in csrc/rowwise.cu), one symmetric array of ``world`` uint32 flag counters — allocated and
    exchanged through ``torch.distributed._symmetric_memory`` — and, in plain device memory, the step
    counter and two local (world * B_local, D) output buffers.  The step number lives in device memory,
    so every launch has the same arguments: the kernels are CUDA-graph capturable.

    ``__call__(hidden)``       synchronous all-gather of this step's CLS rows (PUT | GET in one launch).
    ``put(hidden)``/``get()``  the split form: ``put`` stores + signals and never waits; ``get(lag=1)``
                               collects the step before the last ``put`` (its flags arrived a whole
                               forward ago, so no rank waits for a slower peer), ``get(lag=0)`` the last.
    Results are views of two alternating local buffers: valid until the next-but-one collect."""

    def __init__(self, batch_local: int, dim: int, dtype: torch.dtype, device: torch.device, group=None):
        import torch.distributed._symmetric_memory as symm_mem
        from .kernels import _lib
        self._lib = _lib
        self.group = group if group is not None else dist.group.WORLD
        self.world = dist.get_world_size(self.group)
        self.rank = dist.get_rank(self.group)
        assert self.world <= 16, f"At most 16 peers, provided: {self.world}"
        self.batch_local, self.dim, self.dtype = batch_local, dim, dtype
        self.bufs = symm_mem.empty((4, self.world * batch_local, dim), dtype=dtype, device=device)
        self.flags = symm_mem.empty((self.world,), dtype=torch.int32, device=device)
        self.flags.zero_()
        self._buf_handle = symm_mem.rendezvous(self.bufs, self.group)
        self._flag_handle = symm_mem.rendezvous(self.flags, self.group)
        self.ctrl = torch.zeros((2,), dtype=torch.int32, device=device)
        self.outs = torch.empty((2, self.world * batch_local, dim), dtype=dtype, device=device)
        torch.cuda.synchronize(device)
        dist.barrier(self.group)                       # every rank's flags are zero before anyone writes
        buf_bytes = self.bufs[0].numel() * self.bufs.element_size()
        base = [int(a) for a in self._buf_handle.buffer_ptrs]
        self._out_table = (ctypes.c_void_p * (4 * self.world))(*[a + b * buf_bytes for b in range(4) for a in base])
        self._flag_table = (ctypes.c_void_p * self.world)(*[int(a) for a in self._flag_handle.buffer_ptrs])
        self._collects = 0

    def _launch(self, hidden: Optional[torch.Tensor], out: Optional[torch.Tensor], mode: int, lag: int) -> None:
        _lib = self._lib
        if hidden is not None:
            assert hidden.is_cuda and hidden.dim() == 3, f"Expected CUDA (B, N, D) hidden states, provided: {tuple(hidden.shape)}"
            assert hidden.shape[0] == self.batch_local and hidden.shape[2] == self.dim and hidden.dtype == self.dtype, \
                f"PeerGather was built for ({self.batch_local}, *, {self.dim}) {self.dtype}, provided: {tuple(hidden.shape)} {hidden.dtype}"
            assert hidden.stride(2) == 1 and hidden.stride(0) % 8 == 0
        ref = hidden if hidden is not None else out
        _lib.call("vt_pool_cls_allgather", _lib.ptr(hidden), self.batch_local, self.dim,
                  hidden.stride(0) if hidden is not None else self.dim, _lib.dtype_code(ref),
                  ctypes.cast(self._out_table, ctypes.c_void_p), ctypes.cast(self._flag_table, ctypes.c_void_p),
                  self.rank, self.world, self.ctrl.data_ptr(), _lib.ptr(out), mode, lag, _lib.stream_ptr(ref))

    def _next_out(self) -> torch.Tensor:
        self._collects += 1
        return self.outs[self._collects & 1]

    def __call__(self, hidden: torch.Tensor) -> torch.Tensor:
        out = self._next_out()
        self._launch(hidden, out, self._lib.VT_PG_PUT | self._lib.VT_PG_GET, 0)
        return out

    def put(self, hidden: torch.Tensor) -> None:
        self._launch(hidden, None, self._lib.VT_PG_PUT, 0)

    def get(self, lag: int = 1) -> torch.Tensor:
        out = self._next_out()
        self._launch(None, out, self._lib.VT_PG_GET, lag)
        return out


_DTYPE_CODES = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2, torch.uint8: 3}


class DataParallelVIT(torch.nn.Module):
    """Wraps a replicated ``VIT``: each rank runs its slice of the global batch and all ranks receive
    the gathered (B, D) pooled embeddings."""

    def __init__(self, model: torch.nn.Module, group=None, peer_gather: Optional[bool] = None,
                 output: str = "pooled", interpolate_pos_encoding: bool = False):
        """``output``: "pooled" gathers the CLS embeddings (B, D); "pooler" the HF pooler output
        tanh(dense(CLS)) (B, D) of a model built with ``add_pooling_layer=True``; "logits" the class
        logits (B, num_labels) of a model built with a classifier head (``VIT(num_labels=...)``, or the mean of the
        two DeiT heads of ``VIT(..., distillation_head=True)``); "image_embeds" the CLIP image embeddings
        (B, projection_dim) of ``VIT(..., clip=True, projection_dim=...)`` (on a CLIP model "pooler" gathers its
        ``pooler_output``, post_layernorm of the CLS rows).
        ``peer_gather``: None = use the fused pool + peer-store kernel whenever it applies (CUDA,
        NCCL group, equal shards, symmetric memory available; VT_PEER_GATHER=0 disables), True =
        require it, False = always all-gather through torch.distributed.  Which one runs is decided
        COLLECTIVELY the first time a (local batch, global batch, dtype) combination is seen: every rank
        contributes what it wants and what it holds to one all-reduce, so either all ranks use the
        peer-store kernel with identical shapes or none does.
        ``interpolate_pos_encoding``: passed to every model call (``VIT.forward``'s flag: inputs at any resolution,
        the position table resampled to their patch grid); the gathered rows keep their width, so the collective is
        the same."""
        super().__init__()
        self.model = model
        self.group = group
        self.peer_gather = peer_gather
        assert output in ("pooled", "pooler", "logits", "image_embeds"), \
            f"output must be 'pooled', 'pooler', 'logits' or 'image_embeds', provided: {output}"
        self.output = output
        self.interpolate_pos_encoding = bool(interpolate_pos_encoding)
        self._peer = None          # PeerGather of the current plan
        self._plans = {}           # (B_local, global_batch, dtype) -> PeerGather | None (= torch.distributed)
        self._pending = False      # a put() whose rows have not been collected yet (pipelined form)
        self.gather_impl = "none"  # what the last forward used: "peer-store kernel" | "torch.distributed" | "none"

    @property
    def world_size(self) -> int:
        return dist.get_world_size(self.group) if dist.is_initialized() else 1

    @property
    def rank(self) -> int:
        return dist.get_rank(self.group) if dist.is_initialized() else 0

    def local_slice(self, global_batch: int) -> Tuple[int, int]:
        return shard_bounds(global_batch, self.world_size, self.rank)

    def forward_local(self, x_local: torch.Tensor) -> torch.Tensor:
        """Pooled embeddings (or pooler output / logits) of this rank's images, (B_local, D | num_labels); no
        communication."""
        kw = self._model_kwargs()
        if self.output == "logits":
            return self.model.logits(x_local, **kw)
        if self.output == "pooler":
            return self.model.pooler_output(x_local, **kw)
        if self.output == "image_embeds":
            return self.model.image_embeds(x_local, **kw)
        return self.model.pooled(x_local, **kw)

    def _model_kwargs(self) -> dict:
        # the keyword only when set: the wrapper also takes models whose methods have no such parameter
        return dict(interpolate_pos_encoding=True) if self.interpolate_pos_encoding else {}

    def _rows(self, x_local: torch.Tensor) -> torch.Tensor:
        """(B_local, *, D) tensor whose [:, 0, :] rows this rank contributes: the final hidden states for
        "pooled" (the gather kernel pools them itself), the head's output as a one-token sequence otherwise."""
        if self.output == "pooled":
            kw = self._model_kwargs()
            return self.model.forward_uint8(x_local, **kw) if x_local.dtype == torch.uint8 else self.model(x_local, **kw)
        return self.forward_local(x_local).unsqueeze(1)

    def forward(self, x_local: torch.Tensor, global_batch: Optional[int] = None) -> torch.Tensor:
        """x_local: this rank's shard of the global batch (as laid out by ``local_slice``).
        Returns the pooled embeddings of the WHOLE batch, (B, D), identical on every rank."""
        world = self.world_size
        if world == 1:
            return self.forward_local(x_local)
        assert not self._pending, "forward() called with a submit() outstanding: call flush() first"
        if global_batch is None:
            global_batch = x_local.shape[0] * world
        peer = self._plan(x_local, global_batch)
        if peer is not None:
            self.gather_impl = "peer-store kernel"
            return peer(self._rows(x_local).contiguous())
        self.gather_impl = "torch.distributed"
        return all_gather_rows(self.forward_local(x_local), global_batch, self.group)

    # ------------------------------------------------------------------ pipelined form
    def submit(self, x_local: torch.Tensor, global_batch: Optional[int] = None) -> Optional[torch.Tensor]:
        """Pipelined steps: run this rank's forward, hand its rows to the peers (store + signal, never
        waits) and return the gathered embeddings of the PREVIOUS ``submit`` (None for the first one) —
        their flags arrived a whole forward ago, so no rank ever waits for a slower peer inside a step.
        ``flush()`` returns the last step's.  Falls back to the synchronous gather (returning the CURRENT
        step's result one call late) when the peer-store kernel does not apply."""
        world = self.world_size
        if global_batch is None:
            global_batch = x_local.shape[0] * max(world, 1)
        peer = self._plan(x_local, global_batch) if world > 1 else None
        if peer is None:
            prev = getattr(self, "_late", None)
            self._late = self.forward(x_local, global_batch) if world > 1 else self.forward_local(x_local)
            self._pending_late = True
            return prev
        assert self._peer is None or self._peer is peer or not self._pending, "flush() before changing the batch shape"
        self._peer = peer
        self.gather_impl = "peer-store kernel"
        peer.put(self._rows(x_local).contiguous())
        had = self._pending
        self._pending = True
        return peer.get(lag=1) if had else None

    def flush(self) -> Optional[torch.Tensor]:
        """Gathered embeddings of the last ``submit`` (None if nothing is outstanding)."""
        if getattr(self, "_pending_late", False):
            self._pending_late = False
            out, self._late = self._late, None
            return out
        if not self._pending:
            return None
        self._pending = False
        return self._peer.get(lag=0)

    # ------------------------------------------------------------------ collective plan (cold path)
    def _out_dim(self) -> int:
        if self.output == "logits":
            head = self.model.classifier if self.model.classifier is not None else self.model.cls_classifier
            return head.weight.shape[1]
        if self.output == "image_embeds":
            return self.model.visual_projection.weight.shape[1]
        return int(getattr(self.model, "hidden_dim", 0))

    def _local_want(self, x_local: torch.Tensor, global_batch: int) -> bool:
        if self.peer_gather is False:
            return False
        if self.peer_gather is None and os.environ.get("VT_PEER_GATHER", "1") == "0":
            return False
        ok = x_local.is_cuda and global_batch == x_local.shape[0] * self.world_size and x_local.shape[0] > 0 \
            and dist.get_backend(self.group) == "nccl"
        return bool(ok and self._out_dim() % 8 == 0)             # 16-byte rows for the vector stores

    def _plan(self, x_local: torch.Tensor, global_batch: int) -> Optional[PeerGather]:
        """PeerGather to use for this (local batch, global batch, dtype), or None = torch.distributed.
        First use of a combination is a COLLECTIVE: one MIN and one MAX all-reduce over what every rank
        wants and holds (a rank that disagrees on the batch, width or dtype would otherwise store outside
        a peer's buffer or leave the others spinning in the kernel), then — if all agree on the kernel —
        the symmetric-memory rendezvous, whose success is agreed on the same way."""
        key = (x_local.shape[0], global_batch, x_local.dtype)
        if key in self._plans:
            return self._plans[key]
        want = self._local_want(x_local, global_batch)
        first = next(self.model.parameters(), None)
        out_dtype = first.dtype if first is not None else x_local.dtype
        mine = torch.tensor([int(want), x_local.shape[0], self._out_dim(), _DTYPE_CODES.get(out_dtype, 9), global_batch],
                            dtype=torch.int64, device=x_local.device)
        lo, hi = mine.clone(), mine.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=self.group)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=self.group)
        lo, hi = lo.tolist(), hi.tolist()
        assert lo[4] == hi[4], f"Ranks disagree on the global batch ({lo[4]} .. {hi[4]}): pass the same global_batch on every rank"
        assert lo[2] == hi[2] and lo[3] == hi[3], "Ranks disagree on the output width / dtype of the model"
        agreed = lo[0] == 1 and lo[1] == hi[1]
        peer = None
        if agreed:
            err = None
            try:
                peer = PeerGather(x_local.shape[0], self._out_dim(), out_dtype, x_local.device, self.group)
            except Exception as exc:   # symmetric memory unavailable (no P2P, old driver)
                err = exc
            ok = torch.tensor([0 if peer is None else 1], dtype=torch.int64, device=x_local.device)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=self.group)
            if int(ok.item()) == 0:
                if peer is None:
                    warnings.warn(f"peer-memory gather unavailable ({err!r}); all ranks use the torch.distributed all-gather")
                peer = None
        if self.peer_gather is True:
            assert peer is not None, "peer_gather=True needs CUDA inputs, an NCCL group, equal shards on every rank and symmetric memory"
        self._plans[key] = peer
        return peer
