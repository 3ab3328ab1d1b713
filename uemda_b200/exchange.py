"""Device-side exchange of the per-step statistics between the ranks of a sharded mining job (SURVEY.md section 8e).

One process per GPU; every rank owns a *symmetric region* (csrc/uem_exchange.cu for the layout) that all peers map into
their own address space.  A step's statistics -- prototype partial sums + counts (alignment.py:347-353), the class
histogram (balance.py:45-52) and the rank-local max superpixel id (alignment.py:241) -- are stored straight into every
peer's region by ``send`` (NVLink peer stores, every word paired with a sequence number), polled by ``wait_max_id`` and
folded in rank order by ``fold_finalize``; all three are plain kernel launches on the caller's stream, so a sharded step is captured in CUDA
graphs with no host-issued collective in between.  The pipelined form needs no extra launch at all: the id leaves from the
region-max kernel's tail (``mining.region_phase(..., exchange=(peer, slot, global_id_out))``) and the sums travel inside the
fold + EMA launch (``exchange_fold``).  The NCCL form (``ShardedMiner.exchange``: one all_gather) stays as the
fallback and as the reference the tests compare this one with.

Mapping the regions (tried in this order):
  1. ``torch.distributed._symmetric_memory`` (cuMem + fabric/fd handle exchange done by torch);
  2. cudaIpc handles from the library's own ``uem_peer_alloc`` / ``uem_peer_open``, shipped with ``all_gather_object``.
torch.distributed is plumbing here: rendezvous, barrier, handle exchange.
"""
import ctypes

import torch

from . import _lib as L
from . import ops

__all__ = ["PeerExchange", "ExchangeError"]


class ExchangeError(RuntimeError):
    pass


class PeerExchange:
    """Symmetric regions of all ranks + the three exchange launches.

    ``ptrs``: list of ``world`` ints, entry r = rank r's region as mapped in this process.  ``local_only(...)`` builds a
    world of regions on ONE device (every "rank" is driven by the same process: tests and the one-GPU emulation)."""

    def __init__(self, ptrs, rank, world, c, k, depth, device, keep=None, backend="?"):
        self.ptrs, self.rank, self.world, self.c, self.k, self.depth = [int(p) for p in ptrs], rank, world, c, k, depth
        self.device = device
        self.backend = backend
        self._keep = keep   # whatever owns the mappings
        self._arr = (ctypes.c_void_p * world)(*self.ptrs)

    # ------------------------------------------------------------------ construction
    @staticmethod
    def region_bytes(world, c, k, depth):
        n = L.load().uem_xchg_region_bytes(world, depth, c, k)
        if n < 0:
            raise ExchangeError("exchange region: world %d (<= 16), depth %d (<= 4), c %d, k %d out of range" % (world, depth, c, k))
        return int(n)

    @classmethod
    def create(cls, c, k, depth=3, group=None, device=None, backend="auto"):
        """Collective over ``group``: allocates, zeroes and maps the regions.  backend: 'auto' | 'symm_mem' | 'cuda_ipc'."""
        import torch.distributed as dist
        assert dist.is_initialized(), "PeerExchange.create needs an initialised torch.distributed job (one process per GPU)"
        device = device or torch.device("cuda", torch.cuda.current_device())
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        nbytes = cls.region_bytes(world, c, k, depth)
        errors = []
        ex = None
        if backend in ("auto", "symm_mem"):
            try:
                ex = cls._create_symm_mem(nbytes, c, k, depth, group, device, rank, world)
            except Exception as e:  # noqa: BLE001
                errors.append("symm_mem: %r" % (e,))
        # every rank must take the same branch: agree on the outcome
        if backend == "auto":
            ok = torch.tensor([1 if ex is not None else 0], device=device, dtype=torch.int32)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
            if int(ok.item()) == 0:
                ex = None
        if ex is None and backend in ("auto", "cuda_ipc"):
            try:
                ex = cls._create_cuda_ipc(nbytes, c, k, depth, group, device, rank, world)
            except Exception as e:  # noqa: BLE001
                errors.append("cuda_ipc: %r" % (e,))
        if ex is None:
            raise ExchangeError("could not map the exchange regions across ranks: " + "; ".join(errors))
        torch.cuda.synchronize(device)
        dist.barrier(group=group)   # nobody stores into a region before its owner has zeroed it
        return ex

    @classmethod
    def _create_symm_mem(cls, nbytes, c, k, depth, group, device, rank, world):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        pg = group if group is not None else dist.group.WORLD
        t = symm.empty(nbytes, dtype=torch.uint8, device=device)
        hdl = symm.rendezvous(t, pg.group_name)
        t.zero_()
        ptrs = [int(p) for p in hdl.buffer_ptrs]
        assert len(ptrs) == world and ptrs[rank] == t.data_ptr()
        return cls(ptrs, rank, world, c, k, depth, device, keep=(t, hdl), backend="symm_mem")

    @classmethod
    def _create_cuda_ipc(cls, nbytes, c, k, depth, group, device, rank, world):
        import torch.distributed as dist
        lib = L.load()
        L.check(lib.uem_set_device(device.index))
        local = ctypes.c_void_p()
        handle = (ctypes.c_ubyte * 64)()
        L.check(lib.uem_peer_alloc(nbytes, ctypes.byref(local), handle))
        handles = [None] * world
        dist.all_gather_object(handles, bytes(handle), group=group)
        ptrs = []
        for r in range(world):
            if r == rank:
                ptrs.append(local.value)
                continue
            p = ctypes.c_void_p()
            buf = (ctypes.c_ubyte * 64).from_buffer_copy(handles[r])
            L.check(lib.uem_peer_open(buf, ctypes.byref(p)))
            ptrs.append(p.value)
        return cls(ptrs, rank, world, c, k, depth, device, keep=("ipc", local.value), backend="cuda_ipc")

    @classmethod
    def local_only(cls, world, c, k, depth=3, device=None):
        """``world`` exchanges over regions that all live on ONE device (returns a list, entry r acts as rank r)."""
        device = device or torch.device("cuda", torch.cuda.current_device())
        nbytes = cls.region_bytes(world, c, k, depth)
        regions = [torch.zeros(nbytes, dtype=torch.uint8, device=device) for _ in range(world)]
        ptrs = [t.data_ptr() for t in regions]
        return [cls(ptrs, r, world, c, k, depth, device, keep=regions, backend="local") for r in range(world)]

    # ------------------------------------------------------------------ the three launches (capturable)
    def send(self, partials, max_id, slot, hist=None, global_id_out=None, part="all"):
        """partials: ``ops.proto_accumulate(..., fold=False)`` of this rank's source shard; max_id: (1,) int64 rank-local
        max superpixel id (or None); hist: (c+1,) int64 class histogram of this rank's labels (or None).
        global_id_out: optional (1,) int64 tensor; the launch then also polls the other ranks' ids of this step and leaves the
        batch-global max id there (= ``wait_max_id`` without its own launch).
        part: "all" | "id" (only the max id; ``partials`` may be None) | "sums" (everything else; ends the step's send)."""
        parts = {"all": 7, "id": 2, "sums": 5}[part]   # "id" early + "sums" later = one step sent in two launches
        ws, b = None, 1
        if parts & 1:
            ws, (b, c, k) = partials
            assert (c, k) == (self.c, self.k)
        anchor = ws if ws is not None else max_id
        L.require_cuda(ws, max_id, hist, global_id_out)
        lib = L.bind(anchor)
        L.check(lib.uem_xchg_send_f32(L.ptr(ws), b, self.c, self.k, L.ptr(max_id), L.ptr(hist), self._arr, self.rank, self.world,
                                      self.depth, int(slot), L.ptr(global_id_out), parts, L.stream_of(anchor)))

    def wait_max_id(self, slot, out=None):
        """Blocks the current stream until every rank's vector of ``slot`` has arrived -> batch-global max id (1,) int64."""
        if out is None:
            out = torch.empty(1, dtype=torch.int64, device=self.device)
        lib = L.bind(out)
        L.check(lib.uem_xchg_wait_maxid(ctypes.c_void_p(self.ptrs[self.rank]), self.world, self.depth, int(slot), self.c, self.k,
                                        L.ptr(out), L.stream_of(out)))
        return out

    def fold_finalize(self, slot, proto_old=None, eps=1e-7, decay=None, out=None, want_sums=False, want_hist=False):
        """After ``wait_max_id`` on the same stream: rank-ordered fold (+ keep-old rule + EMA when ``decay`` is given; ``out``
        may be ``proto_old``) and the acknowledgement of the slot.  Returns (proto_new|None, sums|None, counts|None, hist|None)."""
        proto_old, new, omd, d, sums, counts, hist = self._fold_outputs(proto_old, decay, out, want_sums, want_hist)
        lib = L.load()
        stream = ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        L.check(lib.uem_xchg_fold_finalize_ema_f32(self._arr, self.rank, self.world, self.depth, int(slot), self.c, self.k,
                                                   L.ptr(proto_old), ops.f32(eps), omd, d, L.ptr(new), L.ptr(sums), L.ptr(counts),
                                                   L.ptr(hist), stream))
        return new, sums, counts, hist

    def exchange_fold(self, partials, slot, proto_old=None, eps=1e-7, decay=None, out=None, hist=None, want_sums=False,
                      want_hist=False):
        """``send(part="sums")`` + ``fold_finalize`` in one launch (the step's max id must have been sent with part="id").
        Every rank's launch has to be able to run while the others' run: real ranks only, or a world of one."""
        ws, (b, c, k) = partials
        assert (c, k) == (self.c, self.k)
        L.require_cuda(ws, hist, proto_old)
        proto_old, new, omd, d, sums, counts, hist_out = self._fold_outputs(proto_old, decay, out, want_sums, want_hist)
        lib = L.bind(ws)
        L.check(lib.uem_xchg_exchange_fold_ema_f32(L.ptr(ws), b, c, k, L.ptr(hist), self._arr, self.rank, self.world, self.depth,
                                                   int(slot), L.ptr(proto_old), ops.f32(eps), omd, d, L.ptr(new), L.ptr(sums),
                                                   L.ptr(counts), L.ptr(hist_out), L.stream_of(ws)))
        return new, sums, counts, hist_out

    def _fold_outputs(self, proto_old, decay, out, want_sums, want_hist):
        """Arguments and outputs of a fold launch: (proto_old, proto_new, 1 - decay, decay, sums, counts, hist), each output
        None unless asked for (proto_new with ``decay``; it is ``out`` when given)."""
        dev = self.device
        new = sums = counts = hist = None
        omd = d = 0.0
        if decay is not None:
            proto_old = L.f32c(proto_old.detach())
            new = out if out is not None else torch.empty_like(proto_old)
            omd, d = ops.f32(1.0 - decay), ops.f32(decay)
        if want_sums:
            sums = torch.empty((self.c, self.k), dtype=torch.float32, device=dev)
            counts = torch.empty((self.c,), dtype=torch.int64, device=dev)
        if want_hist:
            hist = torch.empty((self.c + 1,), dtype=torch.int64, device=dev)
        return proto_old, new, omd, d, sums, counts, hist

    def status(self):
        """Synchronises the current stream; 0 = fine, bit 8 = a bounded poll timed out (2 s)."""
        out = ctypes.c_int(0)
        stream = ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        L.check(L.load().uem_xchg_status(ctypes.c_void_p(self.ptrs[self.rank]), ctypes.byref(out), stream))
        return int(out.value)

    def check(self):
        s = self.status()
        if s:
            raise ExchangeError("exchange status %d: a peer's vector / acknowledgement did not arrive within 2 s (a rank is gone, "
                                "or send / wait / fold are not issued in lockstep on every rank)" % s)
