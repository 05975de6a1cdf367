"""Time-sharded MultUpdate fit: one process per GPU, host-side collectives between the
split-phase steps of libcmf_sm100 (include/cmf_sm100.h, "split-phase steps").

The reference is single-process (SURVEY.md section 2.1), so there is no reference counterpart;
the scheme is SURVEY.md section 8e: rank r owns columns [t_r, t_{r+1}) of X and H, W is replicated,
X carries a static right halo of L-1 columns, H carries left and right halos of L-1 columns that
are re-exchanged after every H update, and the W-side partials (numW and the H cross-correlation
that yields denomW) are all-reduced.  Every rank then applies the identical W update, so no
broadcast is needed.

The step logic (`ShardedMultFit`) is engine-agnostic: the product engine is `DeviceShard`
(CUDA library, NCCL tensors); tests/ drive the same logic over gloo with a NumPy engine to check
the partition / halo / all-reduce algebra on the CPU.
"""
from __future__ import annotations

import ctypes
import math

from . import _lib
from ._lib import HALS, MULT, Handle, check, parse_dtype
from .model import _alternate, _rescale


class ShardPlan:
    """Balanced contiguous partition of the time axis; every shard needs >= max(L-1, 1) columns."""

    def __init__(self, T, world, L):
        if world < 1 or T < 1:
            raise ValueError("need T >= 1 and world >= 1")
        base, rem = divmod(T, world)
        self.T, self.world, self.L = T, world, L
        self.ranges = []
        t = 0
        for r in range(world):
            n = base + (1 if r < rem else 0)
            self.ranges.append((t, t + n))
            t += n
        if world > 1 and min(b - a for a, b in self.ranges) < max(L - 1, 1):
            raise ValueError(f"T={T} is too short to shard {world} ways with L={L}: "
                             "every shard needs at least L-1 columns")

    def owner(self, t):
        for r, (a, b) in enumerate(self.ranges):
            if a <= t < b:
                return r
        raise IndexError(t)


class _CudaView:
    """Exposes a raw device pointer through __cuda_array_interface__ so torch can alias it."""

    def __init__(self, ptr, count, typestr):
        self.__cuda_array_interface__ = {
            "shape": (int(count),), "typestr": typestr, "data": (int(ptr), False), "version": 2,
            "strides": None,
        }


class DeviceShard(Handle):
    """One rank's shard on one GPU: a libcmf_sm100 handle plus torch views of its exchange buffers."""

    def __init__(self, N, T, t0, t1, K, L, dtype="f32", device=0, use_torch_stream=True, alg="mult", comm=None,
                 ngpu=None, devices=None):
        """``comm=(unique_id_bytes, rank, world)``: the handle of one rank with the NCCL communicator INSIDE the library
        (cmf_create_rank; t0/t1 must be the balanced shard of that rank).  ``ngpu=n``: one group handle driving n GPUs
        from this process (cmf_create_multi; t0/t1 = 0/T).  Neither: a plain (shard) handle whose collectives the host does."""
        import torch

        self.torch = torch
        self.device = device
        self.group = bool(ngpu and ngpu > 1)
        self.in_library_comm = comm is not None or self.group
        super().__init__(N, T, K, L, parse_dtype(dtype), {"mult": MULT, "hals": HALS}[alg], device, t0, t1, comm=comm,
                         ngpu=ngpu, devices=devices)
        if use_torch_stream and not self.group:
            with torch.cuda.device(device):
                s = torch.cuda.current_stream().cuda_stream
            check(_lib.load().cmf_set_stream(self._h, ctypes.c_void_p(s)))
        if not self.group:
            self._views()

    @staticmethod
    def unique_id():
        """128-byte NCCL id for cmf_create_rank (rank 0 creates it, the host hands it to the other ranks)."""
        buf = ctypes.create_string_buffer(128)
        check(_lib.load().cmf_comm_unique_id(buf))
        return bytes(buf.raw)

    def exchange_halos(self):
        check(_lib.load().cmf_exchange_halos(self._h))

    def _views(self):
        torch, lib = self.torch, _lib.load()
        dev = f"cuda:{self.device}"
        ts = {_lib.F64: "<f8", _lib.F32: "<f4"}
        self.exchange = []
        for which in (0, 1, 2, 3):
            p, n, dt = ctypes.c_void_p(), ctypes.c_int64(), ctypes.c_int()
            check(lib.cmf_exchange_buffer(self._h, which, ctypes.byref(p), ctypes.byref(n), ctypes.byref(dt)))
            self.exchange.append(torch.as_tensor(_CudaView(p.value, n.value, ts[dt.value]), device=dev))
        ps = [ctypes.c_void_p() for _ in range(4)]
        n = ctypes.c_int64()
        check(lib.cmf_halo_buffers(self._h, *[ctypes.byref(p) for p in ps], ctypes.byref(n)))
        if n.value > 0:
            v = [torch.as_tensor(_CudaView(p.value, n.value, ts[self.dtype]), device=dev) for p in ps]
        else:
            v = [torch.empty(0, device=dev)] * 4
        self.send_left, self.send_right, self.recv_left, self.recv_right = v

    def scalar_tensor(self, values):
        return self.torch.tensor(values, dtype=self.torch.float64, device=f"cuda:{self.device}")

    # split-phase steps -------------------------------------------------------------------------
    def w_partials(self):
        check(_lib.load().cmf_w_partials(self._h))

    def w_apply(self, l1W, l2W):
        check(_lib.load().cmf_w_apply(self._h, float(l1W), float(l2W)))

    def h_update(self, l1H, l2H):
        check(_lib.load().cmf_h_update(self._h, float(l1H), float(l2H)))

    def loss_partial(self):
        out = ctypes.c_double()
        check(_lib.load().cmf_loss_partial(self._h, ctypes.byref(out)))
        return out.value


class _AlternatingFit:
    """The fit loop shared by ShardedMultFit and LibraryFit, over their ``loss`` and ``iterate``."""

    def fit(self, max_itr=100, check_convergence=True, patience=3, tol=1e-4, **reg):
        """src/algs/alternating.jl:16-71 over shards (every rank takes the same branch because the
        loss is all-reduced)."""
        loss_hist, _, _ = _alternate(self.loss(), lambda: self.iterate(**reg), max_itr, check_convergence=check_convergence,
                                     patience=patience, tol=tol)
        return loss_hist


class ShardedMultFit(_AlternatingFit):
    """The sharded MU iteration (src/algs/mult.jl:23-58 split at its three global dependencies).

    ``shard`` is any engine with the DeviceShard step interface; ``dist`` is torch.distributed
    (initialised by the caller; NCCL on GPUs, gloo in the CPU tests) or None for world == 1."""

    def __init__(self, shard, rank=0, world=1, dist=None):
        self.shard, self.rank, self.world, self.dist = shard, rank, world, dist
        if world > 1 and dist is None:
            raise ValueError("world > 1 needs an initialised torch.distributed module")

    # collectives -------------------------------------------------------------------------------
    def _allreduce(self, tensor):
        if self.world > 1:
            self.dist.all_reduce(tensor)

    def _allreduce_scalars(self, values):
        if self.world == 1:
            return list(values)
        t = self.shard.scalar_tensor(list(values))
        self.dist.all_reduce(t)
        return [float(v) for v in t.tolist()]

    def exchange_halos(self):
        """Left neighbour's recv_right <- my first L-1 columns; right neighbour's recv_left <- my last L-1."""
        if self.world == 1 or self.shard.L <= 1:
            return
        d, s, ops = self.dist, self.shard, []
        if self.rank + 1 < self.world:
            ops.append(d.P2POp(d.isend, s.send_right, self.rank + 1))
            ops.append(d.P2POp(d.irecv, s.recv_right, self.rank + 1))
        if self.rank > 0:
            ops.append(d.P2POp(d.isend, s.send_left, self.rank - 1))
            ops.append(d.P2POp(d.irecv, s.recv_left, self.rank - 1))
        for req in d.batch_isend_irecv(ops):
            req.wait()

    # setup -------------------------------------------------------------------------------------
    def setup_data_norm(self):
        """data_norm = ||X||_F over all shards (mult.jl:13)."""
        (ss,) = self._allreduce_scalars([self.shard.data_sumsq()])
        self.data_norm = math.sqrt(ss)
        self.shard.set_data_norm(self.data_norm)
        return self.data_norm

    def rescale_init(self):
        """The alpha rescale of init_rand (src/model.jl:119-122) with global reductions."""
        dot, nrm2 = self._allreduce_scalars(self.shard.init_scale_partials())
        s = math.sqrt(abs(dot / nrm2))
        self.shard.scale_factors(s)
        return s

    def loss(self):
        (ss,) = self._allreduce_scalars([self.shard.loss_partial()])
        return math.sqrt(ss) / self.data_norm

    # one iteration -----------------------------------------------------------------------------
    def iterate(self, l1W=0.0, l2W=0.0, l1H=0.0, l2H=0.0, eval_mode=False):
        s = self.shard
        if not eval_mode:
            s.w_partials()                       # local numW + Gram partials
            self._allreduce(s.exchange[0])       # numW            (K*N*L)
            self._allreduce(s.exchange[1])       # Gram + H tail   (K*K*L + (L-1)*K doubles)
            s.w_apply(l1W, l2W)                  # identical W update on every rank
        s.h_update(l1H, l2H)                     # owned columns of H
        self.exchange_halos()                    # L-1 columns each way
        loss = self.loss()                       # all-reduce of one double
        if getattr(s, "loss_mode", 0) == 1 and not loss > 0.25:
            s.set_loss_mode(0)                   # the expansion cancels like 1/loss^2 (same rule on every rank)
            loss = self.loss()                   # re-evaluate with the direct pass, as the library's own loop does
        return loss


class LibraryFit(_AlternatingFit):
    """The same fit steps as ``ShardedMultFit`` with every collective INSIDE libcmf_sm100 (NCCL bound by the library:
    ``DeviceShard(comm=...)`` under torchrun, or ``DeviceShard(ngpu=...)`` in one process).  The host only calls the
    reference-facing entry points: update_motifs! / update_feature_maps! / compute_loss (alternating.jl:37,52,54)."""

    def __init__(self, shard):
        self.shard = shard

    def setup_data_norm(self):
        self.data_norm = math.sqrt(self.shard.data_sumsq())       # all-reduced by cmf_set_data / cmf_synth_data
        return self.data_norm

    def rescale_init(self):
        return _rescale(self.shard)                               # the partials are all-reduced by the library

    def exchange_halos(self):
        self.shard.exchange_halos()

    def loss(self):
        return self.shard.loss()

    def iterate(self, l1W=0.0, l2W=0.0, l1H=0.0, l2H=0.0, eval_mode=False):
        if not eval_mode:
            self.shard.update_motifs(l1W, l2W)
        return self.shard.update_feature_maps(l1H, l2H)
