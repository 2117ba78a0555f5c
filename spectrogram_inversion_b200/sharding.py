"""Multi-GPU drivers (one process per GPU, torch.distributed for the plumbing).

* Batch sharding (BASELINE.json configs 2-4): signals are independent on this path, so every rank runs the
  fused kernels on its own slice of the batch and NO collective touches the data path.  The only coupling in
  the reference is that the metric / early-stop test is evaluated over the whole batch
  (torch_specinv/methods.py:181-190): at evaluation iterations (where the host synchronises anyway) the two
  or three partial sums are all-reduced, so every rank takes the same decision the single-device run takes.
* Frame-range sharding of ONE long signal (config 5): see ``FrameShardedGriffinLim`` below.
"""
from __future__ import annotations

import os
from typing import List, Optional, Tuple

import torch
import torch.distributed as dist

from . import _ops
from .engine import ADMMSolver, GriffinLimSolver, METRIC_NAMES, StftPlan, training_loop


def shard_bounds(n: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous chunks of ceil(n / world) items (the last ranks may get fewer, or none)."""
    per = -(-n // world)
    lo = min(n, rank * per)
    return lo, min(n, lo + per)


def _all_reduce_floats(values: List[float], group, device: torch.device) -> List[float]:
    t = torch.tensor(values, dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t.tolist()


def make_sum_reducer(group=None, device: Optional[torch.device] = None):
    """``reduce_sums`` hook for ``training_loop``: sums (d, e) over the ranks of ``group``."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return None
    backend = dist.get_backend(group)
    dev = device if (backend == "nccl" and device is not None) else torch.device("cpu")

    def reduce(d: float, e: float):
        out = _all_reduce_floats([d, e], group, dev)
        return out[0], out[1]
    return reduce


def globalize_solver(solver, group=None) -> None:
    """Make ``solver.g`` and ``solver.n_bins_total`` those of the whole (sharded) batch."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return
    backend = dist.get_backend(group)
    dev = solver.plan.device if (backend == "nccl" and hasattr(solver, "plan")) else torch.device("cpu")
    g, n = _all_reduce_floats([solver.g, float(solver.n_bins_total)], group, dev)
    solver.g, solver.n_bins_total = g, int(round(n))


def _run_sharded(kind: str, spec_shard: torch.Tensor, max_iter, tol, coef, verbose, eva_iter, metric, group,
                 stft_kwargs):
    from . import methods
    assert eva_iter > 0 and max_iter > 0 and tol >= 0
    assert metric.upper() in METRIC_NAMES
    plan, C, mag = methods._setup(spec_shard, stft_kwargs)
    solver = GriffinLimSolver(plan, C, mag, coef) if kind == "gl" else ADMMSolver(plan, C, mag, coef)
    globalize_solver(solver, group)
    rank0 = (not dist.is_initialized()) or dist.get_rank(group) == 0
    training_loop(solver, max_iter, tol, verbose and rank0, eva_iter, metric,
                  reduce_sums=make_sum_reducer(group, plan.device))
    return methods._finish(solver.signal, spec_shard)


def griffin_lim_sharded(spec_shard, max_iter=200, tol=1e-6, alpha=0.99, verbose=True, eva_iter=10, metric="sc",
                        group=None, **stft_kwargs):
    """``griffin_lim`` on this rank's slice of a batch that is sharded over ``group``.  Same result as
    running the whole batch on one device: the evaluation sums are all-reduced so early stopping is decided
    on the whole batch like the reference does."""
    assert alpha >= 0
    return _run_sharded("gl", spec_shard, max_iter, tol, alpha, verbose, eva_iter, metric, group, stft_kwargs)


def ADMM_sharded(spec_shard, max_iter=1000, tol=1e-6, rho=0.1, verbose=1, eva_iter=10, metric="sc", group=None,
                 **stft_kwargs):
    return _run_sharded("admm", spec_shard, max_iter, tol, rho, verbose, eva_iter, metric, group, stft_kwargs)


# =================================================================================================
# Frame-range sharding of one (or a few) very long signal(s): BASELINE.json config 5
# =================================================================================================
class CudaRangeEngine:
    """The kernels a rank runs on ITS frame range [frame_offset, frame_offset + Tg) of the global signal.

    The range is described to the kernels as an un-centred local problem whose buffer holds the padded
    global samples [frame_offset*hop, (frame_offset+Tg-1)*hop + n_fft); its plan carries the GLOBAL envelope
    (``specinv_plan_init_ranged``), so what the fused kernel writes are this rank's partial overlap-add sums
    already divided by the global envelope -- partial sums of neighbouring ranks just add up."""

    def __init__(self, args, n_frames_local: int, batch: int, dtype, device, frame_offset: int, total_frames: int):
        self.args_global = args
        self.plan = StftPlan(args, n_frames_local, batch, dtype, device, frame_offset=frame_offset,
                             total_frames=total_frames)
        self.device, self.dtype = device, dtype
        self.local_len = self.plan.length
        self.pad = args.pad
        self.padded_offset = frame_offset * args.hop_length
        self.signal_len = args.signal_length(total_frames)

    # -- state -------------------------------------------------------------------------------------
    def pack(self, spec_local):
        return self.plan.pack(spec_local)

    def like(self, s):
        return s.like()

    def spec_abs(self, c):
        return self.plan.spec_abs(c)

    def phase_init(self, mag, phase_in):
        p, a = self.plan, self.args_global
        out = p.empty_spec()
        F = p.n_bins
        pin = phase_in if phase_in is not None else torch.empty(0, dtype=torch.float64, device=self.device)
        pout = torch.empty(p.B, F, dtype=torch.float64, device=self.device)
        _ops.phase_init_ex(mag.main, mag.nyq, out.main, out.nyq, pin, pout, a.n_fft, a.hop_length, a.onesided)
        return out, pout

    def mag_sum_sq(self, mag) -> float:
        from .engine import spec_sums
        return float(spec_sums(mag, mag)[2].item())

    def n_bins(self) -> int:
        return self.plan.B * self.plan.n_bins * self.plan.T

    # -- kernels -----------------------------------------------------------------------------------
    def empty_signal(self):
        return self.plan.empty_signal()

    def istft_partial(self, c, out):
        self.plan.istft(c, out)

    def gl_iter(self, x_in, x_out, q_in, q_out, mag, lr, sums):
        # straight through ctypes like the single-GPU solvers (engine._Solver._launch_direct): at 8 ranks an iteration
        # is ~0.2 ms of kernel time, a torch.library dispatch (~45 us) per launch would show
        p = self.plan
        ptrs = _ops.pointers((p.buf, x_in, x_out, q_in.main, q_in.nyq, q_out.main, q_out.nyq, mag.main, mag.nyq))
        _ops.iter_direct("gl_iter", "gl_iter", self.device, p.desc_ref, ptrs, lr,
                         sums.data_ptr() if sums is not None else None)

    def new_sums(self):
        return torch.zeros(2, dtype=torch.float64, device=self.device)

    def halo_sum(self, left, right, out):
        _ops.halo_sum(left, right, out)

    def fill_padding(self, x):
        _ops.fill_padding_direct(x, self.padded_offset, self.pad, self.signal_len, self.plan.pad_mode)


PEER_EXCHANGES = [0]      # halo exchanges done by the peer-memory kernel in this process (tests / bench look at it)


class PeerHalo:
    """NVLink peer-memory plumbing of the one-kernel halo exchange (csrc/specinv_p2p.cu): this rank's receive area
    (cudaMalloc + CUDA IPC handle), the mapped areas of its two neighbours, and the exchange counter.  The 64-byte
    handles travel through ``dist.all_gather_object``; nothing else uses the process group afterwards.

    ``PeerHalo.create`` is the collective constructor: every rank tries to set its side up and the ranks agree
    (all-reduce of an ok flag) whether ALL of them succeeded; otherwise everyone releases what it got and the caller
    falls back to the NCCL send/recv exchange -- no rank is left waiting on a peer that took the other path."""

    def __init__(self, rows: int, ov: int, dtype, device, group, rank: int, world: int):
        self.dtype, self.rows, self.ov, self.device, self.seq = dtype, rows, ov, device, 0
        self.area, self.peers = None, [None, None]
        self.error = None
        handle = bytes(64)
        try:
            with torch.cuda.device(device):
                self.area, handle = _ops.ipc_alloc_halo_area(dtype, rows, ov)
        except Exception as ex:            # keep going: the other ranks are waiting in the all_gather below
            self.error = ex
        infos = [None] * world
        dist.all_gather_object(infos, (handle, torch.cuda.current_device(), self.error is None), group=group)
        if self.error is None and not all(ok for _, _, ok in infos):
            self.error = RuntimeError("a peer rank could not allocate its halo area")
        if self.error is None:
            try:
                with torch.cuda.device(device):
                    me = torch.cuda.current_device()
                    for side, r in ((0, rank - 1), (1, rank + 1)):
                        if not 0 <= r < world:
                            continue
                        peer_dev = infos[r][1]
                        # (with one visible device per process both are device 0 and the question cannot be asked here:
                        # cudaIpcOpenMemHandle then decides)
                        if peer_dev != me and not torch.cuda.can_device_access_peer(me, peer_dev):
                            raise RuntimeError(f"cuda:{me} cannot access its neighbour cuda:{peer_dev} (no P2P)")
                        self.peers[side] = _ops.ipc_open(infos[r][0])
            except Exception as ex:
                self.error = ex

    @classmethod
    def create(cls, rows, ov, dtype, device, group, rank, world, comm_device):
        """Collective over ``group``: a working PeerHalo on every rank, or None on every rank."""
        ph = cls(rows, ov, dtype, device, group, rank, world)
        ok = torch.tensor([0.0 if ph.error is not None else 1.0], device=comm_device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)      # also the barrier: every mapping is in place
        if ok.item() == 1.0:
            return ph
        if ph.error is not None:
            import warnings
            warnings.warn(f"NVLink peer-memory halo exchange unavailable ({ph.error}); using NCCL send/recv")
        ph.close()
        return None

    def exchange(self, x: torch.Tensor) -> None:
        self.seq += 1
        PEER_EXCHANGES[0] += 1
        _ops.halo_exchange(x, self.rows, self.ov, self.area, self.peers[0], self.peers[1], self.seq)

    def check(self) -> None:
        """Raise when an exchange timed out waiting for a neighbour (synchronises the current stream; called where
        the host waits anyway: evaluations and the end of the run)."""
        if self.area is None:
            return
        status = _ops.halo_status(self.device, self.dtype, self.area, self.rows, self.ov)
        if status:
            raise RuntimeError(f"halo exchange {status} timed out waiting for a neighbouring rank "
                               "(SPECINV_P2P_TIMEOUT_MS); the result is incomplete")

    def close(self) -> None:
        if getattr(self, "area", None) is None and not any(bool(p) for p in getattr(self, "peers", [])):
            return
        torch.cuda.synchronize(self.device)
        _ops.ipc_release(self.peers, self.area)
        self.area, self.peers = None, [None, None]

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class FrameShardedGriffinLim:
    """Griffin-Lim on a signal whose FRAMES are sharded over the ranks of ``group`` (rank order = time order).

    Per iteration every rank runs the fused kernel on its own frames and then exchanges, with each neighbour,
    the partial overlap-add sums of the (n_fft - hop) samples they share (12 KiB for n_fft=4096, hop=1024):
    both sides add "left partial + right partial" in that order, so they hold bit-identical samples and the
    next iteration's STFT sees the same signal a single device would.  The exchange is a pairwise
    send/recv (NCCL over NVLink on GPUs); the metric sums are all-reduced at evaluation iterations only."""

    def __init__(self, engine, C_local, mag_local, alpha: float, group=None):
        self.e, self.group = engine, group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        a = engine.args_global
        self.ov = a.n_fft - a.hop_length
        assert engine.local_len >= 2 * self.ov, "every rank needs at least ceil(n_fft/hop) frames"
        if a.center and a.pad_mode == "reflect" and self.rank in (0, self.world - 1):
            # the reflect sources of an edge rank's padding must live in its own buffer (specinv_fill_padding would
            # otherwise have to leave stale padding behind): 2 * pad + 1 samples, i.e. at least two frames
            assert engine.local_len >= 2 * a.pad + 1, "the first / last rank needs at least 2 frames with reflect padding"
        self.lr = alpha / (1 + alpha)
        self.mag = mag_local
        self.q = [C_local, engine.like(C_local)]
        self.x = [engine.empty_signal(), engine.empty_signal()]
        self.cur = 0
        self.sums = engine.new_sums()
        self.g = engine.mag_sum_sq(mag_local)
        self.n_bins_total = engine.n_bins()
        self.plan = getattr(engine, "plan", None)
        if self.world > 1:
            red = _all_reduce_floats([self.g, float(self.n_bins_total)], group, self._comm_device())
            self.g, self.n_bins_total = red[0], int(round(red[1]))
        # NCCL ranks on their own GPUs: the exchange is ONE kernel over NVLink peer memory (SPECINV_P2P=0 keeps the
        # NCCL send/recv path); gloo groups / ranks sharing a GPU use the host-staged path below, unless
        # SPECINV_P2P=force asks for the peer-memory kernel there too (CUDA IPC also maps another process's buffer on
        # the SAME device: how a single-GPU box exercises the kernel, tests/test_gpu_sharding.py)
        self.peer = None
        mode = os.environ.get("SPECINV_P2P", "1")
        if (self.world > 1 and self.x[0].is_cuda and mode != "0"
                and (dist.get_backend(group) == "nccl" or mode == "force")):
            self.peer = PeerHalo.create(self.x[0].shape[0], self.ov, self.x[0].dtype, self.x[0].device, group,
                                        self.rank, self.world, self._comm_device())
        engine.istft_partial(C_local, self.x[0])                  # x_0 = ISTFT(C)  (methods.py:233)
        self._exchange(self.x[0])
        self.iterations = 0

    def _comm_device(self):
        if self.world > 1 and dist.get_backend(self.group) != "nccl":
            return torch.device("cpu")
        return self.x[0].device

    def _exchange(self, x):
        """combine the partial sums of the regions shared with the left / right neighbour, restore padding"""
        if self.peer is not None:
            self.peer.exchange(x)
            self.e.fill_padding(x)
            return
        ov, Lg = self.ov, x.shape[1]
        left = self.rank - 1 if self.rank > 0 else None
        right = self.rank + 1 if self.rank < self.world - 1 else None
        # NCCL moves device buffers directly (NVLink P2P); a gloo group (CPU tests, or several ranks sharing one
        # GPU) is fed through host staging buffers
        stage = x.is_cuda and self.world > 1 and dist.get_backend(self.group) != "nccl"
        ops, recv_l, recv_r = [], None, None
        if right is not None:
            tail = x[:, Lg - ov:].contiguous()
            tail = tail.cpu() if stage else tail
            recv_r = torch.empty_like(tail)
            ops += [dist.P2POp(dist.isend, tail, right, self.group), dist.P2POp(dist.irecv, recv_r, right, self.group)]
        if left is not None:
            head = x[:, :ov].contiguous()
            head = head.cpu() if stage else head
            recv_l = torch.empty_like(head)
            ops += [dist.P2POp(dist.isend, head, left, self.group), dist.P2POp(dist.irecv, recv_l, left, self.group)]
        if ops:
            for req in dist.batch_isend_irecv(ops):
                req.wait()
        if stage:
            recv_l = recv_l.to(x.device) if recv_l is not None else None
            recv_r = recv_r.to(x.device) if recv_r is not None else None
        if left is not None:
            self.e.halo_sum(recv_l, x[:, :ov], x[:, :ov])             # left partial + right partial
        if right is not None:
            self.e.halo_sum(x[:, Lg - ov:], recv_r, x[:, Lg - ov:])   # same order on the other side
        self.e.fill_padding(x)

    def step(self, evaluate: bool = False):
        i, o = self.cur, self.cur ^ 1
        if evaluate:
            self.sums.zero_()
        self.e.gl_iter(self.x[i], self.x[o], self.q[i], self.q[o], self.mag, self.lr, self.sums if evaluate else None)
        self._exchange(self.x[o])
        self.cur = o
        self.iterations += 1
        if evaluate:
            d, e = self.sums.tolist()
            if self.peer is not None:
                self.peer.check()
            return d, e
        return None

    @property
    def signal_local(self):
        return self.x[self.cur]

    def owned_piece(self):
        """(start index in the global unpadded signal, tensor) of the samples this rank owns."""
        if self.peer is not None:
            self.peer.check()
        a, e = self.e.args_global, self.e
        hop, P, L = a.hop_length, a.pad, e.signal_len
        off = e.padded_offset
        lo = off if self.rank > 0 else 0
        hi = off + e.plan.T * hop if self.rank < self.world - 1 else off + e.local_len
        lo, hi = max(lo, P), min(hi, P + L)
        return lo - P, self.x[self.cur][:, lo - off:hi - off]


def griffin_lim_frame_sharded(spec_local, max_iter=200, tol=1e-6, alpha=0.99, verbose=True, eva_iter=10, metric="sc",
                              group=None, gather=True, engine_factory=None, **stft_kwargs):
    """``griffin_lim`` for a signal too long for (or faster on more than) one GPU: every rank passes the
    spectrogram frames it owns, ``spec_local`` of shape (F, Tg) / (B, F, Tg) in rank = time order; returns the
    whole signal on every rank (``gather=True``) or ``(start, piece)``.

    A real ``spec_local`` gets its start from the (sequential-in-time) phase_init: ranks run it once to get
    their phase advance, exchange those (an exclusive scan over ranks) and run it again with the right start."""
    from .stft_args import args_helper, real_dtype_of
    from .engine import compute_device
    assert alpha >= 0 and eva_iter > 0 and max_iter > 0 and tol >= 0
    assert metric.upper() in METRIC_NAMES
    assert 4 > spec_local.dim() > 1
    squeeze = spec_local.dim() == 2
    work = spec_local.detach()
    if squeeze:
        work = work.unsqueeze(0)
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    args = args_helper(work, **stft_kwargs)
    if args.center and args.pad_mode == "circular" and world > 1:
        raise NotImplementedError("circular padding wraps around the whole signal: not supported when frame-sharded")
    B, _, Tg = work.shape
    counts = [Tg]
    if world > 1:
        counts = [None] * world
        dist.all_gather_object(counts, Tg, group=group)
    offset, total = sum(counts[:rank]), sum(counts)
    if engine_factory is None:
        dev = compute_device(work)
        work = work.to(dev)
        engine = CudaRangeEngine(args, Tg, B, real_dtype_of(work.dtype), dev, offset, total)
    else:
        engine = engine_factory(args, Tg, B, real_dtype_of(work.dtype), offset, total)
    if work.is_complex():
        C = engine.pack(work)
        mag = engine.spec_abs(C)
    else:
        mag = engine.pack(work)
        C, adv = engine.phase_init(mag, None)
        if world > 1:
            host = adv.is_cuda and dist.get_backend(group) != "nccl"
            adv_c = adv.cpu() if host else adv
            advs = [torch.empty_like(adv_c) for _ in range(world)]
            dist.all_gather(advs, adv_c, group=group)
            start = torch.zeros_like(adv_c)
            for r in range(rank):
                start += advs[r]
            if rank > 0:
                C, _ = engine.phase_init(mag, start.to(adv.device))
    solver = FrameShardedGriffinLim(engine, C, mag, alpha, group)
    reducer = None
    if world > 1:
        dev = solver._comm_device()

        def reducer(d, e):
            out = _all_reduce_floats([d, e], group, dev)
            return out[0], out[1]
    training_loop(solver, max_iter, tol, verbose and rank == 0, eva_iter, metric, reduce_sums=reducer)
    start, piece = solver.owned_piece()
    if not gather:
        return start, (piece[0] if squeeze else piece)
    if world > 1:
        lens = [None] * world
        dist.all_gather_object(lens, (start, piece.shape[1]), group=group)
        width = max(n for _, n in lens)
        host = piece.is_cuda and dist.get_backend(group) != "nccl"
        padded = torch.zeros(piece.shape[0], width, dtype=piece.dtype, device="cpu" if host else piece.device)
        padded[:, :piece.shape[1]] = piece
        parts = [torch.empty_like(padded) for _ in range(world)]
        dist.all_gather(parts, padded, group=group)
        full = torch.cat([p[:, :n] for p, (_, n) in zip(parts, lens)], dim=1).to(piece.device)
    else:
        full = piece.clone()
    full = full[0] if squeeze else full
    return full.to(spec_local.device) if not spec_local.is_cuda and full.is_cuda else full
