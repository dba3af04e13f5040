"""Start-node sharding over the GPUs of one box, and the one collective of the path.

Walks from different start nodes are independent, so GPU g owns a contiguous block of
start nodes = rows of every M_l (the reference shards the same way over processes,
sparse_sampler.py:90; same ``np.array_split`` boundaries).  The CSR walk graph is
replicated; building Phi needs no communication.  The kernel matvec needs exactly one
exchange: the sum over GPUs of the partials ``U_g = Phi_g[x2]^T V_g`` (N x t), done as an
all-reduce over NCCL/NVLink (gloo on CPU in the tests).
"""

from __future__ import annotations

from typing import Callable, Optional, Sequence, Tuple

import numpy as np
import os

import torch


def shard_bounds(n_nodes: int, world_size: int) -> np.ndarray:
    """Row boundaries [b_0 = 0, ..., b_world = n]; shard g owns [b_g, b_g+1).  Same split as
    ``np.array_split(np.arange(n), world)`` (the first n % world shards get one extra row)."""
    base, extra = divmod(int(n_nodes), int(world_size))
    sizes = np.full(world_size, base, dtype=np.int64)
    sizes[:extra] += 1
    return np.concatenate([[0], np.cumsum(sizes)])


def my_rows(n_nodes: int, world_size: int, rank: int) -> Tuple[int, int]:
    b = shard_bounds(n_nodes, world_size)
    return int(b[rank]), int(b[rank + 1])


def owner_of(ids: torch.Tensor, n_nodes: int, world_size: int) -> torch.Tensor:
    """Rank owning each global row id."""
    bounds = torch.as_tensor(shard_bounds(n_nodes, world_size)[1:], device=ids.device)
    return torch.bucketize(ids.to(torch.int64), bounds, right=True)


def sharded_kernel_matvec(apply_t: Callable, apply: Callable, v_local: torch.Tensor, group=None) -> torch.Tensor:
    """out_g = Phi_g (sum_h Phi_h^T V_h): ``apply_t(v_local) -> U_g [N, t]``, all-reduce, ``apply(U) -> out_g``.

    The two callables are this rank's halves of the product (PhiBlocks.apply_t / apply on a
    GPU; anything with the same contract in the CPU tests)."""
    import torch.distributed as dist

    u = apply_t(v_local).contiguous()
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(u, group=group)
    return apply(u)


def sharded_dot(a: torch.Tensor, b: torch.Tensor, group=None) -> torch.Tensor:
    """Column-wise dot products of row-sharded [n_g, t] blocks (the t-float all-reduce of a
    row-sharded CG iteration)."""
    import torch.distributed as dist

    d = (a * b).sum(dim=0)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(d, group=group)
    return d


def shared_columns(touched: torch.Tensor, group=None, max_fraction: float = 0.5) -> Optional[torch.Tensor]:
    """Columns of Phi touched by at least two row shards (same result on every rank), or None when
    they are more than ``max_fraction`` of all columns (then a plain all-reduce of U is cheaper).

    ``touched``: bool / int [N], this shard's non-empty columns.  A column touched by ONE shard needs
    no communication at all: its sum is that shard's partial, and only that shard reads it in the
    second half of the product.  For a banded Phi the shared columns are just the bands around the
    shard boundaries, so the exchange shrinks from N x t to O(bandwidth x t)."""
    import torch.distributed as dist

    count = touched.to(torch.int32).clone()
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(count, group=group)
    else:
        return torch.zeros(0, dtype=torch.int64, device=touched.device)
    shared = torch.nonzero(count >= 2).flatten()
    if shared.numel() > max_fraction * touched.numel():
        return None
    return shared


def reduce_shared(u: torch.Tensor, shared: Optional[torch.Tensor], buf: Optional[torch.Tensor] = None, group=None):
    """Sum the per-shard partials ``u`` [N, ld] over the ranks, exchanging only the shared columns."""
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1):
        return u
    if shared is None:
        dist.all_reduce(u, group=group)
        return u
    if shared.numel() == 0:
        return u
    if buf is None:
        buf = torch.empty((shared.numel(), u.shape[1]), dtype=u.dtype, device=u.device)
    torch.index_select(u, 0, shared, out=buf)
    dist.all_reduce(buf, group=group)
    u.index_copy_(0, shared, buf)
    return u


def sharded_cg(matmul_closure: Callable, rhs_local: torch.Tensor, tolerance: float = 1e-2, max_iter: int = 1000,
               eps: float = 1e-10, check_every: int = 4, group=None, return_info: bool = False):
    """``cg.linear_cg`` on a row-sharded system: ``rhs_local`` / the solution hold this rank's rows,
    ``matmul_closure`` is the sharded product (its exchange inside), and every dot product is summed over the
    ranks (a t-float all-reduce).  Same normalisation and stopping rule as the single-GPU solver."""
    squeeze = rhs_local.dim() == 1
    b = (rhs_local[:, None] if squeeze else rhs_local).to(torch.float32)
    norm = sharded_dot(b, b, group).sqrt()[None, :]
    norm = torch.where(norm < eps, torch.ones_like(norm), norm)
    b = b / norm
    x = torch.zeros_like(b)
    r = b.clone()
    d = r.clone()
    rs = sharded_dot(r, r, group)[None, :]
    min_iter = min(10, max_iter - 1)
    iters = 0
    for k in range(max_iter):
        ad = matmul_closure(d)
        alpha = rs / sharded_dot(d, ad, group)[None, :].clamp_min(eps)
        x = x + alpha * d
        r = r - alpha * ad
        rs_new = sharded_dot(r, r, group)[None, :]
        iters = k + 1
        if iters >= min_iter and (iters % check_every == 0 or iters == max_iter):
            if float(rs_new.sqrt().mean()) < tolerance:
                break
        d = r + (rs_new / rs.clamp_min(eps)) * d
        rs = rs_new
    out = x * norm
    out = out[:, 0] if squeeze else out
    return (out, {"iterations": iters}) if return_info else out


def pilot_row_cost(graph, cfg, pilot_walks: int = 25, walk_share: float = 0.38) -> torch.Tensor:
    """Per-start-node cost estimate for ``balanced_bounds``: a cheap pilot Phi (``pilot_walks`` walks per node, a
    quarter of a real walk, no transposition) tells how many entries a row produces -- on a power-law graph a start node in the hub
    region fills three times the entries of one in the tail, and everything after the walker (compaction,
    transposition, both halves of the product) scales with entries, not with walks.  Cost = ``walk_share`` x the
    node's share of the walks + the rest x its share of the pilot entries (config 4, one GPU: walker 17.9 ms of
    47 ms).  Same draws on every rank, so every rank computes the same bounds.  The pilot samples neighbours as
    ``cfg`` does: weighted draws reach other rows than uniform ones, so the balance follows the Phi that is built."""
    from . import engine

    pilot = engine.WalkConfig(int(pilot_walks), cfg.p_halt, cfg.max_walk_length, seed=cfg.seed,
                              neighbour_sampling=getattr(cfg, "neighbour_sampling", "uniform"))
    phi = engine.build_phi_blocks(graph, pilot, transpose=False)
    L = phi.n_steps
    ptr = phi.blk_ptr
    nnz = (ptr[L::L] - ptr[:-1:L]).to(torch.float64)
    deg = graph.row_ptr[1:] - graph.row_ptr[:-1]
    walks = torch.where(deg > 0, 1.0, 0.15).to(torch.float64)
    return walk_share * walks / walks.sum() + (1.0 - walk_share) * nnz / nnz.sum()


def balanced_bounds(graph, world_size: int, isolated_weight: float = 0.15, row_cost=None) -> list:
    """Contiguous start-node ranges of equal estimated work (strong scaling of one graph over the GPUs).
    ``row_cost`` (float64 [n_nodes], e.g. ``pilot_row_cost``) replaces the degree-only estimate below.

    Equal COUNTS (``shard_bounds``, what the reference's ``np.array_split`` does) are badly unbalanced on a
    power-law graph whose hubs sit at low ids (R-MAT: the first eighth of the ids holds 44 % of the edge
    endpoints and the last eighth 1.4 %; 42 % of the nodes are isolated).  A start node with neighbours costs
    W halting walks and ~W * S(L) merged records; an isolated one stops at length 0 -- ``isolated_weight`` of
    that.  The boundaries are the equal-weight quantiles of that estimate, computed on the device."""
    n = graph.n_nodes
    if world_size <= 1:
        return [0, n]
    if row_cost is not None:
        w = row_cost.to(torch.float64)
    else:
        deg = graph.row_ptr[1:] - graph.row_ptr[:-1]
        w = torch.where(deg > 0, 1.0, float(isolated_weight)).to(torch.float64)
    cum = torch.cumsum(w, 0)
    targets = cum[-1] * torch.arange(1, world_size, device=cum.device, dtype=torch.float64) / world_size
    cuts = torch.searchsorted(cum, targets).cpu().tolist()
    bounds = [0] + [int(min(max(c, 0), n)) for c in cuts] + [n]
    for i in range(1, len(bounds)):
        bounds[i] = max(bounds[i], bounds[i - 1])
    return bounds


class Exchange:
    """U = sum over the ranks of the partials Phi_g^T V_g, between the two halves of a sharded product.

    ``peer``: every rank's U sits in torch symmetric memory (mapped into every process of the box) and
    ``grf_exchange_sum`` -- one kernel per rank over NVLink peer loads / stores -- leaves the rank-ordered sum
    in all copies.  ``nccl``: a plain all-reduce of a private buffer (also the gloo path of the CPU tests).
    Build it once per (N, leading dimension) and hand it to ``PhiBlocks.plan(..., exchange=...)``: the plan
    then writes its partial straight into ``exchange.u``."""

    def __init__(self, n_cols: int, ld: int, device, group=None, mode: str = "auto"):
        import torch.distributed as dist

        self.group = None if group in (None, True) else group
        self.world = dist.get_world_size(self.group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(self.group) if dist.is_initialized() else 0
        self.n_cols, self.ld, self.device = int(n_cols), int(ld), torch.device(device)
        self.mode, self.epoch, self.why = "nccl", 0, ""
        self.u = None
        if mode in ("auto", "peer") and self.world > 1 and self.device.type == "cuda":
            try:
                self._init_peer()
                self.mode = "peer"
            except Exception as exc:      # no symmetric memory on this box / build: all-reduce instead
                if mode == "peer":
                    raise
                self.why = f"{type(exc).__name__}: {exc}"[:200]
        if self.u is None:
            self.u = torch.empty((max(1, self.n_cols), self.ld), dtype=torch.float32, device=self.device)

    def _init_peer(self):
        import ctypes

        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm

        from . import _lib

        if self.world > 8:
            raise RuntimeError("grf_exchange_sum is built for 2..8 GPUs of one box")
        pg = dist.group.WORLD if self.group is None else self.group
        n_flag = _lib.lib().grf_exchange_flag_bytes(self.world) // 4
        self._u_sym = symm.empty((max(1, self.n_cols), self.ld), dtype=torch.float32, device=self.device)
        self._f_sym = symm.empty((n_flag,), dtype=torch.int32, device=self.device)
        self._f_sym.zero_()
        hu = symm.rendezvous(self._u_sym, pg)
        hf = symm.rendezvous(self._f_sym, pg)
        torch.cuda.synchronize(self.device)
        hf.barrier()                                   # every rank's flags are zero before anyone signals
        self._handles = (hu, hf)
        vp = ctypes.c_void_p
        self._pu = (vp * self.world)(*[vp(int(p)) for p in hu.buffer_ptrs])
        self._pf = (vp * self.world)(*[vp(int(p)) for p in hf.buffer_ptrs])
        self.u = self._u_sym
        # NVSwitch multicast address of U (0 / absent: no NVLS on this box or build): the sum then runs inside
        # the switch -- grf_exchange_sum_nvls -- instead of over (G-1) peer loads per vector
        self._mc = None
        want = os.environ.get("GRF_EXCHANGE_NVLS", "auto")          # "0": never, "1": whenever available, auto: measure
        if want != "0":
            try:
                mc = int(getattr(hu, "multicast_ptr", 0) or 0)
                self._mc = mc if mc else None
            except Exception:
                self._mc = None
        self.tuned = None
        if self._mc and want == "auto":
            self._pick_path(pg)

    def _pick_path(self, pg) -> None:
        """Both paths move the same bytes per link and direction ((G-1)/G of U out for the switch's loads or the
        peer loads, the same in for the multicast or the peer stores); which one is faster depends on the GPU
        count (2 GPUs: peer loads 0.42 ms, in-switch sums 0.71 ms for 268 MB).  Measured once per Exchange on a
        zeroed U, the slower rank decides, every rank takes the same path."""
        import torch.distributed as dist

        mc, times = self._mc, []
        self.u.zero_()
        for use in (None, mc):
            self._mc = use
            for _ in range(2):
                self.reduce()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(torch.cuda.current_stream(self.device))
            for _ in range(5):
                self.reduce()
            b.record(torch.cuda.current_stream(self.device))
            b.synchronize()
            t = torch.tensor([a.elapsed_time(b) / 5], dtype=torch.float64, device=self.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=pg)
            times.append(float(t))
        self._mc = mc if times[1] < 0.95 * times[0] else None
        self.tuned = {"peer_ms": times[0], "nvls_ms": times[1]}

    def describe(self) -> str:
        if self.mode == "peer" and getattr(self, "_mc", None):
            return (f"grf_exchange_sum_nvls: one kernel per rank, sums inside the NVSwitch (multimem.ld_reduce / "
                    f"multimem.st on the multicast address of torch symmetric memory), {self.world} ranks, "
                    f"bit-identical copies" + self._tuned_note())
        if self.mode == "peer":
            return (f"grf_exchange_sum: one kernel per rank over NVLink peer memory (torch symmetric memory), "
                    f"{self.world} ranks, rank-ordered sums (bit-identical copies)" + self._tuned_note())
        return "NCCL all-reduce of U" + (f" (peer memory unavailable: {self.why})" if self.why else "")

    def _tuned_note(self) -> str:
        t = getattr(self, "tuned", None)
        return "" if not t else f"; measured at setup: peer loads {t['peer_ms']:.3f} ms, in-switch sums {t['nvls_ms']:.3f} ms"

    def reduce(self, stream=None) -> torch.Tensor:
        """In stream order: ``self.u`` (this rank's partial) becomes the sum over the ranks."""
        if self.world <= 1:
            return self.u
        if self.mode == "peer":
            import ctypes

            from . import _lib

            self.epoch += 1
            st = stream if stream is not None else ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
            if self._mc:
                _lib.check(_lib.lib().grf_exchange_sum_nvls(ctypes.c_void_p(self._mc), self._pf, self.world, self.rank,
                                                            self.u.numel(), self.epoch & 0xFFFFFFFF or 1, st))
            else:
                _lib.check(_lib.lib().grf_exchange_sum(self._pu, self._pf, self.world, self.rank,
                                                       self.u.numel(), self.epoch & 0xFFFFFFFF or 1, st))
            return self.u
        import torch.distributed as dist

        dist.all_reduce(self.u, group=self.group)
        return self.u


def make_exchange(n_cols: int, ld: int, device, group=None, mode: str = "auto") -> Exchange:
    return Exchange(n_cols, ld, device, group, mode)
