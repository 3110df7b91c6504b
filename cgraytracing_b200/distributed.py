"""render() over the GPUs of one box: one process per GPU, torch.distributed for the plumbing (NCCL over NVLink/NVSwitch).

The reference's render() (main.cpp:169-266) runs its photon loop on 8 OpenMP threads over ONE shared hash table
(main.cpp:225-249). Here the same partitioning is made explicit and replayable (SURVEY.md section 8e):

  eye pass     image rows are split into contiguous tiles, one per rank (main.cpp:185-187 is a plain double loop);
               the per-rank hitpoint records are all-gathered and every rank builds the SAME sorted grid from the union
               (the sort key carries the creation sequence, so the canonical order does not depend on who traced what);
  photon pass  rank g traces the global photon indices [first + g*P/G, first + (g+1)*P/G) of the round — photon k draws the
               same Philox stream whichever GPU traces it — against the replicated hitpoint set. No data-path collective;
  round update one all-reduce(sum) of the per-hitpoint accumulators {dflux.xyz, m}, then every rank applies the same
               radius/flux update (main.cpp:119-122 in its per-round form) and stays bit-identical to its peers.

Stochastic PPM (SPPM, `Context.set_sppm`) shards the same way, except that the eye pass and the exchange of its records run every round:

  per round    rank g traces round r's eye pass over its row tile (the camera of eye path `path` in round r draws from
               (seed, pass 3, path, dim = r), whoever traces it), the tiles are all-gathered and every rank builds the round's grid
               from the same sorted union, with every visible point at its pixel's current radius; then the photon range as above,
               one all-reduce of the round's visible-point accumulators, and the per-pixel fold (identical on every rank).
               The peer-memory exchange is not available under SPPM: its block is sized for a fixed hitpoint count.

`ShardedRenderer` is written against a small engine protocol so that the host logic (ranges, collective order) can be
exercised on CPU with the gloo backend; the product engine is `GpuEngine` (a `Context` behind the C ABI).
"""
from __future__ import annotations

from typing import Tuple

import numpy as np

HP_RECORD_DOUBLES = 12  # CGRT_HP_RECORD_DOUBLES, include/cgrt.h


def split_range(first: int, count: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous, disjoint, covering split of [first, first+count) into `world` parts; the remainder goes to the low ranks."""
    if world <= 0 or not (0 <= rank < world) or count < 0:
        raise ValueError("bad shard request")
    base, rem = divmod(count, world)
    lo = first + rank * base + min(rank, rem)
    return lo, base + (1 if rank < rem else 0)


def photon_shard(round_index: int, photons_per_round: int, rank: int, world: int) -> Tuple[int, int]:
    """Global photon index range of `rank` in round `round_index` (round r owns [r*P, (r+1)*P))."""
    return split_range(round_index * photons_per_round, photons_per_round, rank, world)


def row_shard(height: int, rank: int, world: int) -> Tuple[int, int]:
    """Image rows [y0, y1) of `rank` for the tile-sharded eye pass."""
    y0, n = split_range(0, height, rank, world)
    return y0, y0 + n


class _DevArray:
    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}


def make_native_comm(device: int, rank: int, world: int, group=None) -> int:
    """An NCCL communicator owned by the C ABI side (cgrt_comm_init_rank): rank 0 makes the 128-byte id, torch.distributed only
    carries it to the other ranks. -> ncclComm_t handle for Context.set_comm / allgather_hitpoints."""
    import torch.distributed as dist

    from .binding import comm_init_rank, comm_unique_id

    box = [comm_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0, group=group)
    return comm_init_rank(device, rank, world, box[0])


class GpuEngine:
    """Adapter of a `Context` (C ABI) to the engine protocol; tensors are zero-copy views of ctx-owned device memory.

    With `comm` (a handle from make_native_comm) both collectives of the path run INSIDE the library on its own streams
    (cgrt_allgather_hitpoints; the all-reduce is part of cgrt_round_update and overlaps the next round's trace launches).
    Without it the host framework reduces the accumulator buffer itself (torch.distributed on the library's stream).

    `sppm` (CGRT_SPPM_JITTER / CGRT_SPPM_CORNER) turns stochastic PPM on for the committed context, after the communicator is
    attached (the library requires that order)."""

    def __init__(self, ctx, device: int, comm=None, world: int = 1, rank: int = 0, peer: bool = False, group=None, sppm: int = 0):
        import torch

        self.ctx, self.device, self.torch = ctx, device, torch
        self.comm, self.world, self.rank, self.group = comm, world, rank, group
        self.native_collectives = comm is not None
        # peer = True: the per-round exchange runs over peer memory inside the library (cgrt_peer_*): no collective call in a round,
        # the reduction is fused with the update and overlaps the next round's trace. The communicator then only serves the eye tiles.
        self.peer = bool(peer) and world > 1
        self.sppm = int(sppm)
        if self.sppm and self.peer:
            raise ValueError("SPPM exchanges over NCCL or torch.distributed; the peer-memory exchange is not supported under SPPM")
        if comm is not None and not self.peer:
            ctx.set_comm(comm, world)
        if self.sppm:
            ctx.set_sppm(self.sppm)
        # collectives are enqueued relative to the library's own stream: no host synchronisation between the photon pass, the
        # all-reduce and the update
        self.stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", device))

    def allgather_hitpoints(self):
        self.ctx.allgather_hitpoints(self.comm, self.world)

    def collective_scope(self):
        return self.torch.cuda.stream(self.stream)

    def eye_pass(self, y0, y1):
        self.ctx.eye_pass(y0, y1)

    def sppm_eye_pass(self, r, y0, y1):
        self.ctx.sppm_eye_pass(r, y0, y1)

    def export_hitpoints(self):
        ptr, n = self.ctx.export_hitpoints_dev()
        if n == 0:
            return self.torch.zeros((0, HP_RECORD_DOUBLES), dtype=self.torch.float64, device=f"cuda:{self.device}")
        return self.torch.as_tensor(_DevArray(ptr, n * HP_RECORD_DOUBLES, "<f8"), device=f"cuda:{self.device}").view(n, HP_RECORD_DOUBLES)

    def import_hitpoints(self, rec):
        rec = rec.contiguous()
        self.torch.cuda.synchronize(self.device)
        self.ctx.import_hitpoints_dev(rec.data_ptr(), rec.shape[0])

    def build_grid(self):
        self.ctx.build_grid()
        if self.peer:
            import torch.distributed as dist

            mine = self.ctx.peer_export()
            blobs = [None] * self.world
            dist.all_gather_object(blobs, mine, group=self.group)
            self.ctx.peer_attach(self.rank, self.world, blobs)
        ptr, n = self.ctx.accum_dev()
        ts = {0: "<f8", 1: "<f4", 2: "<i8"}[self.ctx.accum_mode]  # fp64, float, or int64 fixed point (summed exactly by any all-reduce)
        self._acc = self.torch.as_tensor(_DevArray(ptr, n, ts), device=f"cuda:{self.device}") if n else None

    def photon_pass(self, first, count):
        self.ctx.photon_pass(first, count)

    def accum_tensor(self):
        """The live accumulator buffer: reduced in place, in stream order."""
        return self._acc

    def accum_commit(self, t):
        pass

    def round_update(self):
        self.ctx.round_update()

    def gather_image(self, n_emitted):
        return self.ctx.gather_image(n_emitted)


class ShardedRenderer:
    """The host side of a sharded render over an engine. An engine whose `sppm` attribute is non-zero renders stochastic PPM: `eye()`
    then traces the eye pass of the next round (`sppm_eye_pass(round, y0, y1)`) and `render()` calls it before every round."""

    def __init__(self, engine, rank: int = 0, world: int = 1, group=None, shard_eye: bool = True):
        self.e, self.rank, self.world, self.group, self.shard_eye = engine, rank, world, group, shard_eye
        self.sppm = bool(getattr(engine, "sppm", 0))
        self.rounds_done = 0
        self.emitted = 0

    # -- eye pass + grid (SPPM: of round `rounds_done`)
    def _eye_pass(self, y0: int, y1: int):
        if self.sppm:
            self.e.sppm_eye_pass(self.rounds_done, y0, y1)  # also on an empty tile: it starts the round's visible-point set
        elif y1 > y0:
            self.e.eye_pass(y0, y1)

    def eye(self, height: int):
        if self.world == 1 or not self.shard_eye:
            self._eye_pass(0, height)
        else:
            import torch
            import torch.distributed as dist

            y0, y1 = row_shard(height, self.rank, self.world)
            self._eye_pass(y0, y1)
            if getattr(self.e, "native_collectives", False):
                self.e.allgather_hitpoints()
                self.e.build_grid()
                return
            mine = self.e.export_hitpoints()
            counts = torch.zeros(self.world, dtype=torch.int64, device=mine.device)
            counts[self.rank] = mine.shape[0]
            dist.all_reduce(counts, group=self.group)
            counts = [int(c) for c in counts.tolist()]
            cap = max(counts)
            # equal-size all_gather (one NCCL call); ranks pad to the largest tile
            padded = torch.zeros((cap, HP_RECORD_DOUBLES), dtype=torch.float64, device=mine.device)
            padded[: mine.shape[0]] = mine
            parts = [torch.empty_like(padded) for _ in range(self.world)]
            dist.all_gather(parts, padded, group=self.group)
            union = torch.cat([p[:c] for p, c in zip(parts, counts)], 0)
            self.e.import_hitpoints(union)
        self.e.build_grid()

    # -- one round
    def round(self, photons_per_round: int):
        first, count = photon_shard(self.rounds_done, photons_per_round, self.rank, self.world)
        if count:
            self.e.photon_pass(first, count)
        if self.world > 1 and not getattr(self.e, "native_collectives", False) and not getattr(self.e, "peer", False):
            import torch.distributed as dist

            import contextlib

            scope = self.e.collective_scope() if hasattr(self.e, "collective_scope") else contextlib.nullcontext()
            with scope:
                acc = self.e.accum_tensor()
                if acc is not None and acc.numel():
                    dist.all_reduce(acc, group=self.group)
                    self.e.accum_commit(acc)
        self.e.round_update()
        self.rounds_done += 1
        self.emitted += photons_per_round

    def render(self, height: int, rounds: int, photons_per_round: int) -> np.ndarray:
        """The whole of render(): eye pass, `rounds` photon rounds, image gather (identical on every rank). SPPM: an eye pass before
        every round."""
        if not self.sppm:
            self.eye(height)
        for _ in range(rounds):
            if self.sppm:
                self.eye(height)
            self.round(photons_per_round)
        return self.e.gather_image(float(self.emitted))
